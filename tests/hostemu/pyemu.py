"""ctypes binding of tests/hostemu/hostemu.cpp: the product's TALC_HD device code compiled with g++.
A debugging aid for machines without a GPU; the product itself has no CPU path."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libhostemu.so")
SRC = os.path.join(HERE, "hostemu.cpp")
CSRC = os.path.join(HERE, "..", "..", "talc_b200", "csrc")

COUNTER_NAMES = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
                 "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
                 "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out", "reads_ok",
                 "reads_overflow"]


class EmuParams(C.Structure):
    _fields_ = [("K", C.c_uint32), ("MIN_COUNT", C.c_uint32), ("WINDOW_SIZE", C.c_uint32),
                ("MAX_NB_COMPETING_PATHS", C.c_uint32), ("ALPHA", C.c_double), ("SR_ERROR_RATE", C.c_double),
                ("MIN_INNER_SCORE", C.c_double), ("MIN_BORDER_SCORE", C.c_double), ("cycle_mode", C.c_int32),
                ("q11_zero_init", C.c_int32)]


def build(force=False):
    deps = [SRC] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    if force or not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-g", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-x",
                               "c++", SRC, "-o", LIB])


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        L.emu_table_build.restype = C.c_void_p
        L.emu_table_build.argtypes = [C.POINTER(EmuParams), C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                      C.c_uint64, C.c_int]
        L.emu_table_free.argtypes = [C.c_void_p]
        L.emu_correct_reads.argtypes = [C.c_void_p, C.POINTER(EmuParams), C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                        C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        L.emu_correct_interleaved.argtypes = [C.c_void_p, C.POINTER(EmuParams), C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                              C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        L.emu_yields.restype = C.c_uint64
        L.emu_nw.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.emu_lcs.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.emu_overlap.argtypes = [C.c_char_p, C.c_char_p]
        L.emu_xdrop.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                C.POINTER(C.c_int)]
        L.emu_xdrop_reg_fuzz.argtypes = [C.c_uint64, C.c_int, C.c_int]
        L.emu_xdrop_lv_fuzz.argtypes = [C.c_uint64, C.c_int, C.c_int]
        L.emu_xdrop_lv_fuzz_realistic.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int]
        L.emu_xdrop_lv_mode.argtypes = [C.c_int]
        L.emu_seed_extend.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_uint32, C.POINTER(C.c_int32),
                                      C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.emu_align_slices.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int,
                                       C.c_uint32, C.c_void_p]
        L.emu_std_sort_perm.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.emu_tag_next_nodes.argtypes = [C.POINTER(EmuParams), C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p,
                                         C.c_void_p]
        L.emu_test_model.argtypes = [C.POINTER(EmuParams), C.c_int, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def params_from(p) -> EmuParams:
    return EmuParams(p.K, p.MIN_COUNT, p.WINDOW_SIZE, p.MAX_NB_COMPETING_PATHS, p.ALPHA, p.SR_ERROR_RATE,
                     p.MIN_INNER_SCORE, p.MIN_BORDER_SCORE, p.cycle_mode, p.q11_zero_init)


class EmuTable:
    def __init__(self, p: EmuParams, keys, counts, jkeys=None, jcounts=None):
        self.p = p
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        counts = np.ascontiguousarray(counts, dtype=np.int64)
        uj = jkeys is not None
        jk = np.ascontiguousarray(jkeys if uj else [], dtype=np.uint64)
        jc = np.ascontiguousarray(jcounts if uj else [], dtype=np.int64)
        self.h = lib().emu_table_build(C.byref(p), _ptr(keys), _ptr(counts), len(keys), _ptr(jk), _ptr(jc), len(jk),
                                       1 if uj else 0)

    def __del__(self):
        try:
            lib().emu_table_free(self.h)
        except Exception:
            pass

    def correct(self, reads, offsets, arena_bytes=48 * 1024, wide=False, split=False, pause_every=0, state_machine=False):
        reads = np.ascontiguousarray(reads, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        cap = int(offsets[-1]) * 4 + 4096 * n + 4096
        out = np.zeros(cap, dtype=np.uint8)
        ooff = np.zeros(n + 1, dtype=np.uint64)
        status = np.zeros(max(n, 1), dtype=np.uint8)
        ctr = np.zeros(len(COUNTER_NAMES), dtype=np.uint64)
        rc = lib().emu_correct_reads(self.h, C.byref(self.p), _ptr(reads), _ptr(offsets), n, arena_bytes, (1 if wide else 0) | (2 if split else 0) | (4 if state_machine else 0) | ((pause_every & 0xFF) << 8),
                                     _ptr(out), cap, _ptr(ooff), _ptr(status), _ptr(ctr))
        if rc != 0:
            raise RuntimeError("emu output buffer too small")
        return out[: int(ooff[-1])], ooff, status[:n], dict(zip(COUNTER_NAMES, [int(x) for x in ctr]))


def align_slices(op: int, reads, desc, aux: int = 0, aux2: int = 0, k: int = 21) -> np.ndarray:
    """emu_align_slices: talc_test_align_slices (ops 0-5) with the scalar forms, same arguments and result layout."""
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(r) for r in reads])
    data = np.frombuffer(b"".join(reads) + b"\0", dtype=np.uint8).copy()
    desc = np.ascontiguousarray(desc, dtype=np.int32).reshape(-1, 8)
    n = len(desc)
    wide = 3 <= op <= 5
    res = np.zeros(n * (4 if wide else 1), dtype=np.int32)
    if lib().emu_align_slices(op, _ptr(data), _ptr(off), _ptr(desc), n, aux, aux2, k, _ptr(res)) != 0:
        raise ValueError("op %d is not emulated" % op)
    return res.reshape(n, 4) if wide else res


def correct_interleaved(table: EmuTable, reads, offsets, arena_bytes=1 << 20):
    """Two read contexts multiplexed on one thread (the fused kernel's control warp); same outputs as EmuTable.correct."""
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = len(offsets) - 1
    cap = int(offsets[-1]) * 4 + 4096 * n + 4096
    out = np.zeros(cap, dtype=np.uint8)
    ooff = np.zeros(n + 1, dtype=np.uint64)
    status = np.zeros(max(n, 1), dtype=np.uint8)
    ctr = np.zeros(len(COUNTER_NAMES), dtype=np.uint64)
    rc = lib().emu_correct_interleaved(table.h, C.byref(table.p), _ptr(reads), _ptr(offsets), n, arena_bytes, _ptr(out), cap,
                                       _ptr(ooff), _ptr(status), _ptr(ctr))
    if rc != 0:
        raise RuntimeError("emu output buffer too small")
    return out[: int(ooff[-1])], ooff, status[:n], dict(zip(COUNTER_NAMES, [int(x) for x in ctr]))


def test_model(p: EmuParams, op: int, args, use_tabs: bool) -> np.ndarray:
    """emu_test_model: talc_test_model with the g++ build of the same functions, without (use_tabs=False) or with
    host-filled model tables; same argument and result layout."""
    a = np.asarray(args, dtype=np.uint32).reshape(len(args), -1)
    full = np.zeros((len(a), 8), dtype=np.uint32)
    full[:, :a.shape[1]] = a
    out = np.zeros((max(len(a), 1), 9), dtype=np.uint64)
    lib().emu_test_model(C.byref(p), op, _ptr(full), len(a), 1 if use_tabs else 0, _ptr(out))
    return out[:len(a)]
