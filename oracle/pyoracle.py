"""ctypes binding of the CPU restatement (oracle/talc_oracle*.cpp).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs -- never by the product package.  PARITY UNPINNED (see oracle/talc_oracle.hpp).
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_build", "libtalc_oracle.so")
BIN = os.path.join(HERE, "_build", "talc_oracle")


class OrcParams(C.Structure):
    _fields_ = [("K", C.c_uint32), ("MIN_COUNT", C.c_uint32), ("WINDOW_SIZE", C.c_uint32),
                ("MAX_NB_COMPETING_PATHS", C.c_uint32), ("ALPHA", C.c_double), ("SR_ERROR_RATE", C.c_double),
                ("MIN_INNER_SCORE", C.c_double), ("MIN_BORDER_SCORE", C.c_double), ("cycle_mode", C.c_int32),
                ("q11_zero_init", C.c_int32)]


def make_params(k=21, min_count=2, window=9, max_branches=7, alpha=2.57, sr_error=0.025, min_inner=0.7,
                min_border=0.7, cycle_mode=0, q11=1) -> OrcParams:
    return OrcParams(k, min_count, window, max_branches, alpha, sr_error, min_inner, min_border, cycle_mode, q11)


def build(force: bool = False) -> None:
    if force or not (os.path.exists(LIB) and os.path.exists(BIN)):
        subprocess.check_call(["make", "-C", HERE, "-s"], stdout=subprocess.DEVNULL)


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        L.orc_table_new.restype = C.c_void_p
        L.orc_table_new.argtypes = [C.c_int]
        L.orc_table_free.argtypes = [C.c_void_p]
        L.orc_table_size.restype = C.c_uint64
        L.orc_table_size.argtypes = [C.c_void_p]
        L.orc_table_load_dump.argtypes = [C.c_void_p, C.POINTER(OrcParams), C.c_char_p, C.c_char_p]
        L.orc_table_build_packed.argtypes = [C.c_void_p, C.POINTER(OrcParams), C.c_void_p, C.c_void_p, C.c_uint64,
                                             C.c_void_p, C.c_void_p, C.c_uint64, C.c_int]
        L.orc_table_lookup.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.orc_coverage.restype = C.c_uint64
        L.orc_coverage.argtypes = [C.c_void_p, C.c_uint32, C.c_char_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.orc_correct_reads.argtypes = [C.c_void_p, C.POINTER(OrcParams), C.c_void_p, C.c_void_p, C.c_uint32, C.c_int,
                                        C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_char_p, C.c_uint64,
                                        C.POINTER(C.c_double)]
        L.orc_correct_reads2.argtypes = L.orc_correct_reads.argtypes + [C.c_void_p]
        L.orc_nw.argtypes = [C.c_char_p, C.c_char_p]
        L.orc_lcs.argtypes = [C.c_char_p, C.c_char_p]
        L.orc_overlap.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.orc_xdrop.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.orc_xdrop_counted.argtypes = L.orc_xdrop.argtypes + [C.POINTER(C.c_uint64)]
        L.orc_seed_extend.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_uint32, C.POINTER(C.c_int32),
                                      C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                      C.POINTER(C.c_int32)]
        L.orc_horspool.restype = C.c_long
        L.orc_horspool.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.orc_is_expected_model.argtypes = [C.c_uint32, C.c_uint32, C.c_double, C.c_int]
        L.orc_is_expected_lastnode.argtypes = [C.c_uint32, C.c_uint32, C.c_double]
        L.orc_tag_next_nodes.argtypes = [C.POINTER(OrcParams), C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p,
                                         C.c_void_p]
        L.orc_std_sort_perm.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.orc_read_stages.argtypes = [C.c_void_p, C.POINTER(OrcParams), C.c_char_p, C.c_uint64, C.c_void_p,
                                      C.POINTER(C.c_double), C.c_void_p, C.POINTER(C.c_int32), C.c_void_p,
                                      C.POINTER(C.c_int32), C.c_int32, C.c_char_p, C.c_uint64]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class OracleTable:
    def __init__(self, params: OrcParams, ordered: bool = False):
        self.p = params
        self.h = lib().orc_table_new(1 if ordered else 0)

    def __del__(self):
        try:
            lib().orc_table_free(self.h)
        except Exception:
            pass

    def load_dump(self, dump: str, junctions: str | None = None):
        lib().orc_table_load_dump(self.h, C.byref(self.p), dump.encode(), junctions.encode() if junctions else None)
        return self

    def build_packed(self, keys, counts, jkeys=None, jcounts=None):
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        counts = np.ascontiguousarray(counts, dtype=np.int64)
        uj = jkeys is not None
        jk = np.ascontiguousarray(jkeys if uj else [], dtype=np.uint64)
        jc = np.ascontiguousarray(jcounts if uj else [], dtype=np.int64)
        lib().orc_table_build_packed(self.h, C.byref(self.p), _ptr(keys), _ptr(counts), len(keys), _ptr(jk), _ptr(jc),
                                     len(jk), 1 if uj else 0)
        return self

    def size(self) -> int:
        return int(lib().orc_table_size(self.h))

    def lookup(self, kmer: str):
        c, col = C.c_uint32(0), C.c_uint32(0)
        found = lib().orc_table_lookup(self.h, kmer.encode(), C.byref(c), C.byref(col))
        return bool(found), c.value, col.value

    def coverage(self, seq: bytes):
        n = max(0, len(seq) - self.p.K + 1)
        cnt = np.zeros(max(n, 1), dtype=np.uint32)
        col = np.zeros(max(n, 1), dtype=np.uint32)
        lib().orc_coverage(self.h, self.p.K, seq, len(seq), _ptr(cnt), _ptr(col))
        return cnt[:n], col[:n]

    def correct(self, reads: np.ndarray, offsets: np.ndarray, threads: int = 1):
        """reads: uint8 ASCII concatenated; offsets: uint64 [n+1].  Returns (out, out_offsets, status, counters, secs)."""
        reads = np.ascontiguousarray(reads, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        cap = int(offsets[-1]) * 4 + 4096 * n + 4096
        out = np.zeros(cap, dtype=np.uint8)
        ooff = np.zeros(n + 1, dtype=np.uint64)
        status = np.zeros(max(n, 1), dtype=np.uint8)
        cj = C.create_string_buffer(8192)
        secs = C.c_double(0)
        rc = lib().orc_correct_reads(self.h, C.byref(self.p), _ptr(reads), _ptr(offsets), n, threads, _ptr(out), cap,
                                     _ptr(ooff), _ptr(status), cj, 8192, C.byref(secs))
        if rc != 0:
            raise RuntimeError("oracle output buffer too small")
        return out[: int(ooff[-1])], ooff, status[:n], json.loads(cj.value.decode()), secs.value

    def read_stats(self, reads: np.ndarray, offsets: np.ndarray, threads: int = 1) -> np.ndarray:
        """[n, 2] {span of the solid regions, number of regions} per read after correction: the kernel-side columns of
        the per-read statistics row (Read.cpp:418-433)."""
        reads = np.ascontiguousarray(reads, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        cap = int(offsets[-1]) * 4 + 4096 * n + 4096
        out = np.zeros(cap, dtype=np.uint8)
        ooff = np.zeros(n + 1, dtype=np.uint64)
        status = np.zeros(max(n, 1), dtype=np.uint8)
        stats = np.zeros((max(n, 1), 2), dtype=np.uint32)
        secs = C.c_double(0)
        lib().orc_correct_reads2(self.h, C.byref(self.p), _ptr(reads), _ptr(offsets), n, threads, _ptr(out), cap, _ptr(ooff),
                                 _ptr(status), None, 0, C.byref(secs), _ptr(stats))
        return stats[:n]

    def stages(self, seq: bytes, max_regions: int = 4096):
        n = max(1, len(seq))
        cov = np.zeros(n, dtype=np.uint32)
        thr = C.c_double(0)
        rf = np.zeros(2 * max_regions, dtype=np.int32)
        rl = np.zeros(2 * max_regions, dtype=np.int32)
        nf, nl = C.c_int32(0), C.c_int32(0)
        trace = C.create_string_buffer(1 << 20)
        st = lib().orc_read_stages(self.h, C.byref(self.p), seq, len(seq), _ptr(cov), C.byref(thr), _ptr(rf), C.byref(nf),
                                   _ptr(rl), C.byref(nl), max_regions, trace, 1 << 20)
        return dict(status=st, threshold=thr.value, found=rf[: 2 * nf.value].reshape(-1, 2),
                    final=rl[: 2 * nl.value].reshape(-1, 2), trace=trace.value.decode())


def nw(a: bytes, b: bytes) -> int:
    return lib().orc_nw(a, b)


def lcs(a: bytes, b: bytes) -> int:
    return lib().orc_lcs(a, b)


def overlap(ref: bytes, cand: bytes, right: bool) -> int:
    return lib().orc_overlap(ref, cand, 1 if right else 0)


def xdrop(query: bytes, database: bytes, left: bool, x: int):
    r, c = C.c_uint64(0), C.c_uint64(0)
    lib().orc_xdrop(query, database, 1 if left else 0, x, C.byref(r), C.byref(c))
    return r.value, c.value


def xdrop_counted(query: bytes, database: bytes, left: bool, x: int):
    """xdrop() plus the number of DP cells the extension visited: (ext_rows, ext_cols, cells)."""
    r, c, n = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    lib().orc_xdrop_counted(query, database, 1 if left else 0, x, C.byref(r), C.byref(c), C.byref(n))
    return r.value, c.value, n.value


def seed_extend(reference: bytes, candidate: bytes, x: int, right: bool, k: int):
    a, b, p, st = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
    s = C.c_double(0)
    lib().orc_seed_extend(reference, candidate, x, 1 if right else 0, k, C.byref(a), C.byref(b), C.byref(p), C.byref(s),
                          C.byref(st))
    return a.value, b.value, p.value, s.value, bool(st.value)


def horspool(h: bytes, n: bytes, mode: int) -> int:
    return lib().orc_horspool(h, n, mode)


def std_sort_perm(keys) -> np.ndarray:
    keys = np.ascontiguousarray(keys, dtype=np.int64)
    perm = np.zeros(len(keys), dtype=np.uint32)
    lib().orc_std_sort_perm(_ptr(keys), len(keys), _ptr(perm))
    return perm


def tag_next_nodes(p: OrcParams, counts4, colours4, count: int, complex_: bool):
    c4 = np.ascontiguousarray(counts4, dtype=np.uint32)
    l4 = np.ascontiguousarray(colours4, dtype=np.uint32)
    tags = np.zeros(4, dtype=np.int32)
    dist = np.zeros(4, dtype=np.float64)
    n = lib().orc_tag_next_nodes(C.byref(p), _ptr(c4), _ptr(l4), count, 1 if complex_ else 0, _ptr(tags), _ptr(dist))
    return n, tags, dist
