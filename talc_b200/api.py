"""ctypes binding of libtalc_b200.so (include/talc_b200.h).

This is the harness side used by tests and bench.py; the product is the shared library and the `talc`
command line built on it.  There is no CPU path: creating a context without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import build as _build


class TalcParams(C.Structure):
    _fields_ = [("K", C.c_uint32), ("min_count", C.c_uint32), ("window_size", C.c_uint32),
                ("max_nb_branches", C.c_uint32), ("alpha", C.c_double), ("sr_error_rate", C.c_double),
                ("min_inner_score", C.c_double), ("min_border_score", C.c_double), ("cycle_mode", C.c_int32),
                ("q11_zero_init", C.c_int32)]


COUNTER_U64 = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
               "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
               "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out", "reads_ok",
               "reads_overflow", "reads", "bases_in", "reads_second_tier", "kernel_launches", "rounds"]
COUNTER_F64 = ["ms_h2d", "ms_coverage", "ms_correct", "ms_correct_tier2", "ms_gather", "ms_d2h", "ms_total"]


class TalcCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in COUNTER_U64] + [(n, C.c_double) for n in COUNTER_F64]

    def as_dict(self):
        return {n: getattr(self, n) for n in COUNTER_U64 + COUNTER_F64}


STATUS_MESSAGES = {1: "No solid kmer could be found.", 2: "Unable to define convenient structure."}
STATUS_RESOURCE = 4  # TALC_READ_RESOURCE: passed through uncorrected, not a reference status
STRAND_MODES = {"forward": 0, "reverse": 1, "auto": 2}  # TALC_STRAND_FORWARD / _REVERSE / _AUTO
SR_SENSE, SR_ANTISENSE, SR_BOTH = 0, 1, 2  # TALC_SR_*: orientation of a short-read file
DUMP_CANONICAL = 1  # TALC_DUMP_CANONICAL
PIECE_MODES = {"off": 0, "trim": 1, "split": 2}  # TALC_PIECES_OFF / _TRIM / _SPLIT

_lib = None


def lib():
    global _lib
    if _lib is None:
        import os
        path = os.environ.get("TALC_LIB") or _build.build_library()  # TALC_LIB: tuning builds only
        L = C.CDLL(path)
        vp, u64p = C.c_void_p, C.POINTER(C.c_uint64)
        L.talc_params_default.argtypes = [C.POINTER(TalcParams), C.c_uint32]
        L.talc_ctx_create.argtypes = [C.POINTER(TalcParams), C.c_int, C.POINTER(vp)]
        L.talc_ctx_destroy.argtypes = [vp]
        L.talc_ctx_create_lane.argtypes = [vp, C.POINTER(vp)]
        L.talc_last_error.restype = C.c_char_p
        L.talc_last_error.argtypes = [vp]
        L.talc_ctx_set_scratch.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32]
        L.talc_ctx_set_exec.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32]
        L.talc_ctx_set_reverse.argtypes = [vp, C.c_int]
        L.talc_ctx_set_strand.argtypes = [vp, C.c_int]
        L.talc_orient_batch.argtypes = [vp, vp, vp, C.c_uint32, vp, vp, vp]
        L.talc_last_strands.argtypes = [vp, vp, C.c_uint32]
        L.talc_stream_strands.argtypes = [vp, C.POINTER(vp)]
        L.talc_ctx_set_pieces.argtypes = [vp, C.c_int, C.c_uint32]
        L.talc_last_pieces.argtypes = [vp, vp, vp, C.c_uint64, u64p]
        L.talc_pieces_batch.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_int, C.c_uint32, vp, vp, C.c_uint64, u64p]
        L.talc_stream_pieces.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
        L.talc_table_load_dump.argtypes = [vp, C.c_char_p, C.c_char_p, u64p, u64p]
        L.talc_table_load_dump_host.argtypes = [vp, C.c_char_p, C.c_char_p, u64p, u64p]
        L.talc_dump_write_packed.argtypes = [C.c_char_p, vp, vp, C.c_uint64, C.c_uint32]
        L.talc_table_count_reads.argtypes = [vp, C.POINTER(C.c_char_p), C.c_int, C.c_uint64, C.c_char_p, u64p, u64p, u64p]
        L.talc_table_count_reads_oriented.argtypes = [vp, C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.c_int, C.c_uint64,
                                                      C.c_char_p, u64p, u64p, u64p]
        L.talc_table_load_dump_ex.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_uint32, u64p, u64p]
        L.talc_table_load_cache_for_ex.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, u64p]
        L.talc_table_load_packed.argtypes = [vp, vp, vp, C.c_uint64, vp, vp, C.c_uint64, C.c_int, u64p]
        L.talc_table_info.argtypes = [vp, u64p, u64p, u64p]
        L.talc_table_alloc.argtypes = [vp, C.c_uint64]
        L.talc_table_device_ptr.argtypes = [vp, C.POINTER(vp)]
        L.talc_table_seal.argtypes = [vp, C.c_uint64]
        L.talc_table_copy.argtypes = [vp, vp]
        L.talc_table_save.argtypes = [vp, C.c_char_p]
        L.talc_table_load_cache.argtypes = [vp, C.c_char_p, u64p]
        L.talc_table_load_cache_for.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_char_p, u64p]
        L.talc_bench_random_sectors.argtypes = [vp, C.c_uint64, C.c_int, C.c_uint32, C.POINTER(C.c_double),
                                                C.POINTER(C.c_double)]
        L.talc_table_export_device.argtypes = [vp, vp, C.c_uint64]
        L.talc_table_import_device.argtypes = [vp, vp, C.c_uint64, C.c_uint64]
        L.talc_table_lookup.argtypes = [vp, vp, C.c_uint64, vp, vp, vp]
        L.talc_correct_batch.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_uint64, vp, vp, C.POINTER(TalcCounters)]
        L.talc_correct_batch_device.argtypes = [vp, vp, vp, C.c_uint32, C.c_uint64, vp, C.c_uint64, vp, vp,
                                                C.POINTER(TalcCounters)]
        L.talc_coverage_batch.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_uint64]
        L.talc_table_replicate.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.talc_nccl_unique_id.argtypes = [vp]
        L.talc_table_broadcast.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
        L.talc_stream_open.argtypes = [vp, C.c_int, C.POINTER(vp)]
        L.talc_stream_submit.argtypes = [vp, vp, vp, C.c_uint32]
        L.talc_stream_reserve.argtypes = [vp, C.c_uint32, C.c_uint64]
        L.talc_stream_next.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_uint32), C.POINTER(vp),
                                       C.POINTER(TalcCounters)]
        L.talc_stream_pending.restype = C.c_uint64
        L.talc_stream_pending.argtypes = [vp]
        L.talc_stream_last_error.restype = C.c_char_p
        L.talc_stream_last_error.argtypes = [vp]
        L.talc_stream_close.argtypes = [vp]
        L.talc_test_align.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_uint32, C.c_int, C.c_int, vp]
        L.talc_test_align_slices.argtypes = [vp, C.c_int, vp, vp, C.c_uint32, vp, C.c_uint32, C.c_int, C.c_int, vp]
        L.talc_test_sort.argtypes = [vp, vp, C.c_uint32, vp]
        L.talc_test_successors.argtypes = [vp, C.c_int, vp, C.c_uint32, vp, vp, u64p]
        L.talc_test_model.argtypes = [vp, C.c_int, vp, C.c_uint32, vp]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def default_params(k: int, **kw) -> TalcParams:
    p = TalcParams()
    lib().talc_params_default(C.byref(p), k)
    for key, v in kw.items():
        setattr(p, key, v)
    return p


class TalcError(RuntimeError):
    pass


class Talc:
    """One context = one GPU = one replica of the k-mer table."""

    def __init__(self, params: TalcParams, device: int = 0):
        self.params = params
        self.h = C.c_void_p()
        rc = lib().talc_ctx_create(C.byref(params), device, C.byref(self.h))
        if rc != 0:
            raise TalcError("talc_ctx_create failed (%d): %s" % (rc, lib().talc_last_error(None).decode()))

    def create_lane(self) -> "Talc":
        """A second context on the same device borrowing this one's tables (talc_ctx_create_lane): batches corrected
        through both from two threads overlap their tails on the device.  Close it before this context."""
        lane = Talc.__new__(Talc)
        lane.params = self.params
        lane.h = C.c_void_p()
        self._check(lib().talc_ctx_create_lane(self.h, C.byref(lane.h)), "talc_ctx_create_lane")
        return lane

    def close(self):
        if self.h:
            lib().talc_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise TalcError("%s failed (%d): %s" % (what, rc, lib().talc_last_error(self.h).decode()))

    def set_scratch(self, tier1_bytes=0, tier2_bytes=0, tier2_threads=0):
        self._check(lib().talc_ctx_set_scratch(self.h, tier1_bytes, tier2_bytes, tier2_threads), "talc_ctx_set_scratch")

    def set_exec(self, split_walk=0, read_contexts=0, walk_step_cap=0):
        """split_walk: 1 = suspendable reads + walk kernel, 2 = one monolithic kernel (the default); 0 keeps a value."""
        self._check(lib().talc_ctx_set_exec(self.h, split_walk, read_contexts, walk_step_cap), "talc_ctx_set_exec")

    def set_reverse(self, reverse: bool):
        """talc --reverse: reads are corrected on the opposite strand; corrected reads come back in their input
        orientation, all others reverse-complemented (talc_ctx_set_reverse).  Raises on a lane."""
        self._check(lib().talc_ctx_set_reverse(self.h, 1 if reverse else 0), "talc_ctx_set_reverse")

    def set_strand(self, mode):
        """talc --strand: "forward", "reverse" (= set_reverse(True)) or "auto" (each read corrected on the strand where
        it finds more of the table, every read returned in its input orientation), or 0 / 1 / 2 (talc_ctx_set_strand).
        Raises on a lane."""
        m = STRAND_MODES[mode] if isinstance(mode, str) else int(mode)
        self._check(lib().talc_ctx_set_strand(self.h, m), "talc_ctx_set_strand")

    def orient(self, reads: np.ndarray, offsets: np.ndarray):
        """The auto-mode strand decision without correcting, in any mode (talc_orient_batch):
        (strand uint8[n] in {0,1}, found_fwd uint32[n], found_rc uint32[n])."""
        reads = np.ascontiguousarray(reads, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        strand = np.zeros(max(n, 1), dtype=np.uint8)
        ff = np.zeros(max(n, 1), dtype=np.uint32)
        fr = np.zeros(max(n, 1), dtype=np.uint32)
        self._check(lib().talc_orient_batch(self.h, _ptr(reads), _ptr(offsets), n, _ptr(strand), _ptr(ff), _ptr(fr)),
                    "talc_orient_batch")
        return strand[:n], ff[:n], fr[:n]

    def last_strands(self, n: int, out=None):
        """Strands of the first n reads of the last batch corrected through this context (talc_last_strands); all 0
        unless it ran in auto mode.  out: a uint8 torch tensor on the context's device to fill instead of a new array."""
        if out is not None:
            self._check(lib().talc_last_strands(self.h, C.c_void_p(out.data_ptr()), n), "talc_last_strands")
            return out
        dst = np.zeros(max(n, 1), dtype=np.uint8)
        self._check(lib().talc_last_strands(self.h, _ptr(dst), n), "talc_last_strands")
        return dst[:n]

    def set_pieces(self, mode, min_len: int = 1):
        """talc --trim / --split: "off", "trim" (one piece per read, first to last table-supported base) or "split" (one
        piece per supported stretch), or 0 / 1 / 2; pieces shorter than min_len are dropped (talc_ctx_set_pieces).
        Raises on a lane."""
        m = PIECE_MODES[mode] if isinstance(mode, str) else int(mode)
        self._check(lib().talc_ctx_set_pieces(self.h, m, min_len), "talc_ctx_set_pieces")

    def pieces(self, reads: np.ndarray, offsets: np.ndarray, flip=None, mode="split", min_len: int = 1):
        """The pieces rule on any reads without correcting them (talc_pieces_batch): flip[r] != 0 judges read r on its
        reverse complement.  Returns (piece_off uint64[n+1], bounds uint32[total, 2] of [start, end))."""
        reads = np.ascontiguousarray(reads, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        fl = None if flip is None else np.ascontiguousarray(flip, dtype=np.uint8)
        cap = (int(offsets[-1]) + n) // (self.params.K + 1) + 1
        po = np.zeros(n + 1, dtype=np.uint64)
        b = np.zeros((cap, 2), dtype=np.uint32)
        total = C.c_uint64(0)
        m = PIECE_MODES[mode] if isinstance(mode, str) else int(mode)
        self._check(lib().talc_pieces_batch(self.h, _ptr(reads), _ptr(offsets), n, _ptr(fl), m, min_len, _ptr(po), _ptr(b),
                                            cap, C.byref(total)), "talc_pieces_batch")
        return po, b[:total.value]

    def last_pieces(self, n: int):
        """(piece_off uint64[n+1], bounds uint32[total, 2]) of the last batch of n reads corrected through this
        context with pieces on (talc_last_pieces)."""
        total = C.c_uint64(0)
        rc = lib().talc_last_pieces(self.h, None, None, 0, C.byref(total))
        if rc not in (0, -5):  # TALC_ERR_CAPACITY: total is set
            self._check(rc, "talc_last_pieces")
        po = np.zeros(n + 1, dtype=np.uint64)
        b = np.zeros((max(total.value, 1), 2), dtype=np.uint32)
        self._check(lib().talc_last_pieces(self.h, _ptr(po), _ptr(b), total.value, C.byref(total)), "talc_last_pieces")
        return po, b[:total.value]

    # ---- table
    def load_dump(self, dump: str, junctions: Optional[str] = None, canonical: bool = False):
        """canonical=True: the dump holds `jellyfish count -C` counts; each line (x, c) also stands for (rc(x), c)
        (talc_table_load_dump_ex with TALC_DUMP_CANONICAL).  Returns (dump lines, entries kept)."""
        nl, nk = C.c_uint64(0), C.c_uint64(0)
        j = junctions.encode() if junctions else None
        if canonical:
            self._check(lib().talc_table_load_dump_ex(self.h, dump.encode(), j, DUMP_CANONICAL, C.byref(nl), C.byref(nk)),
                        "talc_table_load_dump_ex")
        else:
            self._check(lib().talc_table_load_dump(self.h, dump.encode(), j, C.byref(nl), C.byref(nk)),
                        "talc_table_load_dump")
        return nl.value, nk.value

    def load_dump_host(self, dump: str, junctions: Optional[str] = None):
        """The round-1 host parser, kept for A/B timing against load_dump (GPU parser)."""
        nl, nk = C.c_uint64(0), C.c_uint64(0)
        self._check(lib().talc_table_load_dump_host(self.h, dump.encode(), junctions.encode() if junctions else None,
                                                    C.byref(nl), C.byref(nk)), "talc_table_load_dump_host")
        return nl.value, nk.value

    def count_reads(self, paths, orient=None, expected_distinct: int = 0, junctions: Optional[str] = None):
        """Row f3: build the table by counting k-mers of short-read FASTQ/FASTA files on the GPU.  orient: one
        SR_SENSE / SR_ANTISENSE / SR_BOTH per file (talc_table_count_reads_oriented); None counts every file as it is
        (talc_table_count_reads).  Returns (count increments, distinct k-mers, entries kept)."""
        arr = (C.c_char_p * len(paths))(*[p.encode() for p in paths])
        a, b, d = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        j = junctions.encode() if junctions else None
        if orient is None:
            self._check(lib().talc_table_count_reads(self.h, arr, len(paths), expected_distinct, j, C.byref(a), C.byref(b),
                                                     C.byref(d)), "talc_table_count_reads")
        else:
            if len(orient) != len(paths):
                raise ValueError("count_reads: one orientation per file")
            o = (C.c_int * len(paths))(*[int(x) for x in orient])
            self._check(lib().talc_table_count_reads_oriented(self.h, arr, o, len(paths), expected_distinct, j, C.byref(a),
                                                              C.byref(b), C.byref(d)), "talc_table_count_reads_oriented")
        return a.value, b.value, d.value

    def load_packed(self, keys, counts, jkeys=None, jcounts=None) -> int:
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        counts = np.ascontiguousarray(counts, dtype=np.int64)
        uj = jkeys is not None
        jk = np.ascontiguousarray(jkeys if uj else [], dtype=np.uint64)
        jc = np.ascontiguousarray(jcounts if uj else [], dtype=np.int64)
        nk = C.c_uint64(0)
        self._check(lib().talc_table_load_packed(self.h, _ptr(keys), _ptr(counts), len(keys), _ptr(jk), _ptr(jc), len(jk),
                                                 1 if uj else 0, C.byref(nk)), "talc_table_load_packed")
        return nk.value

    def table_save(self, path: str) -> None:
        self._check(lib().talc_table_save(self.h, path.encode()), "talc_table_save")

    def table_load_cache(self, path: str) -> int:
        n = C.c_uint64(0)
        self._check(lib().talc_table_load_cache(self.h, path.encode(), C.byref(n)), "talc_table_load_cache")
        return n.value

    def table_load_cache_for(self, path: str, dump: str, junctions: Optional[str] = None, canonical: bool = False) -> int:
        """canonical: the cache must have been saved from a table loaded with load_dump(..., canonical=True), and
        without it from one that was not (talc_table_load_cache_for_ex)."""
        n = C.c_uint64(0)
        j = junctions.encode() if junctions else None
        if canonical:
            self._check(lib().talc_table_load_cache_for_ex(self.h, path.encode(), dump.encode(), j, DUMP_CANONICAL,
                                                           C.byref(n)), "talc_table_load_cache_for_ex")
        else:
            self._check(lib().talc_table_load_cache_for(self.h, path.encode(), dump.encode(), j, C.byref(n)),
                        "talc_table_load_cache_for")
        return n.value

    def bench_random_sectors(self, buffer_bytes: int = 4 << 30, dependent: bool = False, warps_per_sm: int = 64):
        """(GB/s of random 32-byte sectors, ns per dependent load) -- the roofline of the hash probes."""
        g, ns = C.c_double(0), C.c_double(0)
        self._check(lib().talc_bench_random_sectors(self.h, buffer_bytes, 1 if dependent else 0, warps_per_sm, C.byref(g),
                                                    C.byref(ns)), "talc_bench_random_sectors")
        return g.value, ns.value

    def table_info(self):
        cap, nbytes, n = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        rc = lib().talc_table_info(self.h, C.byref(cap), C.byref(nbytes), C.byref(n))
        return dict(ready=(rc == 0), capacity=cap.value, bytes=nbytes.value, entries=n.value)

    def table_alloc(self, capacity: int):
        self._check(lib().talc_table_alloc(self.h, capacity), "talc_table_alloc")

    def table_device_ptr(self) -> int:
        p = C.c_void_p()
        self._check(lib().talc_table_device_ptr(self.h, C.byref(p)), "talc_table_device_ptr")
        return p.value

    def table_seal(self, n_entries: int):
        self._check(lib().talc_table_seal(self.h, n_entries), "talc_table_seal")

    def table_export_device(self, tensor):
        self._check(lib().talc_table_export_device(self.h, tensor.data_ptr(), tensor.numel() * tensor.element_size()),
                    "talc_table_export_device")

    def table_import_device(self, tensor, capacity: int, n_entries: int):
        self._check(lib().talc_table_import_device(self.h, tensor.data_ptr(), capacity, n_entries),
                    "talc_table_import_device")

    def table_broadcast(self, unique_id: np.ndarray, rank: int, world: int, root: int = 0) -> float:
        uid = np.ascontiguousarray(unique_id, dtype=np.uint8)
        ms = C.c_double(0)
        self._check(lib().talc_table_broadcast(self.h, _ptr(uid), rank, world, root, C.byref(ms)), "talc_table_broadcast")
        return ms.value

    def lookup(self, keys):
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        n = len(keys)
        cnt = np.zeros(n, dtype=np.uint32)
        col = np.zeros(n, dtype=np.uint32)
        found = np.zeros(n, dtype=np.uint8)
        self._check(lib().talc_table_lookup(self.h, _ptr(keys), n, _ptr(cnt), _ptr(col), _ptr(found)), "talc_table_lookup")
        return cnt, col, found

    # ---- correction, host buffers
    def correct(self, reads: np.ndarray, offsets: np.ndarray, out: np.ndarray = None, out_offsets: np.ndarray = None,
                status: np.ndarray = None):
        reads = np.ascontiguousarray(reads, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        cap = 2 * int(offsets[-1]) + 64 * n + 4096
        if out is None:
            out = np.empty(cap, dtype=np.uint8)
        if out_offsets is None:
            out_offsets = np.zeros(n + 1, dtype=np.uint64)
        if status is None:
            status = np.zeros(max(n, 1), dtype=np.uint8)
        ctr = TalcCounters()
        self._check(lib().talc_correct_batch(self.h, _ptr(reads), _ptr(offsets), n, _ptr(out), len(out), _ptr(out_offsets),
                                             _ptr(status), C.byref(ctr)), "talc_correct_batch")
        return out[: int(out_offsets[n])], out_offsets, status[:n], ctr.as_dict()

    # ---- correction, device-resident torch tensors
    def correct_device(self, d_reads, d_offsets, total_bases: int, d_out, d_out_offsets, d_status):
        n = d_offsets.numel() - 1
        ctr = TalcCounters()
        self._check(lib().talc_correct_batch_device(self.h, d_reads.data_ptr(), d_offsets.data_ptr(), n, total_bases,
                                                    d_out.data_ptr(), d_out.numel(), d_out_offsets.data_ptr(),
                                                    d_status.data_ptr(), C.byref(ctr)), "talc_correct_batch_device")
        return ctr.as_dict()

    def coverage(self, reads: np.ndarray, offsets: np.ndarray) -> np.ndarray:
        reads = np.ascontiguousarray(reads, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        lens = (offsets[1:] - offsets[:-1]).astype(np.int64)
        k = self.params.K
        total = int(np.maximum(lens - k + 1, 0).sum())
        counts = np.zeros(max(total, 1), dtype=np.uint32)
        self._check(lib().talc_coverage_batch(self.h, _ptr(reads), _ptr(offsets), n, _ptr(counts), len(counts)),
                    "talc_coverage_batch")
        return counts[:total]

    def stream(self, read_stats: bool = False) -> "TalcStream":
        return TalcStream(self, read_stats)

    # ---- device self-tests
    def test_align(self, op: int, a_list, b_list, aux: int = 0, aux2: int = 0) -> np.ndarray:
        def cat(lst):
            off = np.zeros(len(lst) + 1, dtype=np.uint64)
            for i, s in enumerate(lst):
                off[i + 1] = off[i] + len(s)
            data = np.frombuffer(b"".join(lst) + b"\0", dtype=np.uint8).copy()
            return data, off
        a, ao = cat(a_list)
        b, bo = cat(b_list)
        n = len(a_list)
        res = np.zeros(n * (4 if op >= 3 else 1), dtype=np.int32)
        self._check(lib().talc_test_align(self.h, op, _ptr(a), _ptr(ao), _ptr(b), _ptr(bo), n, aux, aux2, _ptr(res)),
                    "talc_test_align")
        return res.reshape(n, 4) if op >= 3 else res

    def test_align_slices(self, op: int, reads, desc, aux: int = 0, aux2: int = 0) -> np.ndarray:
        """talc_test_align_slices: `reads` a list of byte strings, `desc` an [n, 8] array of {read, start, step, len}
        for side a, then side b."""
        off = np.zeros(len(reads) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(r) for r in reads])
        data = np.frombuffer(b"".join(reads) + b"\0", dtype=np.uint8).copy()
        desc = np.ascontiguousarray(desc, dtype=np.int32).reshape(-1, 8)
        n = len(desc)
        wide = 3 <= op <= 5
        res = np.zeros(n * (4 if wide else 1), dtype=np.int32)
        self._check(lib().talc_test_align_slices(self.h, op, _ptr(data), _ptr(off), len(reads), _ptr(desc), n, aux, aux2,
                                                 _ptr(res)), "talc_test_align_slices")
        return res.reshape(n, 4) if wide else res

    def test_successors(self, kmers, right: bool):
        """talc_test_successors: the walk's successor-table look-up of each k-mer, (cnt uint32[n, 4], colmask uint32[n],
        buckets per successor table)."""
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
        n = len(kmers)
        cnt = np.zeros((max(n, 1), 4), dtype=np.uint32)
        cm = np.zeros(max(n, 1), dtype=np.uint32)
        cap = C.c_uint64(0)
        self._check(lib().talc_test_successors(self.h, 1 if right else 0, _ptr(kmers), n, _ptr(cnt), _ptr(cm),
                                               C.byref(cap)), "talc_test_successors")
        return cnt[:n], cm[:n], cap.value

    def test_model(self, op: int, args) -> np.ndarray:
        """talc_test_model: `args` an [n, <=8] array of uint32 (zero-padded to 8 columns); returns uint64[n, 9]."""
        a = np.asarray(args, dtype=np.uint32).reshape(len(args), -1)
        full = np.zeros((len(a), 8), dtype=np.uint32)
        full[:, :a.shape[1]] = a
        out = np.zeros((max(len(a), 1), 9), dtype=np.uint64)
        self._check(lib().talc_test_model(self.h, op, _ptr(full), len(a), _ptr(out)), "talc_test_model")
        return out[:len(a)]

    def test_sort(self, keys) -> np.ndarray:
        keys = np.ascontiguousarray(keys, dtype=np.int64)
        perm = np.zeros(len(keys), dtype=np.uint32)
        self._check(lib().talc_test_sort(self.h, _ptr(keys), len(keys), _ptr(perm)), "talc_test_sort")
        return perm


def write_dump(path: str, keys, counts, k: int) -> None:
    """Jellyfish `dump -c` text from packed k-mers (fast C writer: 49 M lines in seconds)."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    counts = np.ascontiguousarray(counts, dtype=np.int64)
    rc = lib().talc_dump_write_packed(path.encode(), _ptr(keys), _ptr(counts), len(keys), k)
    if rc != 0:
        raise TalcError("talc_dump_write_packed failed (%d)" % rc)


def table_copy(dst: Talc, src: Talc) -> None:
    dst._check(lib().talc_table_copy(dst.h, src.h), "talc_table_copy")


def table_replicate(ctxs) -> float:
    """ctxs[0] holds the table; one NCCL broadcast issued by the library fills the others.  Returns its device ms."""
    arr = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
    ms, used = C.c_double(0), C.c_int(0)
    ctxs[0]._check(lib().talc_table_replicate(arr, len(ctxs), C.byref(ms), C.byref(used)), "talc_table_replicate")
    return ms.value if used.value else -1.0


def nccl_unique_id() -> np.ndarray:
    buf = np.zeros(128, dtype=np.uint8)
    rc = lib().talc_nccl_unique_id(_ptr(buf))
    if rc != 0:
        raise TalcError("talc_nccl_unique_id failed (%d): libnccl.so.2 not loadable" % rc)
    return buf


class TalcStream:
    """talc_stream_*: batches in, corrected batches out in submission order, copies and kernels overlapped."""

    def __init__(self, ctx: Talc, read_stats: bool = False):
        self.ctx = ctx
        self.h = C.c_void_p()
        self._n = 0
        ctx._check(lib().talc_stream_open(ctx.h, 1 if read_stats else 0, C.byref(self.h)), "talc_stream_open")

    def _check(self, rc, what):
        if rc != 0:
            raise TalcError("%s failed (%d): %s" % (what, rc, lib().talc_stream_last_error(self.h).decode()))

    def reserve(self, max_reads: int, max_bases: int):
        self._check(lib().talc_stream_reserve(self.h, max_reads, max_bases), "talc_stream_reserve")

    def submit(self, reads: np.ndarray, offsets: np.ndarray):
        reads = np.ascontiguousarray(reads, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        self._check(lib().talc_stream_submit(self.h, _ptr(reads), _ptr(offsets), len(offsets) - 1), "talc_stream_submit")

    def pending(self) -> int:
        return int(lib().talc_stream_pending(self.h))

    def next(self, copy: bool = True):
        """(out, out_offsets, status, read_stats or None, counters) of the oldest batch; views into the stream's pinned
        buffers unless copy=True (they are recycled by the following call)."""
        po, pf, ps, pt = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        n = C.c_uint32(0)
        ctr = TalcCounters()
        self._check(lib().talc_stream_next(self.h, C.byref(po), C.byref(pf), C.byref(ps), C.byref(n), C.byref(pt),
                                           C.byref(ctr)), "talc_stream_next")
        nn = n.value
        off = np.ctypeslib.as_array(C.cast(pf, C.POINTER(C.c_uint64)), shape=(nn + 1,))
        total = int(off[nn])
        out = np.ctypeslib.as_array(C.cast(po, C.POINTER(C.c_uint8)), shape=(max(total, 1),))[:total]
        st = np.ctypeslib.as_array(C.cast(ps, C.POINTER(C.c_uint8)), shape=(max(nn, 1),))[:nn]
        stats = None
        if pt.value:
            stats = np.ctypeslib.as_array(C.cast(pt, C.POINTER(C.c_uint32)), shape=(max(nn, 1), 2))[:nn]
        if copy:
            out, off, st = out.copy(), off.copy(), st.copy()
            stats = stats.copy() if stats is not None else None
        self._n = nn
        return out, off, st, stats, ctr.as_dict()

    def strands(self, copy: bool = True):
        """uint8[n] strands of the batch last returned by next() (talc_stream_strands), None unless it ran in auto
        mode; a view into the stream's pinned buffer unless copy=True."""
        p = C.c_void_p()
        self._check(lib().talc_stream_strands(self.h, C.byref(p)), "talc_stream_strands")
        if not p.value:
            return None
        nn = self._n
        st = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(nn, 1),))[:nn]
        return st.copy() if copy else st

    def pieces(self, copy: bool = True):
        """(piece_off uint64[n+1], bounds uint32[total, 2]) of the batch last returned by next() (talc_stream_pieces),
        None unless it ran with pieces on; views into the stream's pinned buffers unless copy=True."""
        po, pb = C.c_void_p(), C.c_void_p()
        self._check(lib().talc_stream_pieces(self.h, C.byref(po), C.byref(pb)), "talc_stream_pieces")
        if not po.value:
            return None
        nn = self._n
        off = np.ctypeslib.as_array(C.cast(po, C.POINTER(C.c_uint64)), shape=(nn + 1,))
        total = int(off[nn])
        b = np.ctypeslib.as_array(C.cast(pb, C.POINTER(C.c_uint32)), shape=(max(total, 1), 2))[:total]
        return (off.copy(), b.copy()) if copy else (off, b)

    def close(self):
        if self.h:
            lib().talc_stream_close(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
