"""ctypes binding of tests/hostemu/strand_emu.cpp: --strand auto's decision through the product's TALC_HD helpers
compiled with g++.  A test aid for machines without a GPU; the product itself has no CPU path.  The library is built
into the temporary directory, keyed by the hash of its sources, so that the tree may be read-only."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "strand_emu.cpp")
CSRC = os.path.join(HERE, "..", "..", "talc_b200", "csrc")

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in [SRC] + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")):
            h.update(open(p, "rb").read())
        so = os.path.join(tempfile.gettempdir(), "talc_strand_emu_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++",
                                   SRC, "-o", tmp])
            os.replace(tmp, so)
        L = C.CDLL(so)
        vp = C.c_void_p
        L.emu_orient_reads.argtypes = [C.c_uint32, C.c_uint32, vp, vp, C.c_uint64, vp, vp, C.c_uint32, vp, vp, vp]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def orient(k: int, keys, counts, reads, offsets, min_count: int = 2):
    """(strand uint8[n], found_fwd uint32[n], found_rc uint32[n]) of the reads against the table of keys / counts"""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    counts = np.ascontiguousarray(counts, dtype=np.int64)
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = len(offsets) - 1
    strand = np.zeros(max(n, 1), dtype=np.uint8)
    ff = np.zeros(max(n, 1), dtype=np.uint32)
    fr = np.zeros(max(n, 1), dtype=np.uint32)
    lib().emu_orient_reads(k, min_count, _ptr(keys), _ptr(counts), len(keys), _ptr(reads), _ptr(offsets), n, _ptr(strand),
                           _ptr(ff), _ptr(fr))
    return strand[:n], ff[:n], fr[:n]
