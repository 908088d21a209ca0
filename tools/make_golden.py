"""Generates tests/golden/tiny_case.npz: a small seeded workload (k-mer table lines, junction lines, reads) and
the ORACLE's answer for it (corrected reads, status, counters), so that every implementation -- the oracle
itself on another machine, the host-emulated device code, the CUDA path -- can be pinned to the same bytes.
Run from the repository root:  python tools/make_golden.py"""
import io, json, os, sys, zipfile
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from oracle import pyoracle as po
from talc_b200 import synth


def save_npz_lzma(path, arrays):
    """np.savez with LZMA members (np.load reads them): the random k-mer keys make a deflated file pass 1 MB."""
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for name, a in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(a))
            z.writestr(name + ".npy", buf.getvalue())


out = {}
for name, (ci, scale, n, usej) in {"c1": (1, 0.012, 48, False), "c3": (3, 0.0005, 40, True), "c5": (5, 0.06, 40, False)}.items():
    cfg = synth.baseline_config(ci, scale)
    cfg.n_reads = n
    w = synth.make_workload(cfg)
    keys, counts = w.keys.numpy().astype(np.uint64), w.counts.numpy().astype(np.int64)
    jk, jc = w.jkeys.numpy().astype(np.uint64), w.jcounts.numpy().astype(np.int64)
    reads, off = w.reads.numpy(), w.read_off.numpy().astype(np.uint64)
    t = po.OracleTable(po.make_params(k=cfg.k)).build_packed(keys, counts, jk if usej else None, jc if usej else None)
    o_out, o_off, o_st, ctr, _ = t.correct(reads, off, threads=4)
    out.update({name + "_k": np.array([cfg.k]), name + "_keys": keys, name + "_counts": counts.astype(np.int32),
                name + "_jkeys": jk if usej else np.zeros(0, np.uint64), name + "_jcounts": (jc if usej else np.zeros(0)).astype(np.int32),
                name + "_reads": reads, name + "_off": off, name + "_out": o_out, name + "_ooff": o_off, name + "_status": o_st,
                name + "_ctr": np.frombuffer(json.dumps(ctr).encode(), dtype=np.uint8)})
    print(name, "keys", len(keys), "reads", n, "bases", int(off[-1]), {k: ctr[k] for k in ("gaps", "gaps_bridged", "ev_gardening", "ev_garden_q16", "ev_frontier_over50", "ev_cycle", "ev_q9")})
save_npz_lzma(os.path.join("tests", "golden", "tiny_case.npz"), out)
print(os.path.getsize("tests/golden/tiny_case.npz"), "bytes")
