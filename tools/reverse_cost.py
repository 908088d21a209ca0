"""Cost of --reverse (talc_ctx_set_reverse) on the bench workload: forward mode on batches X against reverse mode on
RC(X), the reverse complement of every read.  Both do exactly the same correction work (same status, counters and
k-mer look-ups); what differs is the reverse-complement pass over the input and the reversed copy of the corrected
reads in gather_kernel, so the ratio of the two rates is the cost of the feature.

  device-resident  the context and one lane from two host threads, one output buffer set per step, CUDA events around
                   each window of steps (bench.py's timed leg); windows alternate forward / reverse, same slices
  end to end       talc_stream_submit / talc_stream_next with host buffers, host clock around each window; alternating

Every timed step is checked afterwards: reverse-mode output == forward-mode output with the corrected reads
reverse-complemented, identical status, offsets and algorithmic counters.  Kernel times of revcomp_reads_kernel and
gather_kernel come from torch.profiler (CUDA activities) in a separate run after the timed windows.  Prints one JSON
line; --out also writes it to a file.  Needs a CUDA device.

  python tools/reverse_cost.py [--rounds 3] [--window 4] [--batch-reads 131072] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHARED = ["lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border", "frontier_sum", "cells_nw",
          "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged", "gap_attempts", "borders",
          "borders_corrected", "ev_gardening", "ev_bridge", "ev_edge", "ev_cycle", "bases_out", "reads_ok"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--batch-reads", type=int, default=131072)
    ap.add_argument("--rounds", type=int, default=3, help="forward / reverse window pairs of the device-resident leg")
    ap.add_argument("--window", type=int, default=4, help="steps per window (split over the context and its lane)")
    ap.add_argument("--e2e-rounds", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    from talc_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("reverse_cost.py: no CUDA device -- the correction path has no CPU fallback")
    dev = "cuda:0"
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()

    cfg = synth.baseline_config(args.config, args.scale)
    use_j = args.config == 3
    tr = synth.make_transcriptome(cfg, dev)
    keys, counts, jk, jc = synth.make_counts(cfg, tr, dev)
    ctx = api.Talc(api.default_params(cfg.k))
    ctx.load_packed(keys.cpu().numpy().astype(np.uint64), counts.cpu().numpy(),
                    jk.cpu().numpy().astype(np.uint64) if use_j else None, jc.cpu().numpy() if use_j else None)
    entries = ctx.table_info()["entries"]
    del keys, counts, jk, jc
    B, W = args.batch_reads, args.window
    nsteps = args.rounds * W + 1
    reads, roff = synth.make_reads(cfg, tr, B * nsteps, dev, seed_offset=3)
    del tr
    roff = roff.to(torch.int64)
    lut = torch.full((256,), ord("N"), dtype=torch.uint8, device=dev)
    for a, b in zip(b"ACGTacgt", b"TGCATGCA"):
        lut[a] = b

    def revcomp(x, off):  # every read of a batch reverse-complemented (off[0] == 0)
        idx = torch.repeat_interleave(off[:-1] + off[1:] - 1, off[1:] - off[:-1]) - torch.arange(int(off[-1]), device=dev)
        return lut[x[idx].long()]

    batches = []  # (X, offsets, bases, RC(X)) per step
    for i in range(nsteps):
        lo, hi = i * B, (i + 1) * B
        b0, b1 = int(roff[lo]), int(roff[hi])
        x, o = reads[b0:b1].contiguous(), (roff[lo:hi + 1] - roff[lo]).contiguous()
        batches.append((x, o, b1 - b0, revcomp(x, o)))
    del reads

    maxb = max(b[2] for b in batches)

    def buffers():
        return (torch.empty(2 * maxb + 64 * B + 4096, dtype=torch.uint8, device=dev),
                torch.zeros(B + 1, dtype=torch.int64, device=dev), torch.zeros(B, dtype=torch.uint8, device=dev))

    def check(fwd, rev):
        """reverse mode on RC(X) against forward mode on X"""
        (fo, ff, fs, fc), (ro, rf, rs, rc_) = fwd, rev
        assert torch.equal(fs, rs), "status differs"
        assert torch.equal(ff, rf), "output offsets differ"
        diff = {k: (fc[k], rc_[k]) for k in SHARED if fc[k] != rc_[k]}
        assert not diff, "counters differ: %s" % diff
        n = int(ff[-1])
        a, b = fo[:n], ro[:n]
        ok = torch.repeat_interleave(fs == 0, ff[1:] - ff[:-1])
        assert torch.equal(torch.where(ok, revcomp(a, ff), a), b), "bytes differ"

    lanes = [ctx, ctx.create_lane()]
    L = len(lanes)
    bufs = [buffers() for _ in range(2 * W)]
    for rev in (False, True, False, True):  # warm-up: both modes on both lanes (scratch, rcBases)
        ctx.set_reverse(rev)
        for l in range(L):
            x, o, nb, rx = batches[-1]
            lanes[l].correct_device(rx if rev else x, o, nb, *bufs[l])
    torch.cuda.synchronize()

    def window(rev, steps, bset):
        ctx.set_reverse(rev)  # no batch pending: every thread of the previous window has joined
        res = [None] * len(steps)
        errors = []

        def run(l):
            try:
                for j in range(l, len(steps), L):
                    x, o, nb, rx = batches[steps[j]]
                    res[j] = lanes[l].correct_device(rx if rev else x, o, nb, *bset[j])
            except Exception as e:  # noqa: BLE001 -- reported below
                errors.append(e)

        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        th = [threading.Thread(target=run, args=(l,)) for l in range(L)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        torch.cuda.synchronize()
        e1.record()
        e1.synchronize()
        if errors:
            raise errors[0]
        return e0.elapsed_time(e1), res

    ms = {False: 0.0, True: 0.0}
    bases = {False: 0, True: 0}
    per_window = []
    checked = 0
    for r in range(args.rounds):
        steps = list(range(r * W, (r + 1) * W))
        order = (False, True) if r % 2 == 0 else (True, False)
        got = {}
        for rev in order:
            bset = bufs[W:] if rev else bufs[:W]
            t, res = window(rev, steps, bset)
            ms[rev] += t
            bases[rev] += sum(batches[s][2] for s in steps)
            per_window.append({"reverse": rev, "ms": round(t, 3), "mbps": sum(batches[s][2] for s in steps) / 1e3 / t})
            got[rev] = [(bset[j][0], bset[j][1], bset[j][2], res[j]) for j in range(W)]
        for j in range(W):
            check(got[False][j], got[True][j])
            checked += 1
    lanes[1].close()
    mbps = {m: bases[m] / 1e3 / ms[m] for m in (False, True)}

    # ---- end to end through the stream, host buffers in and out
    E = min(W, nsteps - 1)
    host = [(batches[s][0].cpu().numpy(), batches[s][1].cpu().numpy().astype(np.uint64), batches[s][2],
             batches[s][3].cpu().numpy()) for s in range(E)]
    stream = ctx.stream()
    e2e_ms = {False: 0.0, True: 0.0}
    e2e_bases = {False: 0, True: 0}
    e2e_checked = 0

    def e2e_window(rev, timed=True):
        ctx.set_reverse(rev)  # the stream is drained between windows
        outs = []
        t0 = time.perf_counter()
        for s in range(E):
            x, o, nb, rx = host[s]
            stream.submit(rx if rev else x, o)
            if s >= 1:
                outs.append(stream.next())
        outs.append(stream.next())
        t = (time.perf_counter() - t0) * 1e3
        if timed:
            e2e_ms[rev] += t
            e2e_bases[rev] += sum(h[2] for h in host)
        return outs

    e2e_window(False, timed=False)
    e2e_window(True, timed=False)
    for r in range(args.e2e_rounds):
        got = {}
        for rev in ((False, True) if r % 2 == 0 else (True, False)):
            got[rev] = e2e_window(rev)
        for (fo, ff, fs, _, fc), (ro, rf, rs, _, rc_) in zip(got[False], got[True]):
            t = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.int64) if a.dtype == np.uint64 else a).to(dev)
            check((t(fo), t(ff), t(fs), fc), (t(ro), t(rf), t(rs), rc_))
            e2e_checked += 1
    stream.close()
    e2e = {m: e2e_bases[m] / 1e3 / e2e_ms[m] for m in (False, True)}

    # ---- kernel times, profiler on, after the timed windows
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    x, o, nb, rx = batches[0]
    for rev in (False, True):
        ctx.set_reverse(rev)
        ctx.correct_device(rx if rev else x, o, nb, *bufs[0])
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.correct_device(rx if rev else x, o, nb, *bufs[0])
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            for name in ("revcomp_reads_kernel", "gather_kernel"):
                if name in ev.key:
                    us = getattr(ev, "device_time_total", None)
                    if us is None:
                        us = ev.cuda_time_total
                    kern["%s_%s_ms" % (name, "reverse" if rev else "forward")] = us / 1e3 / max(1, ev.count)
    ctx.close()

    line = {
        "metric": "reverse-mode throughput over forward-mode throughput, bench workload",
        "ratio": mbps[True] / mbps[False], "forward_mbps": mbps[False], "reverse_mbps": mbps[True],
        "e2e_ratio": e2e[True] / e2e[False], "e2e_forward_mbps": e2e[False], "e2e_reverse_mbps": e2e[True],
        "strand_check": "passed on %d device-resident and %d end-to-end step pairs" % (checked, e2e_checked),
        "kernel_ms": kern, "kernel_ms_source": "torch.profiler CUDA activities, one call per mode after the timed windows",
        "windows": per_window,
        "workload": {"config": args.config, "scale": args.scale, "k": cfg.k, "table_entries": entries,
                     "reads_per_step": B, "steps_per_window": W, "rounds": args.rounds, "lanes": L,
                     "bases_per_step": [batches[s][2] for s in range(args.rounds * W)]},
        "e2e_note": "talc_stream_submit / talc_stream_next, host clock around %d steps per window, results copied out "
                    "of the stream's pinned buffers in the timed region (both modes alike)" % E,
        "device": smi,
    }
    s = json.dumps(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    print(s)


if __name__ == "__main__":
    main()
