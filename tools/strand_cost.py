"""Cost and effect of --strand auto (talc_ctx_set_strand(ctx, TALC_STRAND_AUTO)) on the bench workload.

  (a) all-sense input   the bench reads as they are: windows of forward mode and auto mode alternate on the same
                        slices, device-resident (the context and one lane from two host threads, CUDA events around
                        each window, bench.py's timed leg) and end to end (talc_stream_submit / talc_stream_next with
                        host buffers, host clock around each window).  The ratio of the two rates is the cost of the
                        orientation probes.
  (b) mixed input       a seeded half of the reads reverse-complemented, as a cDNA library of both orientations gives
                        them: forward mode against auto mode, reads corrected, corrected bases and Mbp/s.
  (c) kernel rate       orient_kernel against coverage_kernel, torch.profiler (CUDA activities) in a separate run after
                        the timed windows: achieved random-sector GB/s (2 * sum(C) * 32 B / time for orient_kernel, which
                        probes both strands, sum(C) * 32 B / time for coverage_kernel) next to the independent-load peak
                        of talc_bench_random_sectors.

Every timed auto-mode step is checked afterwards against what the oracle defines: forward mode on the oriented batch
(each strand-1 read reverse-complemented) with the strand-1 reads flipped back -- same bytes, status, offsets and
algorithmic counters; every timed forward step against an untimed forward run of the same slice.  Prints one JSON line;
--out also writes it to a file.  Needs a CUDA device.

  python tools/strand_cost.py [--rounds 3] [--window 4] [--batch-reads 131072] [--out FILE]
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
    ap.add_argument("--rounds", type=int, default=3, help="forward / auto window pairs of the device-resident leg")
    ap.add_argument("--window", type=int, default=4, help="steps per window (split over the context and its lane)")
    ap.add_argument("--e2e-rounds", type=int, default=2)
    ap.add_argument("--mixed-rounds", type=int, default=1)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    from talc_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("strand_cost.py: no CUDA device -- the correction path has no CPU fallback")
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

    def flip(x, off, sel):
        """the reads of a batch with sel[r] != 0 reverse-complemented (Dna5), the others unchanged (off[0] == 0)"""
        lens = off[1:] - off[:-1]
        idx = torch.repeat_interleave(off[:-1] + off[1:] - 1, lens) - torch.arange(int(off[-1]), device=dev)
        pick = torch.repeat_interleave(sel.to(torch.bool), lens)
        return torch.where(pick, lut[x[idx].long()], x)

    gen = torch.Generator(device=dev)
    gen.manual_seed(20)
    batches = []  # (X, offsets, bases, mixed(X), k-mer windows) per step
    for i in range(nsteps):
        lo, hi = i * B, (i + 1) * B
        b0, b1 = int(roff[lo]), int(roff[hi])
        x, o = reads[b0:b1].contiguous(), (roff[lo:hi + 1] - roff[lo]).contiguous()
        half = torch.rand(B, device=dev, generator=gen) < 0.5
        windows = int(torch.clamp(o[1:] - o[:-1] - cfg.k + 1, min=0).sum())
        batches.append((x, o, b1 - b0, flip(x, o, half), windows))
    del reads
    torch.cuda.synchronize()

    maxb = max(b[2] for b in batches)

    def buffers():  # out, out offsets, status, strands
        return (torch.empty(2 * maxb + 64 * B + 4096, dtype=torch.uint8, device=dev),
                torch.zeros(B + 1, dtype=torch.int64, device=dev), torch.zeros(B, dtype=torch.uint8, device=dev),
                torch.zeros(B, dtype=torch.uint8, device=dev))

    def snapshot(bset, c):
        o, f, s, st = bset
        return o[: int(f[-1])].clone(), f.clone(), s.clone(), st.clone(), c

    ref = buffers()

    def check(x, o, nb, got):
        """auto (or forward) result of batch x against forward mode on the oriented batch, strand-1 reads flipped back"""
        out, off, st, strand, c = got
        ctx.set_strand("forward")
        oriented = flip(x, o, strand)
        torch.cuda.synchronize()  # the library's streams do not wait for torch's
        rc_ = ctx.correct_device(oriented, o, nb, *ref[:3])
        fo, ff, fs = ref[0][: int(ref[1][-1])], ref[1], ref[2]
        assert torch.equal(st, fs), "status differs"
        assert torch.equal(off, ff), "output offsets differ"
        diff = {k: (c[k], rc_[k]) for k in SHARED if c[k] != rc_[k]}
        assert not diff, "counters differ: %s" % diff
        assert torch.equal(out, flip(fo, ff, strand)), "bytes differ"

    lanes = [ctx, ctx.create_lane()]
    L = len(lanes)
    bufs = [buffers() for _ in range(2 * W)]
    for mode in ("forward", "auto", "forward", "auto"):  # warm-up: both modes on both lanes (scratch, rcBases, covRc)
        ctx.set_strand(mode)
        for l in range(L):
            x, o, nb, mx, _ = batches[-1]
            lanes[l].correct_device(x, o, nb, *bufs[l][:3])
    torch.cuda.synchronize()

    def window(mode, inputs, bset):
        ctx.set_strand(mode)  # no batch pending: every thread of the previous window has joined
        res = [None] * len(inputs)
        errors = []

        def run(l):
            try:
                for j in range(l, len(inputs), L):
                    x, o, nb = inputs[j]
                    res[j] = lanes[l].correct_device(x, o, nb, *bset[j][:3])
                    lanes[l].last_strands(len(o) - 1, out=bset[j][3])
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
        return e0.elapsed_time(e1), [snapshot(bset[j], res[j]) for j in range(len(inputs))]

    # ---- (a) all-sense input, device-resident
    ms = {"forward": 0.0, "auto": 0.0}
    nbases = {"forward": 0, "auto": 0}
    per_window = []
    checked = 0
    antisense_chosen = 0
    sense_ok = {"forward": 0, "auto": 0}
    sense_reads = {"forward": 0, "auto": 0}
    for r in range(args.rounds):
        steps = list(range(r * W, (r + 1) * W))
        inputs = [batches[s][:3] for s in steps]
        for mode in (("forward", "auto") if r % 2 == 0 else ("auto", "forward")):
            bset = bufs[W:] if mode == "auto" else bufs[:W]
            t, got = window(mode, inputs, bset)
            ms[mode] += t
            nb = sum(batches[s][2] for s in steps)
            nbases[mode] += nb
            per_window.append({"input": "sense", "mode": mode, "ms": round(t, 3), "mbps": nb / 1e3 / t})
            for j, s in enumerate(steps):
                check(*batches[s][:3], got[j])
                checked += 1
                sense_ok[mode] += int((got[j][2] == 0).sum())
                sense_reads[mode] += len(got[j][2])
                if mode == "auto":
                    antisense_chosen += int(got[j][3].sum())
    mbps = {m: nbases[m] / 1e3 / ms[m] for m in ms}

    # ---- (b) mixed input, device-resident
    mix = {m: {"ms": 0.0, "bases": 0, "reads": 0, "reads_ok": 0, "bases_corrected": 0} for m in ("forward", "auto")}
    mixed_checked = 0
    for r in range(args.mixed_rounds):
        steps = list(range(r * W, (r + 1) * W))
        inputs = [(batches[s][3], batches[s][1], batches[s][2]) for s in steps]
        for mode in (("forward", "auto") if r % 2 == 0 else ("auto", "forward")):
            bset = bufs[W:] if mode == "auto" else bufs[:W]
            t, got = window(mode, inputs, bset)
            d = mix[mode]
            d["ms"] += t
            d["bases"] += sum(batches[s][2] for s in steps)
            per_window.append({"input": "mixed", "mode": mode, "ms": round(t, 3),
                               "mbps": sum(batches[s][2] for s in steps) / 1e3 / t})
            for j, s in enumerate(steps):
                out, off, st, strand, c = got[j]
                ok = st == 0
                d["reads"] += len(st)
                d["reads_ok"] += int(ok.sum())
                d["bases_corrected"] += int(((off[1:] - off[:-1]) * ok).sum())
                check(*inputs[j], got[j])
                mixed_checked += 1
    for d in mix.values():
        d["mbps"] = d["bases"] / 1e3 / d["ms"]
        d["reads_ok_fraction"] = d["reads_ok"] / max(1, d["reads"])
    lanes[1].close()

    # ---- (a) end to end through the stream, host buffers in and out
    E = min(W, nsteps - 1)
    host = [(batches[s][0].cpu().numpy(), batches[s][1].cpu().numpy().astype(np.uint64), batches[s][2]) for s in range(E)]
    stream = ctx.stream()
    e2e_ms = {"forward": 0.0, "auto": 0.0}
    e2e_bases = {"forward": 0, "auto": 0}
    e2e_checked = 0

    def e2e_window(mode, timed=True):
        ctx.set_strand(mode)  # the stream is drained between windows
        outs = []
        t0 = time.perf_counter()
        for s in range(E):
            x, o, nb = host[s]
            stream.submit(x, o)
            if s >= 1:
                outs.append(stream.next() + (stream.strands(),))
        outs.append(stream.next() + (stream.strands(),))
        t = (time.perf_counter() - t0) * 1e3
        if timed:
            e2e_ms[mode] += t
            e2e_bases[mode] += sum(h[2] for h in host)
        return outs

    e2e_window("forward", timed=False)
    e2e_window("auto", timed=False)
    for r in range(args.e2e_rounds):
        for mode in (("forward", "auto") if r % 2 == 0 else ("auto", "forward")):
            outs = e2e_window(mode)
            for s, (o, f, st, _, c, strand) in enumerate(outs):
                assert (strand is None) == (mode == "forward")
                strand = np.zeros(len(st), np.uint8) if strand is None else strand
                t = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.int64) if a.dtype == np.uint64 else a).to(dev)
                check(*batches[s][:3], (t(o), t(f), t(st), t(strand), c))
                e2e_checked += 1
    stream.close()
    e2e = {m: e2e_bases[m] / 1e3 / e2e_ms[m] for m in e2e_ms}

    # ---- (c) kernel times, profiler on, after the timed windows
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    x, o, nb, _, windows = batches[0]
    for mode, name in (("forward", "coverage_kernel"), ("auto", "orient_kernel")):
        ctx.set_strand(mode)
        ctx.correct_device(x, o, nb, *bufs[0][:3])
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ctx.correct_device(x, o, nb, *bufs[0][:3])
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if name in ev.key:
                us = getattr(ev, "device_time_total", None)
                if us is None:
                    us = ev.cuda_time_total
                kern[name + "_ms"] = us / 1e3 / max(1, ev.count)
    peak_gbs, _ = ctx.bench_random_sectors(4 << 30, dependent=False)
    sectors = {"coverage_kernel": windows, "orient_kernel": 2 * windows}
    rate = {k: sectors[k] * 32 / (kern[k + "_ms"] * 1e-3) / 1e9 for k in sectors if k + "_ms" in kern}
    ctx.close()

    line = {
        "metric": "auto-mode throughput over forward-mode throughput on all-sense input, bench workload",
        "ratio": mbps["auto"] / mbps["forward"], "forward_mbps": mbps["forward"], "auto_mbps": mbps["auto"],
        "e2e_ratio": e2e["auto"] / e2e["forward"], "e2e_forward_mbps": e2e["forward"], "e2e_auto_mbps": e2e["auto"],
        "sense_reads_put_on_strand_1": antisense_chosen,
        "sense_reads_ok_fraction": {m: sense_ok[m] / max(1, sense_reads[m]) for m in sense_ok},
        "mixed": mix,
        "kernel_ms": kern, "kernel_ms_source": "torch.profiler CUDA activities, 3 calls per mode after the timed windows",
        "random_sector_gbs": rate, "random_sector_peak_gbs": peak_gbs,
        "orient_fraction_of_peak": rate.get("orient_kernel", 0) / peak_gbs,
        "coverage_fraction_of_peak": rate.get("coverage_kernel", 0) / peak_gbs,
        "peak_source": "talc_bench_random_sectors, 4 GiB buffer, independent loads",
        "check": "passed on %d sense, %d mixed device-resident and %d end-to-end steps: forward mode on the oriented "
                 "batch, strand-1 reads flipped back" % (checked, mixed_checked, e2e_checked),
        "windows": per_window,
        "workload": {"config": args.config, "scale": args.scale, "k": cfg.k, "table_entries": entries,
                     "reads_per_step": B, "steps_per_window": W, "rounds": args.rounds, "lanes": L,
                     "bases_per_step": [batches[s][2] for s in range(args.rounds * W)]},
        "e2e_note": "talc_stream_submit / talc_stream_next / talc_stream_strands, host clock around %d steps per window, "
                    "results copied out of the stream's pinned buffers in the timed region (both modes alike)" % E,
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
