"""Cost of --split (talc_ctx_set_pieces(ctx, TALC_PIECES_SPLIT, 1)) on the bench workload.

  (a) device-resident   windows of pieces-off and split alternate on the same slices (the context and one lane from two
                        host threads, CUDA events around each window, bench.py's timed leg)
  (b) end to end        talc_stream_submit / talc_stream_next (and talc_stream_pieces with split) with host buffers, host
                        clock around each window, the two settings alternating
  (c) kernel rate       pieces_kernel under torch.profiler (CUDA activities) in a separate run after the timed windows:
                        ms per step and achieved random-sector GB/s (sum over reads of the output's K-mer windows * 32 B
                        / time) next to the independent-load peak of talc_bench_random_sectors

Every timed split step is checked against the pieces-off step of the same slice: same bytes, offsets and status.
Prints one JSON line; --out also writes it to a file.  Needs a CUDA device.

  python tools/pieces_cost.py [--rounds 3] [--window 4] [--batch-reads 131072] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--batch-reads", type=int, default=131072)
    ap.add_argument("--rounds", type=int, default=3, help="off / split window pairs of the device-resident leg")
    ap.add_argument("--window", type=int, default=4, help="steps per window (split over the context and its lane)")
    ap.add_argument("--e2e-rounds", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    from talc_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("pieces_cost.py: no CUDA device -- the correction path has no CPU fallback")
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
    nsteps = args.rounds * W
    reads, roff = synth.make_reads(cfg, tr, B * nsteps, dev, seed_offset=3)
    del tr
    roff = roff.to(torch.int64)
    batches = []
    for i in range(nsteps):
        lo, hi = i * B, (i + 1) * B
        b0, b1 = int(roff[lo]), int(roff[hi])
        batches.append((reads[b0:b1].contiguous(), (roff[lo:hi + 1] - roff[lo]).contiguous(), b1 - b0))
    del reads
    torch.cuda.synchronize()
    maxb = max(b[2] for b in batches)

    def buffers():  # out, out offsets, status
        return (torch.empty(2 * maxb + 64 * B + 4096, dtype=torch.uint8, device=dev),
                torch.zeros(B + 1, dtype=torch.int64, device=dev), torch.zeros(B, dtype=torch.uint8, device=dev))

    lanes = [ctx, ctx.create_lane()]
    L = len(lanes)
    bufs = {"off": [buffers() for _ in range(W)], "split": [buffers() for _ in range(W)]}
    for mode in ("off", "split", "off", "split"):  # warm-up: both settings on both lanes
        ctx.set_pieces(mode)
        for l in range(L):
            lanes[l].correct_device(*batches[-1], *bufs[mode][l])
    torch.cuda.synchronize()

    def window(mode, steps):
        ctx.set_pieces(mode)  # no batch pending: every thread of the previous window has joined
        errors, pieces = [], [0] * len(steps)

        def run(l):
            try:
                for j in range(l, len(steps), L):
                    lanes[l].correct_device(*batches[steps[j]], *bufs[mode][j])
                    if mode == "split":
                        pieces[j] = len(lanes[l].last_pieces(B)[1])
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
        return e0.elapsed_time(e1), sum(pieces)

    # ---- (a) device-resident
    ms = {"off": 0.0, "split": 0.0}
    nbases = {"off": 0, "split": 0}
    per_window, checked, n_pieces = [], 0, 0
    for r in range(args.rounds):
        steps = list(range(r * W, (r + 1) * W))
        for mode in (("off", "split") if r % 2 == 0 else ("split", "off")):
            t, np_ = window(mode, steps)
            ms[mode] += t
            nb = sum(batches[s][2] for s in steps)
            nbases[mode] += nb
            n_pieces += np_
            per_window.append({"mode": mode, "ms": round(t, 3), "mbps": nb / 1e3 / t})
        for j in range(W):
            a, b = bufs["off"][j], bufs["split"][j]
            assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]), "offsets or status differ with pieces on"
            assert torch.equal(a[0][: int(a[1][-1])], b[0][: int(b[1][-1])]), "bytes differ with pieces on"
            checked += 1
    mbps = {m: nbases[m] / 1e3 / ms[m] for m in ms}
    lanes[1].close()

    # ---- (b) end to end through the stream, host buffers in and out
    E = min(W, nsteps)
    host = [(batches[s][0].cpu().numpy(), batches[s][1].cpu().numpy().astype(np.uint64), batches[s][2]) for s in range(E)]
    stream = ctx.stream()
    e2e_ms = {"off": 0.0, "split": 0.0}
    e2e_bases = {"off": 0, "split": 0}
    ref = {}

    def e2e_window(mode, timed=True):
        ctx.set_pieces(mode)  # the stream is drained between windows
        outs = []
        t0 = time.perf_counter()
        for s in range(E):
            x, o, _ = host[s]
            stream.submit(x, o)
            if s >= 1:
                outs.append(stream.next()[:3] + (stream.pieces(),))
        outs.append(stream.next()[:3] + (stream.pieces(),))
        t = (time.perf_counter() - t0) * 1e3
        if timed:
            e2e_ms[mode] += t
            e2e_bases[mode] += sum(h[2] for h in host)
        return outs

    ref["off"] = e2e_window("off", timed=False)
    e2e_window("split", timed=False)
    e2e_checked = 0
    for r in range(args.e2e_rounds):
        for mode in (("off", "split") if r % 2 == 0 else ("split", "off")):
            outs = e2e_window(mode)
            for (o, f, st, p), (ro, rf, rst, _) in zip(outs, ref["off"]):
                assert (p is None) == (mode == "off")
                assert np.array_equal(o, ro) and np.array_equal(f, rf) and np.array_equal(st, rst), "stream results differ"
                e2e_checked += 1
    stream.close()
    e2e = {m: e2e_bases[m] / 1e3 / e2e_ms[m] for m in e2e_ms}

    # ---- (c) pieces_kernel time, profiler on, after the timed windows
    from torch.profiler import ProfilerActivity, profile
    ctx.set_pieces("split")
    x, o, nb = batches[0]
    out = bufs["split"][0]
    ctx.correct_device(x, o, nb, *out)
    torch.cuda.synchronize()
    lens = out[1][1:] - out[1][:-1]
    windows = int(torch.clamp(lens - cfg.k + 1, min=0).sum())
    kern = {}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            ctx.correct_device(x, o, nb, *out)
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        for name in ("pieces_kernel", "pieces_compact_kernel", "coverage_kernel"):
            if ev.key.split("(")[0].split(" ")[-1] == name:
                us = getattr(ev, "device_time_total", None)
                if us is None:
                    us = ev.cuda_time_total
                kern[name + "_ms"] = us / 1e3 / max(1, ev.count)
    peak_gbs, _ = ctx.bench_random_sectors(4 << 30, dependent=False)
    rate = windows * 32 / (kern["pieces_kernel_ms"] * 1e-3) / 1e9 if "pieces_kernel_ms" in kern else None
    ctx.close()

    line = {
        "metric": "split-mode throughput over pieces-off throughput, bench workload",
        "ratio": mbps["split"] / mbps["off"], "off_mbps": mbps["off"], "split_mbps": mbps["split"],
        "e2e_ratio": e2e["split"] / e2e["off"], "e2e_off_mbps": e2e["off"], "e2e_split_mbps": e2e["split"],
        "pieces_per_step": n_pieces / max(1, args.rounds * W), "reads_per_step": B,
        "kernel_ms_per_step": kern,
        "kernel_ms_source": "torch.profiler CUDA activities, 3 split-mode steps after the timed windows",
        "pieces_random_sector_gbs": rate, "random_sector_peak_gbs": peak_gbs,
        "pieces_fraction_of_peak": rate / peak_gbs if rate else None,
        "peak_source": "talc_bench_random_sectors, 4 GiB buffer, independent loads",
        "check": "passed on %d device-resident and %d end-to-end steps: bytes, offsets and status equal to pieces off"
                 % (checked, e2e_checked),
        "windows": per_window,
        "workload": {"config": args.config, "scale": args.scale, "k": cfg.k, "table_entries": entries,
                     "reads_per_step": B, "steps_per_window": W, "rounds": args.rounds, "lanes": L,
                     "output_windows_step0": windows},
        "e2e_note": "talc_stream_submit / talc_stream_next (+ talc_stream_pieces in split mode), host clock around %d "
                    "steps per window" % E,
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
