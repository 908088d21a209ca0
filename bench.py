#!/usr/bin/env python
"""bench.py -- corrected long-read Mbp/s of the TALC correction hot path on B200.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
  python bench.py --impl reference --gpus N --steps K ...   # the CPU restatement of the reference, host cores

Workload = BASELINE.json configs[1]: a 200k-transcript synthetic transcriptome (8k genes + isoforms),
its ~30M-entry k=21 count table, ONT-like long reads (10% error).  A step is one pass of the hot path over
one batch of `--batch-reads` reads of that set (a different slice every step); the table always has its
full size, so the probes miss L2 as they would on the full run.  Multi-GPU is weak scaling: every rank holds
a replica of the table (built on rank 0, one NCCL broadcast) and corrects its own batches; no per-read
communication.  `value` = bases of all ranks / device time (max over ranks) with inputs resident in HBM;
`e2e` = the same through the host-buffer C-ABI call, copies included.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "corrected long-read Mbp/s"
TRAFFIC_SOURCE = ("profiles/r02_traffic_correct_kernel.csv (ncu dram__bytes_read.sum + dram__bytes_write.sum, one launch "
                  "of this workload; captured in round 2 by `tools/r2_gpu_session.sh launches`, kernel sources unchanged since)")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="talc_b200", choices=["talc_b200", "reference"])
    ap.add_argument("--config", type=int, default=2, help="BASELINE.json config index (1-based): 2, 3 (junctions) or 1/5")
    ap.add_argument("--scale", type=float, default=1.0, help="scales transcripts and reads (1.0 = the named config)")
    ap.add_argument("--batch-reads", type=int, default=131072, help="reads per step and per rank")
    ap.add_argument("--cpu-sample-reads", type=int, default=16384, help="reads of the bounded CPU sample (about 10-30 s of host work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=2, help="batches on the device at once in the device-resident leg (1 = one at a time)")
    ap.add_argument("--no-table-load", action="store_true", help="skip the table-load timings (text dump on GPU / host parser / cache)")
    ap.add_argument("--cli-clock", type=int, default=0, metavar="READS",
                    help="also time the `talc` command line end to end (process start -> .fa closed) on READS reads, "
                         "from the text dump and from --tableCache (SURVEY 8d second clock)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="CUDA path only: write what the last timed step computed (rank 0) to DIR/*.npy, so that two "
                         "builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "talc_b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path; --impl reference has none")
    return args


def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one correct_kernel launch of this very workload (131072 reads),
    from the committed metrics-only ncu capture (tools/r2_gpu_session.sh launches); None when the capture is absent."""
    p = os.path.join(ROOT, "profiles", "r02_traffic_correct_kernel.csv")
    if not os.path.exists(p):
        return None
    import csv
    tot = 0
    for row in csv.reader(open(p)):
        if len(row) > 14 and row[12] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += int(row[14])
    return tot or None


def measured_instructions():
    """smsp__inst_executed.sum (warp-instructions) of the same captured launch; None when the capture is absent."""
    p = os.path.join(ROOT, "profiles", "r02_traffic_correct_kernel.csv")
    if not os.path.exists(p):
        return None
    import csv
    for row in csv.reader(open(p)):
        if len(row) > 14 and row[12] == "smsp__inst_executed.sum":
            return int(float(row[14]))
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload_name(args, cfg):
    return ("config%d: %d transcripts (%d genes + isoforms), k=%d count table, ONT-like reads %.0f%% error; "
            "step = batch of %d reads per GPU" % (args.config, cfg.n_transcripts, cfg.n_genes, cfg.k,
                                                   100 * cfg.read_error, args.batch_reads))


# ----------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference's CPU implementation of the path = the oracle restatement (the real binary needs SeqAn2,
    absent here), ordered std::map table as in the reference, all host threads, bounded sample per step."""
    if rank != 0:
        return
    import numpy as np
    import torch
    from oracle import pyoracle as po
    from talc_b200 import synth
    cfg = synth.baseline_config(args.config, args.scale)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    tr = synth.make_transcriptome(cfg, dev)
    keys, counts, jk, jc = synth.make_counts(cfg, tr, dev)
    use_j = args.config == 3
    nsample = max(64, args.cpu_sample_reads // 4)  # per step; the whole run stays within a few minutes
    reads, roff = synth.make_reads(cfg, tr, nsample * (args.steps + args.warmup), dev, seed_offset=3)
    reads, roff = reads.cpu().numpy(), roff.cpu().numpy().astype(np.uint64)
    threads = os.cpu_count() or 1
    t0 = time.time()
    ot = po.OracleTable(po.make_params(k=cfg.k), ordered=True)
    ot.build_packed(keys.cpu().numpy().astype(np.uint64), counts.cpu().numpy(),
                    jk.cpu().numpy().astype(np.uint64) if use_j else None, jc.cpu().numpy() if use_j else None)
    t_table = time.time() - t0
    times, bases = [], 0
    for it in range(args.warmup + args.steps):
        lo, hi = it * nsample, (it + 1) * nsample
        sub = reads[int(roff[lo]):int(roff[hi])]
        so = roff[lo:hi + 1] - roff[lo]
        _, _, _, _, secs = ot.correct(sub, so, threads=threads)
        if it >= args.warmup:
            times.append(secs)
            bases += int(so[-1])
    total = sum(times)
    v = bases / 1e6 / total
    line = {"metric": METRIC, "value": v, "unit": "Mbp/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64/f64 (integer k-mer and DP arithmetic, double decisions)", "data": "synthetic",
            "impl": "reference",
            "config": {"workload": workload_name(args, cfg), "table_entries_kept": ot.size(), "table": "std::map (ordered, as the reference)",
                       "sample_reads_per_step": nsample, "table_build_s": round(t_table, 1)},
            "cpu_baseline": {"value": v, "unit": "Mbp/s", "cores": threads, "kind": "port",
                             "sample": "%d reads per step of the same read set (oracle restatement, OpenMP over reads)" % nsample},
            "e2e": {"value": v, "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ----------------------------------------------------------------------------------------------------------
def run_gpu(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    from talc_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the correction path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = "cuda:%d" % local_rank
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    cfg = synth.baseline_config(args.config, args.scale)
    use_j = args.config == 3
    t0 = time.time()
    tr = synth.make_transcriptome(cfg, dev)
    ctx = api.Talc(api.default_params(cfg.k), device=local_rank)
    keys = counts = jk = jc = None
    t_build = 0.0
    if rank == 0:
        keys, counts, jk, jc = synth.make_counts(cfg, tr, dev)
        tb = time.time()
        ctx.load_packed(keys.cpu().numpy().astype(np.uint64), counts.cpu().numpy(),
                        jk.cpu().numpy().astype(np.uint64) if use_j else None, jc.cpu().numpy() if use_j else None)
        t_build = time.time() - tb
    info = ctx.table_info()
    t_bcast_ms = 0.0
    if world > 1:
        # replicate: ONE ncclBroadcast of the raw slot array over NVLink, issued by the library itself
        # (talc_table_broadcast); torch.distributed only carries the 128-byte NCCL id to the other ranks
        # (NCCL prints a version banner through C stdio when first initialised: see _claim_stdout)
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.from_numpy(api.nccl_unique_id()))
        dist.broadcast(uid, 0)
        t_bcast_ms = ctx.table_broadcast(uid.cpu().numpy(), rank, world, 0)
        info = ctx.table_info()
    # this rank's reads: batch_reads per step, a different slice every step (and every rank)
    nsteps = args.warmup + args.steps + 1  # +1 slice for the e2e leg warm-up
    B = args.batch_reads
    reads, roff = synth.make_reads(cfg, tr, B * nsteps, dev, seed_offset=3 + 17 * rank)
    cpu_keys = (keys, counts, jk, jc)
    tr_keep = tr if world > 1 else None
    tr_cli = tr if args.cli_clock else None
    del tr
    t_gen = time.time() - t0
    roff = roff.to(torch.int64)

    def batch(i):
        lo, hi = (i % nsteps) * B, (i % nsteps + 1) * B
        b0, b1 = int(roff[lo]), int(roff[hi])
        return reads[b0:b1].contiguous(), (roff[lo:hi + 1] - roff[lo]).contiguous(), b1 - b0

    maxb = max(int(roff[(i + 1) * B] - roff[i * B]) for i in range(nsteps))
    d_out = torch.empty(2 * maxb + 64 * B + 4096, dtype=torch.uint8, device=dev)
    d_ooff = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    d_st = torch.zeros(B, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg: W warm-up steps, then exactly K timed steps.  The steps go through the context and its
    # lane (talc_ctx_create_lane: same tables, own stream and scratch) from two host threads, step i on lane i mod 2,
    # so that the tail of one batch (a few long reads, one warp each) overlaps the start of the next; --lanes 1 runs
    # them one after the other as round 1 did.  Timed with CUDA events recorded on an idle device on both sides.
    import threading
    lanes = [ctx] + [ctx.create_lane() for _ in range(max(1, min(args.lanes, 4)) - 1)]
    L = len(lanes)
    bufs = [(d_out, d_ooff, d_st)] + [(torch.empty_like(d_out), torch.zeros_like(d_ooff), torch.zeros_like(d_st)) for _ in range(L - 1)]
    for i in range(max(args.warmup, L)):
        r, o, nb = batch(i)
        lanes[i % L].correct_device(r, o, nb, *bufs[i % L])
    step_ids = list(range(args.warmup, args.warmup + args.steps))
    work = [[batch(i) for i in step_ids[l::L]] for l in range(L)]  # slices made before the clock starts
    results = [[] for _ in range(L)]
    errors = []

    def run_lane(l):
        try:
            for r, o, nb in work[l]:
                results[l].append((lanes[l].correct_device(r, o, nb, *bufs[l]), nb))
        except Exception as e:  # noqa: BLE001 -- reported by the main thread
            errors.append(e)

    sampler = ClockSampler(local_rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    wall0 = time.time()
    ev0.record()
    threads = [threading.Thread(target=run_lane, args=(l,)) for l in range(L)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    torch.cuda.synchronize()
    ev1.record()
    ev1.synchronize()
    dev_ms = ev0.elapsed_time(ev1)
    barrier()
    wall = time.time() - wall0
    clocks = sampler.stop()
    if errors:
        raise errors[0]
    if args.dump_outputs and rank == 0:
        # timed step j ran on lane j mod L, into that lane's buffers; read them before the runs below reuse lane 0's
        last = (args.steps - 1) % L
        dump_outputs(args.dump_outputs, *bufs[last], B, results[last][-1][0])
    bases, agg, launches = 0, None, 0
    for c, nb in [x for l in range(L) for x in results[l]]:
        bases += nb
        launches += 6 + (1 if c["reads_second_tier"] else 0)  # kmer_count, coverage, cost_key, correct(+tier2), len_to_u64, gather
        if agg is None:
            agg = dict(c)
        else:
            for k2, v2 in c.items():
                agg[k2] += v2
    # the dominant kernels timed one launch at a time (what ncu sees, and round 1's figure): two more steps, untimed above
    ser_ids = step_ids if len(step_ids) <= 8 else [step_ids[(j * len(step_ids)) // 8] for j in range(8)]  # spread over the timed steps
    ser = [ctx.correct_device(*batch(i), d_out, d_ooff, d_st) for i in ser_ids]
    ser_ms = sum(c["ms_correct"] + c["ms_correct_tier2"] for c in ser) / len(ser)
    ser_cov_ms = sum(c["ms_coverage"] for c in ser) / len(ser)
    ser_total_ms = sum(c["ms_total"] for c in ser) / len(ser)
    ser_agg = {k2: sum(c[k2] for c in ser) / len(ser) for k2 in ("lookups_deg", "lookups_walk", "lookups_seg", "bases_in", "bases_out")}
    for ln in lanes[1:]:
        ln.close()
    tmax = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(bases)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    value = float(tot) / 1e6 / (float(tmax) / 1e3)

    # ---- end-to-end leg: host (pinned) buffers through talc_correct_batch, copies inside the timed region; ALL
    # steps, timed by the host wall clock around the calls (barrier + synchronize on both sides), max over ranks
    host_out = torch.empty(2 * maxb + 64 * B + 4096, dtype=torch.uint8).pin_memory().numpy()
    host_ooff = np.zeros(B + 1, dtype=np.uint64)
    host_st = np.zeros(B, dtype=np.uint8)
    pinned = []
    for i in range(3):  # three pinned input batches, cycled (a different slice every step, bounded pinned memory)
        r, o, nb = batch(args.warmup + i)
        pinned.append((r.cpu().pin_memory().numpy(), o.cpu().numpy().astype(np.uint64), nb))
    # the call a user of a multi-batch job makes: talc_stream_submit / talc_stream_next (pinned ring of slots, copies
    # of batch i+1 and i-1 overlapped with the kernels of batch i); every step's result is read back on the host
    os.environ["TALC_STREAM_LANES"] = str(L)  # the stream keeps as many batches on the device as the leg above
    stream = ctx.stream()
    depth = L + 1  # batches in flight: the ring has L + 2 slots and one is held by the caller between two next()
    for w_ in range(L + 2):  # warm-up of the host path: every slot of the ring allocates its pinned / device buffers once
        stream.submit(pinned[(w_ + 2) % 3][0], pinned[(w_ + 2) % 3][1])
        if w_ >= depth - 1:
            stream.next(copy=False)
    for w_ in range(depth - 1):
        stream.next(copy=False)
    e2e_bases, h2d, d2h, e2e_dev_ms = 0, 0, 0, 0.0
    barrier()
    w0 = time.perf_counter()
    fetched = 0
    for s_ in range(args.steps):
        hr, ho, nb = pinned[s_ % 3]
        stream.submit(hr, ho)
        e2e_bases += nb
        h2d = nb + 8 * (B + 1)
        if s_ - fetched >= depth - 1:
            out, ooff, st, _, c = stream.next(copy=False)
            e2e_dev_ms += c["ms_total"]
            d2h = int(ooff[-1]) + 8 * (B + 1) + B
            fetched += 1
    while fetched < args.steps:
        out, ooff, st, _, c = stream.next(copy=False)
        e2e_dev_ms += c["ms_total"]
        d2h = int(ooff[-1]) + 8 * (B + 1) + B
        fetched += 1
    barrier()
    e2e_wall_ms = (time.perf_counter() - w0) * 1e3
    stream.close()
    emax = torch.tensor([e2e_wall_ms], dtype=torch.float64, device=dev)
    etot = torch.tensor([float(e2e_bases)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(emax, op=dist.ReduceOp.MAX)
        dist.all_reduce(etot, op=dist.ReduceOp.SUM)
    e2e_value = float(etot) / 1e6 / (float(emax) / 1e3)

    # ---- correctness of what was just timed.  Every rank corrects the SAME batch (rank 0's step-0 slice): the
    # digests of (bytes, offsets, status) must agree across the replicas of the table, and on rank 0 the first
    # `--cpu-sample-reads` reads are compared byte for byte with the oracle below (parity field).
    import hashlib
    if world > 1:
        shared_reads, shared_off = synth.make_reads(cfg, tr_keep, B, dev, seed_offset=3)
        shared_off = shared_off.to(torch.int64)
        sb_r, sb_o, sb_n = shared_reads.contiguous(), shared_off.contiguous(), int(shared_off[-1])
    else:
        sb_r, sb_o, sb_n = batch(0)
    ctx.correct_device(sb_r, sb_o, sb_n, d_out, d_ooff, d_st)
    torch.cuda.synchronize()
    g_off = d_ooff.cpu().numpy().astype(np.uint64)
    g_out = d_out[: int(g_off[-1])].cpu().numpy()
    g_st = d_st.cpu().numpy()
    digest = hashlib.sha256(g_out.tobytes() + g_off.tobytes() + g_st.tobytes()).digest()
    replica_parity = None
    if world > 1:
        mine = torch.tensor(list(digest), dtype=torch.uint8, device=dev)
        allv = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        same = all(bool((v == allv[0]).all()) for v in allv)
        replica_parity = "ok" if same else "MISMATCH"

    if rank == 0:
        peak, peak_src = peaks()
        # dominant kernel = correct_kernel.  Algorithmic bytes per launch (SURVEY 8d): one 32-byte sector per
        # logical k-mer look-up (getOutDegree + whatsNext calls, 4 each) + 2 bits per input base + 1 byte per output base
        steps = args.steps
        lookups = agg["lookups_deg"] + agg["lookups_walk"]
        alg_bytes_region = (32.0 * lookups + agg["bases_in"] / 4.0 + agg["bases_out"]) / steps
        # per-launch figures: the same launches give the bytes and the duration (timed one at a time; inside the timed
        # region consecutive launches overlap by their tails)
        alg_bytes = 32.0 * (ser_agg["lookups_deg"] + ser_agg["lookups_walk"]) + ser_agg["bases_in"] / 4.0 + ser_agg["bases_out"]
        k_ms = ser_ms
        achieved = alg_bytes / 1e9 / (k_ms / 1e3)
        eff_ms = float(tmax) / steps
        cov_bytes = 32.0 * ser_agg["lookups_seg"] + ser_agg["bases_in"] / 4.0 + 4.0 * ser_agg["lookups_seg"]
        cov_ms = ser_cov_ms
        line = {"metric": METRIC, "value": value, "unit": "Mbp/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": float(tmax) / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u64/f64 (integer k-mer and DP arithmetic, double decisions)",
                "data": "synthetic", "impl": "talc_b200",
                "config": {"workload": workload_name(args, cfg), "table_entries_kept": info["entries"],
                           "table_bytes": info["bytes"], "reads_per_step_per_gpu": B,
                           "l2": "inputs larger than L2: %.2f GB table + %.0f MB of reads per step" % (info["bytes"] / 1e9, bases / steps / 1e6),
                           "generate_s": round(t_gen, 1), "table_build_s": round(t_build, 2),
                           "table_broadcast_ms": round(t_bcast_ms, 2), "wall_s_timed_region": round(wall, 3),
                           "lanes": L},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": measured_traffic() if B == 131072 and args.config == 2 and args.scale == 1.0 else None,
                             "traffic_source": TRAFFIC_SOURCE,
                             "kernel": "correct_kernel", "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms_per_launch": k_ms,
                             "kernel_ms_note": "correct_kernel timed one launch at a time (CUDA events around the launch; %d of the timed steps run "
                                               "again after the timed region); in the timed region %d lanes overlap consecutive launches" % (len(ser), L),
                             "ms_per_step_one_at_a_time": ser_total_ms,
                             "achieved_in_timed_region": alg_bytes_region / 1e9 / (eff_ms / 1e3),
                             "frac_in_timed_region": alg_bytes_region / 1e9 / (eff_ms / 1e3) / peak,
                             "coverage_kernel": {"achieved": cov_bytes / 1e9 / (cov_ms / 1e3), "ms_per_launch": cov_ms,
                                                 "algorithmic_bytes_per_launch": cov_bytes,
                                                 "frac": cov_bytes / 1e9 / (cov_ms / 1e3) / peak}},
                "e2e": {"value": e2e_value, "unit": "Mbp/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": args.steps, "clock": "host wall clock around all steps through talc_stream_submit / talc_stream_next "
                                 "(host buffers in, pinned host results out, every result fetched), max over ranks",
                        "wall_ms": float(emax)},
                "replica_parity": replica_parity,
                # stage-4 integer work (SURVEY 8d): DP cell updates of the reference algorithm per second of correct_kernel
                "dp": {"cells_per_launch": (agg["cells_nw"] + agg["cells_lcs"] + agg["cells_ovl"] + agg["cells_xdrop"]) / steps,
                       "gcups": (agg["cells_nw"] + agg["cells_lcs"] + agg["cells_ovl"] + agg["cells_xdrop"]) / steps / 1e9 / (k_ms / 1e3),
                       "note": "cells the reference's DP visits (oracle-equal counters); bit-parallel rows, the register X-drop band "
                               "and the end-cell score mean far fewer machine operations than cells"},
                "gpu_launches": launches,
                "clocks": clocks,
                "counters": {k2: agg[k2] for k2 in ("lookups_seg", "lookups_deg", "lookups_walk", "steps_inner", "steps_border",
                                                     "cells_nw", "cells_lcs", "cells_ovl", "cells_xdrop", "gaps", "gaps_bridged",
                                                     "reads_second_tier", "reads_ok", "reads")},
                "cpu_baseline": None}
        if world == 1 and not args.no_table_load:
            line["table_load"] = table_load_timings(api, cfg, cpu_keys, use_j)
        if world == 1 and args.cli_clock:
            line["cli_clock"] = cli_clock(args, cfg, cpu_keys, use_j, tr_cli, dev)
        # what actually bounds correct_kernel: instruction issue.  Warp-instructions of one launch (ncu capture of this
        # workload) / (SMs x 4 schedulers x one instruction per cycle at the measured SM clock) = the shortest possible
        # launch with this instruction count; frac = that / the measured launch
        n_inst = measured_instructions() if B == 131072 and args.config == 2 and args.scale == 1.0 else None
        if n_inst and clocks.get("sm_mhz"):
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            min_ms = n_inst / (sms * 4 * clocks["sm_mhz"] * 1e6) * 1e3
            line["roofline"]["issue"] = {"warp_instructions_per_launch": n_inst, "source": TRAFFIC_SOURCE,
                                         "schedulers": sms * 4, "sm_mhz": clocks["sm_mhz"],
                                         "ms_per_launch_at_one_instruction_per_cycle": min_ms, "frac": min_ms / k_ms,
                                         "note": "the kernel is bound by instruction issue of a serial per-read program "
                                                 "(8 warps per SM, 231 registers), not by HBM: this is its issue-slot utilisation"}
        rnd = random_sector_peaks(ctx)
        line["roofline"].update(rnd)
        if rnd.get("peak_random"):
            line["roofline"]["frac_random"] = achieved / rnd["peak_random"]
            line["roofline"]["coverage_kernel"]["frac_random"] = line["roofline"]["coverage_kernel"]["achieved"] / rnd["peak_random"]
        bad = 0
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"], line["parity"] = cpu_baseline(args, cfg, cpu_keys, use_j, reads, roff, (g_out, g_off, g_st))
            bad = line["parity"]["mismatch"]
        emit(line)
        if bad or replica_parity == "MISMATCH":
            print("bench.py: PARITY FAILURE -- the numbers above are void", file=sys.stderr, flush=True)
            if world > 1:
                dist.destroy_process_group()
            sys.exit(1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_MAX_READS = 1 << 20
DUMP_SAMPLE_READS = 6144
DUMP_MAX_BASES = 10 << 20


def read_digests(out, off, m):
    """48 bits of BLAKE2b over each of the first m corrected reads: exact in a float64, so that a difference in any
    base of any read shows in a float array."""
    import hashlib
    import numpy as np
    return np.array([int.from_bytes(hashlib.blake2b(out[off[i]:off[i + 1]].tobytes(), digest_size=6).digest(), "little")
                     for i in range(m)], dtype=np.float64)


def dump_outputs(path, d_out, d_ooff, d_st, n, counters):
    """What one talc_correct_batch_device call hands back for a batch of n reads, as .npy files.  For the first
    DUMP_MAX_READS reads: out_offsets.npy (float64, offsets into the corrected bases), status.npy (float32) and
    read_digests.npy (float64, read_digests of the corrected bases).  For a fixed seeded sample of DUMP_SAMPLE_READS
    reads (sample_reads.npy, their indices): their corrected bases as ASCII codes (sample_bases.npy, float32, at most
    DUMP_MAX_BASES of them).  counter_<name>.npy (float64): the call's counters, except its ms_* timings.
    At most 63 MB in all (42 MB for the default config-2 batch of 131072 reads)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    off = d_ooff[: n + 1].cpu().numpy().astype(np.int64)
    out = d_out[: int(off[-1])].cpu().numpy()
    idx = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_SAMPLE_READS), replace=False))
    bases = np.concatenate([out[off[i]:off[i + 1]] for i in idx])[:DUMP_MAX_BASES]
    m = min(n, DUMP_MAX_READS)
    np.save(os.path.join(path, "out_offsets.npy"), off[: m + 1].astype(np.float64))
    np.save(os.path.join(path, "status.npy"), d_st[:m].cpu().numpy().astype(np.float32))
    np.save(os.path.join(path, "read_digests.npy"), read_digests(out, off, m))
    np.save(os.path.join(path, "sample_reads.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "sample_bases.npy"), bases.astype(np.float32))
    for name, v in counters.items():
        if not name.startswith("ms_"):
            np.save(os.path.join(path, "counter_%s.npy" % name), np.array([v], dtype=np.float64))


def table_load_timings(api, cfg, cpu_keys, use_j):
    """Row f1: seconds to get from the Jellyfish text dump of this workload to a sealed table in HBM -- parsed on the
    GPU (talc_table_load_dump), by the threaded host parser of round 1 (talc_table_load_dump_host), and from the
    binary cache (talc_table_load_cache_for)."""
    import tempfile
    import numpy as np
    keys, counts, jk, jc = cpu_keys
    d = tempfile.mkdtemp(prefix="talc_bench_")
    dump, jdump, cache = os.path.join(d, "sr.dump"), os.path.join(d, "j.dump"), os.path.join(d, "table.bin")
    t0 = time.time()
    api.write_dump(dump, keys.cpu().numpy().astype(np.uint64), counts.cpu().numpy(), cfg.k)
    if use_j:
        api.write_dump(jdump, jk.cpu().numpy().astype(np.uint64), jc.cpu().numpy(), cfg.k)
    t_write = time.time() - t0
    res = {"dump_bytes": os.path.getsize(dump), "dump_lines": int(keys.numel()), "write_dump_s": round(t_write, 2)}
    j = jdump if use_j else None
    for name, fn in (("gpu_parser_s", "load_dump"), ("host_parser_s", "load_dump_host")):
        t = api.Talc(api.default_params(cfg.k))
        t0 = time.time()
        nl, nk = getattr(t, fn)(dump, j)
        res[name] = round(time.time() - t0, 2)
        res["entries_kept"] = nk
        if name == "gpu_parser_s":
            t0 = time.time()
            t.table_save(cache)
            res["cache_write_s"] = round(time.time() - t0, 2)
        t.close()
    t = api.Talc(api.default_params(cfg.k))
    t0 = time.time()
    t.table_load_cache_for(cache, dump, j)
    res["cache_load_s"] = round(time.time() - t0, 2)
    t.close()
    for f in (dump, jdump, cache):
        if os.path.exists(f):
            os.remove(f)
    os.rmdir(d)
    return res


def cli_clock(args, cfg, cpu_keys, use_j, tr, dev):
    """SURVEY 8d second clock: the `talc` command line, process start -> .fa closed, on `--cli-clock` reads of this
    workload: table from the text dump, then from --tableCache."""
    import tempfile
    import numpy as np
    from talc_b200 import api, build, synth
    keys, counts, jk, jc = cpu_keys
    d = tempfile.mkdtemp(prefix="talc_cli_")
    dump, jdump = os.path.join(d, "sr.dump"), os.path.join(d, "j.dump")
    api.write_dump(dump, keys.cpu().numpy().astype(np.uint64), counts.cpu().numpy(), cfg.k)
    if use_j:
        api.write_dump(jdump, jk.cpu().numpy().astype(np.uint64), jc.cpu().numpy(), cfg.k)
    reads, roff = synth.make_reads(cfg, tr, args.cli_clock, dev, seed_offset=3)
    synth.write_fasta(os.path.join(d, "reads.fa"), reads, roff)
    bases = int(roff[-1])
    cli = build.build_cli()
    common = [cli, "reads.fa", "--SRCounts", "sr.dump", "-k", str(cfg.k), "-t", str(min(16, os.cpu_count() or 1))] + \
             (["--junctions", "j.dump"] if use_j else [])
    res = {"reads": args.cli_clock, "bases": bases, "fasta_bytes": os.path.getsize(os.path.join(d, "reads.fa"))}
    for name, extra in (("text_dump", ["-o", "a"]), ("cache_cold", ["-o", "b", "--tableCache", "t.bin"]),
                        ("cache_warm", ["-o", "c", "--tableCache", "t.bin"])):
        t0 = time.time()
        rc = subprocess.call(common + extra, cwd=d, stdout=subprocess.DEVNULL)
        secs = time.time() - t0
        res[name] = {"rc": rc, "seconds": round(secs, 2), "mbp_per_s": round(bases / 1e6 / secs, 1)}
    import hashlib
    res["fa_identical"] = len({hashlib.sha256(open(os.path.join(d, x + ".fa"), "rb").read()).hexdigest() for x in "abc"}) == 1
    import shutil
    shutil.rmtree(d, ignore_errors=True)
    return res


def random_sector_peaks(ctx):
    """Random-32-byte-sector read peaks of this GPU, measured now (talc_bench_random_sectors, 4 GiB buffer): the
    independent-load peak bounds the coverage kernel's probes, the dependent-chain figure the walk's."""
    try:
        ind, _ = ctx.bench_random_sectors(4 << 30, dependent=False, warps_per_sm=64)
        dep, ns = ctx.bench_random_sectors(4 << 30, dependent=True, warps_per_sm=64)
        dep8, ns8 = ctx.bench_random_sectors(4 << 30, dependent=True, warps_per_sm=8)
        return {"dependent_8_warps_per_sm": {"gbs": dep8, "hop_ns": ns8,
                                             "note": "one dependent chain per thread at the correction kernel's residency "
                                                     "(8 warps per SM): hop_ns is the latency of one random sector"},"peak_random": ind, "peak_random_unit": "GB/s of uniformly random 32 B sectors over 4 GiB, 8 loads in flight per thread, 64 warps/SM",
                "peak_random_dependent": dep, "dependent_hop_ns": ns}
    except Exception as e:  # noqa: BLE001
        return {"peak_random": None, "peak_random_error": str(e)}


def cpu_baseline(args, cfg, cpu_keys, use_j, reads, roff, gpu):
    """The oracle port on this box's host cores, on a bounded sample of the same reads (rank 0, N=1 only), and the
    byte-for-byte comparison of its output with what the GPU produced for those very reads."""
    import numpy as np
    from oracle import pyoracle as po
    keys, counts, jk, jc = cpu_keys
    threads = os.cpu_count() or 1
    ot = po.OracleTable(po.make_params(k=cfg.k), ordered=False)
    ot.build_packed(keys.cpu().numpy().astype(np.uint64), counts.cpu().numpy(),
                    jk.cpu().numpy().astype(np.uint64) if use_j else None, jc.cpu().numpy() if use_j else None)
    n = min(args.cpu_sample_reads, args.batch_reads)
    sub = reads[: int(roff[n])].cpu().numpy()
    so = roff[: n + 1].cpu().numpy().astype(np.uint64)
    o_out, o_off, o_st, _, secs = ot.correct(sub, so, threads=threads)
    g_out, g_off, g_st = gpu
    mismatch = int((g_st[:n] != o_st[:n]).sum())
    if not np.array_equal(g_off[: n + 1], o_off[: n + 1]) or not np.array_equal(g_out[: int(o_off[n])], o_out[: int(o_off[n])]):
        for r in range(n):
            a = g_out[int(g_off[r]):int(g_off[r + 1])]
            b = o_out[int(o_off[r]):int(o_off[r + 1])]
            if len(a) != len(b) or not np.array_equal(a, b):
                mismatch += 1
    base = {"value": int(so[-1]) / 1e6 / secs, "unit": "Mbp/s", "cores": threads, "kind": "port",
            "sample": "first %d reads of the step-0 batch (%.2f Mbp), oracle restatement with a hashed table, %.1f s" % (
                n, int(so[-1]) / 1e6, secs)}
    parity = {"reads": n, "mismatch": mismatch,
              "what": "corrected bytes, offsets and status of the GPU for the first %d reads of the step-0 batch (full-size "
                      "table, full batch in flight) against the oracle" % n}
    return base, parity


_JSON_FD = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line.  Libraries underneath (NCCL's version banner -- torch's communicator and
    the library's own --, anything else that writes to fd 1 through C stdio) would add lines, so the process keeps a
    private duplicate of the real stdout for that line and points fd 1 at stderr for everything else."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        os.write(1, data)
    else:
        os.write(_JSON_FD, data)


def main():
    args = parse_args()
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
