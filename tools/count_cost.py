"""Cost of counting the k-mer table from short reads in each orientation, and of reading a canonical dump.

  (a) counting      talc_table_count_reads_oriented on a synthetic paired-end short-read set (FASTQ, 100 bp, 0.5 %
                    substitutions, about 10x over a random 'transcriptome' of --bases bases, so that about that many
                    distinct k-mers are on one strand: 30 M at the default, the size of bench configuration 2).  The
                    pairs are fr-firststrand (R1 antisense, R2 sense), so every mode below sees both strands and keeps
                    50 - 60 M k-mers.  Every file SENSE, every file ANTISENSE, every file BOTH: host clock around the
                    whole call (file read
                    from the page cache, copies, line scan, counting, final table and successor tables), input GB/s and
                    count increments/s; then count_kmers_kernel alone per mode (torch.profiler, CUDA activities, in a
                    run of its own after the timed calls).
  (b) old entry     talc_table_count_reads against talc_table_count_reads_oriented with every file SENSE, calls
                    alternated, same inputs: the two must be equal within run-to-run noise.
  (c) dump          talc_table_load_dump against talc_table_load_dump_ex(TALC_DUMP_CANONICAL) on the same canonical dump
                    of the transcriptome's k-mers, calls alternated.

Every mode's result is checked: the same (increments, distinct, kept) for both SENSE entries, ANTISENSE = SENSE, BOTH
increments = 2 x SENSE (K odd: no reverse palindromes).  The inputs (about 0.6 GB at the default) are written to a
temporary directory that is removed at the end; they are larger than the 126 MB L2, and the first call of each mode is
a warm-up.  Prints one JSON line; --out also writes it to a file.  Needs a CUDA device.

  python tools/count_cost.py [--bases 30000000] [--coverage 10] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip()


def write_fastq(path, seqs):
    """seqs: uint8 [n, L] ASCII; one FASTQ record per row, written in one piece"""
    import numpy as np
    n, L = seqs.shape
    head = b"@r\n"
    rec = np.empty((n, len(head) + L + 3 + L + 1), dtype=np.uint8)
    rec[:, :3] = np.frombuffer(head, dtype=np.uint8)
    rec[:, 3:3 + L] = seqs
    rec[:, 3 + L:6 + L] = np.frombuffer(b"\n+\n", dtype=np.uint8)
    rec[:, 6 + L:6 + 2 * L] = ord("I")
    rec[:, -1] = ord("\n")
    with open(path, "wb") as f:
        f.write(rec.tobytes())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bases", type=int, default=30_000_000, help="transcriptome size = distinct k-mers on one strand")
    ap.add_argument("--coverage", type=float, default=10.0)
    ap.add_argument("--read-len", type=int, default=100)
    ap.add_argument("--k", type=int, default=21)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    from talc_b200 import api
    if not torch.cuda.is_available():
        raise SystemExit("count_cost.py: no CUDA device -- k-mer counting has no CPU path")
    dev = "cuda:0"
    smi_before = smi()
    k, L = args.k, args.read_len
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    pool = torch.randint(0, 4, (args.bases,), generator=g, device=dev, dtype=torch.uint8)
    n_pairs = int(args.bases * args.coverage / (2 * L))
    letters = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    comp = torch.tensor(list(b"TGCA"), dtype=torch.uint8, device=dev)
    tmp = tempfile.mkdtemp(prefix="talc_count_cost_")
    try:
        paths = []
        for mate in (1, 2):  # R1 = reverse complement of a fragment end, R2 = sense (fr-firststrand)
            starts = torch.randint(0, args.bases - L, (n_pairs,), generator=g, device=dev)
            idx = starts[:, None] + torch.arange(L, device=dev)[None, :]
            codes = pool[idx]
            err = torch.rand(codes.shape, generator=g, device=dev) < 0.005
            codes = torch.where(err, torch.randint(0, 4, codes.shape, generator=g, device=dev, dtype=torch.uint8), codes)
            seqs = comp[codes.long()].flip(1) if mate == 1 else letters[codes.long()]
            p = os.path.join(tmp, "sr_%d.fq" % mate)
            write_fastq(p, seqs.cpu().numpy())
            paths.append(p)
            del idx, codes, err, seqs
        in_bytes = sum(os.path.getsize(p) for p in paths)
        windows = 2 * n_pairs * (L - k + 1)

        t = api.Talc(api.default_params(k))

        def timed(fn):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            return time.perf_counter() - t0, r

        # (a) + (b): warm-up of every mode, then rounds with the calls alternated
        modes = {"sense": [0, 0], "antisense": [1, 1], "both": [2, 2]}
        calls = {"old_entry": lambda: t.count_reads(paths)}
        for m, o in modes.items():
            calls[m] = (lambda o=o: t.count_reads(paths, o))
        res, secs = {}, {m: [] for m in calls}
        for m, fn in calls.items():
            res[m] = timed(fn)[1]
        for _ in range(args.rounds):
            for m, fn in calls.items():
                s, r = timed(fn)
                assert r == res[m], (m, r, res[m])
                secs[m].append(s)
        assert res["old_entry"] == res["sense"], "talc_table_count_reads differs from all-SENSE _oriented"
        assert res["antisense"] == res["sense"]
        assert res["sense"][0] == windows and res["both"][0] == 2 * windows  # no N; K odd: no reverse palindromes
        counting = {}
        for m in calls:
            med = statistics.median(secs[m])
            counting[m] = {"increments": res[m][0], "distinct": res[m][1], "kept": res[m][2], "call_s_median": med,
                           "call_s_min": min(secs[m]), "call_s_max": max(secs[m]), "call_s_all": secs[m],
                           "input_gbs": in_bytes / med / 1e9, "increments_per_s": res[m][0] / med}

        # (a) kernel alone, profiler on, after the timed calls
        from torch.profiler import ProfilerActivity, profile
        kern = {}
        for m, o in modes.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                t.count_reads(paths, o)
                torch.cuda.synchronize()
            tot, n = 0.0, 0
            for ev in prof.key_averages():
                if "count_kmers_kernel<" in ev.key:
                    us = getattr(ev, "device_time_total", None)
                    tot += us if us is not None else ev.cuda_time_total
                    n += ev.count
            ms = tot / 1e3
            kern[m] = {"kernel_ms_total": ms, "launches": n, "input_gbs": in_bytes / (ms * 1e-3) / 1e9 if ms else None,
                       "increments_per_s": res[m][0] / (ms * 1e-3) if ms else None}
            if not n:
                kern[m]["kernels_seen"] = [ev.key for ev in prof.key_averages()]

        # (c) one canonical dump of the transcriptome's k-mers (min(x, rc x)), loaded both ways, alternated
        kk = torch.zeros(args.bases - k + 1, dtype=torch.int64, device=dev)
        rr = torch.zeros_like(kk)
        b64 = pool.to(torch.int64)
        for j in range(k):
            kk = (kk << 2) | b64[j:args.bases - k + 1 + j]
            rr = rr | ((3 - b64[j:args.bases - k + 1 + j]) << (2 * j))
        can = torch.unique(torch.minimum(kk, rr))
        cnt = torch.randint(1, 40, (can.numel(),), generator=g, device=dev)
        perm = torch.randperm(can.numel(), generator=g, device=dev)
        dump = os.path.join(tmp, "can.dump")
        api.write_dump(dump, can[perm].cpu().numpy().astype(np.uint64), cnt[perm].cpu().numpy().astype(np.int64), k)
        del kk, rr, b64, can, cnt, perm
        d = api.Talc(api.default_params(k))
        dres, dsecs = {}, {"load_dump": [], "load_dump_ex_canonical": []}
        dcalls = {"load_dump": lambda: d.load_dump(dump), "load_dump_ex_canonical": lambda: d.load_dump(dump, canonical=True)}
        for m, fn in dcalls.items():
            dres[m] = timed(fn)[1]
        for _ in range(args.rounds):
            for m, fn in dcalls.items():
                s, r = timed(fn)
                assert r == dres[m]
                dsecs[m].append(s)
        dumpres = {m: {"lines": dres[m][0], "kept": dres[m][1], "call_s_median": statistics.median(dsecs[m]),
                       "call_s_min": min(dsecs[m]), "call_s_max": max(dsecs[m]), "call_s_all": dsecs[m]} for m in dcalls}
        smi_after = smi()
        line = {
            "metric": "k-mer counting from short reads per orientation; canonical dump loading",
            "counting": counting,
            "count_kmers_kernel": kern,
            "old_over_oriented_sense": counting["old_entry"]["call_s_median"] / counting["sense"]["call_s_median"],
            "dump": dumpres,
            "canonical_over_plain_dump": dumpres["load_dump_ex_canonical"]["call_s_median"] / dumpres["load_dump"]["call_s_median"],
            "workload": {"k": k, "transcriptome_bases": args.bases, "read_len": L, "pairs": n_pairs,
                         "files": 2, "input_bytes": in_bytes, "windows": windows, "substitution_rate": 0.005,
                         "dump_bytes": os.path.getsize(dump), "rounds": args.rounds,
                         "note": "calls alternated per round after one warm-up call each; inputs from the page cache"},
            "device": {"before": smi_before, "after": smi_after,
                       "fields": "name, power.limit, clocks.sm, clocks.max.sm, temperature.gpu"},
        }
        s = json.dumps(line)
        print(s)
        if args.out:
            with open(args.out, "w") as f:
                f.write(s + "\n")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
