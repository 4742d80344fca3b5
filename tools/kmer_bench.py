#!/usr/bin/env python3
"""Errors from k-mer counts on the GPU: kernel times, table size and load, and the whole k-mer path next to the
corrected-file path on the same reads.  Prints one JSON line (and writes it to --out).

    python tools/kmer_bench.py                      # 10 M x 150 bp, 30x of a 50 Mb genome, k = 23
    python tools/kmer_bench.py --cpu-only --reads 20000 --genome 100000 --oracle-reads 2000

Input: kbbq.synth.genome_reads (1 % substitutions).  GPU leg: the four device entry points on torch buffers, each
between CUDA events, --repeats times; then kbbq_recalibrate_kmer_host and kbbq_recalibrate_host (fed corrected reads
that differ at the bases the GPU flagged) by wall clock, host buffers in and out, twice each.  CPU leg: the C oracle
(tests/kmer_oracle.c, compiled into a temporary directory) on the first --oracle-reads reads.  --cpu-only stops before
the GPU leg.

--correct adds the correcting walk (DESIGN.md §10): kbbq_kmer_correct between CUDA events on the same table, the
precision and recall of both rules against the true errors, the whole path kbbq_recalibrate_kmer_rule_host with it,
and the table lookups per read the walk makes, counted by its oracle (tests/kmer_correct_oracle.c) on --oracle-reads
reads of a genome scaled to the same coverage.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "kbbq-py_b200"), os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", os.environ.get("KBBQ_DEVICE", "0")], capture_output=True, text=True, timeout=60)
        return out.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def quality(mask, err):
    tp = int((mask & err).sum())
    return dict(flagged=int(mask.sum()), precision=round(tp / max(1, int(mask.sum())), 6),
                recall=round(tp / max(1, int(err.sum())), 6))


def gpu_leg(args, seq, qual, err, second, res):
    import torch
    from kbbq import _native
    if not torch.cuda.is_available():
        raise SystemExit("the GPU leg needs a CUDA device (--cpu-only runs the rest)")
    lib = _native.lib()
    N, L, k = seq.shape[0], args.L, args.k
    res["card"] = card()
    res["torch_device"] = torch.cuda.get_device_name(0)
    cap, tbytes = _native.kmer_table_bytes(N, L, k)
    res.update(capacity=cap, table_bytes=tbytes)
    p = lambda t: C.c_void_p(t.data_ptr())
    d_seq = torch.from_numpy(seq.ravel()).cuda()
    table = torch.empty(2 * cap, dtype=torch.int64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    hist = torch.zeros(256, dtype=torch.int64, device="cuda")
    bits = torch.empty((N * L + 31) // 32, dtype=torch.int32, device="cuda")
    cbits = torch.empty_like(bits) if args.correct else None
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    times = {"clear": [], "count": [], "histogram": [], "flag": []}
    if args.correct:
        times["correct"] = []
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    t_used = None
    for _ in range(args.repeats):
        status.zero_()
        ev[0].record()
        _native.check(lib.kbbq_kmer_clear(p(table), cap, stream))
        ev[1].record()
        _native.check(lib.kbbq_kmer_count(p(d_seq), N, L, k, p(table), cap, p(status), stream))
        ev[2].record()
        _native.check(lib.kbbq_kmer_histogram(p(table), cap, p(hist), stream))
        ev[3].record()
        h = hist.cpu().numpy().astype(np.uint64)   # the threshold is taken on the host, as the entry points do
        t_used = args.min_count or _native.kmer_min_count(h)
        ev[3].record()
        _native.check(lib.kbbq_kmer_flag(p(d_seq), N, L, k, p(table), cap, t_used, p(bits), p(status), stream))
        ev[4].record()
        if args.correct:
            _native.check(lib.kbbq_kmer_correct(p(d_seq), N, L, k, p(table), cap, t_used, p(cbits), p(status), stream))
            ev[5].record()
        torch.cuda.synchronize()
        for name, a, b in (("clear", 0, 1), ("count", 1, 2), ("histogram", 2, 3), ("flag", 3, 4), ("correct", 4, 5)):
            if name in times:
                times[name].append(ev[a].elapsed_time(ev[b]))
        assert int(status.cpu()[0]) == 0, "k-mer table full"
    windows = N * max(0, L - k + 1)
    distinct = int(h.sum())
    load = distinct / cap
    # linear probing at load a: ~(1 + 1 / (1 - a)) / 2 slots per successful search, one random 32-byte sector each
    probes = 0.5 * (1 + 1 / (1 - load))
    best = {name: min(v) for name, v in times.items()}
    res.update(min_count_used=t_used, windows=windows, distinct_kmers=distinct, load_factor=round(load, 4),
               probes_per_window_model=round(probes, 3), kernel_ms={n: [round(x, 3) for x in v] for n, v in times.items()},
               count_windows_per_s=windows / (best["count"] / 1e3), flag_windows_per_s=windows / (best["flag"] / 1e3),
               count_sectors_per_s_model=windows * probes / (best["count"] / 1e3),
               flag_sectors_per_s_model=windows * probes / (best["flag"] / 1e3),
               table_bytes_per_s_clear=tbytes / (best["clear"] / 1e3),
               table_bytes_per_s_histogram=tbytes / (best["histogram"] / 1e3),
               flagged_bases=int(np.unpackbits(bits.cpu().numpy().view(np.uint8)).sum()))
    from kbbq.kmer import bits_to_mask
    mask = bits_to_mask(bits.cpu().numpy().view(np.uint32), N, L)
    if args.correct:
        cmask = bits_to_mask(cbits.cpu().numpy().view(np.uint32), N, L)
        res.update(correct_windows_per_s=windows / (best["correct"] / 1e3), boundaries_quality=quality(mask, err),
                   correct_quality=quality(cmask, err))
    del d_seq, table, status, hist, bits, cbits
    torch.cuda.empty_cache()

    wall_kmer, wall_corr = [], []
    out_k = out_c = None
    for _ in range(2):
        t0 = time.perf_counter()
        out_k, t = _native.recalibrate_kmer_host(seq, qual, None, second, L, 1, 6, k, args.min_count)
        wall_kmer.append(time.perf_counter() - t0)
    swap = np.arange(256, dtype=np.uint8)
    swap[[65, 67, 71, 84]] = [67, 65, 84, 71]
    corr = np.where(mask, swap[seq], seq)
    for _ in range(2):
        t0 = time.perf_counter()
        out_c = _native.recalibrate_host(seq, qual, corr, None, second, L, 1, 6)
        wall_corr.append(time.perf_counter() - t0)
    if args.correct:
        wall_walk = []
        for _ in range(2):
            t0 = time.perf_counter()
            out_w, _ = _native.recalibrate_kmer_host(seq, qual, None, second, L, 1, 6, k, args.min_count, correct=True)
            wall_walk.append(time.perf_counter() - t0)
        corr = np.where(cmask, swap[seq], seq)
        out_wc = _native.recalibrate_host(seq, qual, corr, None, second, L, 1, 6)
        res.update(recalibrate_kmer_correct_host_s=[round(x, 4) for x in wall_walk],
                   correct_same_qualities=bool(np.array_equal(out_w, out_wc)))
    _native.lib().kbbq_host_release(_native.DEVICE)
    res.update(recalibrate_kmer_host_s=[round(x, 4) for x in wall_kmer],
               recalibrate_host_corrected_s=[round(x, 4) for x in wall_corr],
               same_qualities=bool(np.array_equal(out_k, out_c)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--L", type=int, default=150)
    ap.add_argument("--genome", type=int, default=50_000_000)
    ap.add_argument("--k", type=int, default=23)
    ap.add_argument("--min-count", type=int, default=0)
    ap.add_argument("--sub-rate", type=float, default=0.01)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--oracle-reads", type=int, default=200_000)
    ap.add_argument("--cpu-only", action="store_true")
    ap.add_argument("--correct", action="store_true", help="add the correcting walk (kbbq_kmer_correct)")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not 1 <= args.k <= 31 or args.reads < 2 or args.L < 1 or args.min_count < 0 or args.repeats < 1:
        ap.error("need 1 <= k <= 31, reads >= 2, L >= 1, min-count >= 0, repeats >= 1")
    from kbbq import synth
    import kmer_oracle
    import kmer_correct_oracle
    res = dict(reads=args.reads, L=args.L, genome=args.genome, k=args.k, min_count=args.min_count,
               sub_rate=args.sub_rate, coverage=round(args.reads * args.L / args.genome, 2))
    t0 = time.perf_counter()
    seq, qual, err, second = synth.genome_reads(args.seed, args.genome, args.reads, args.L, args.sub_rate)
    res["generate_s"] = round(time.perf_counter() - t0, 2)

    n = min(args.oracle_reads, args.reads)
    t0 = time.perf_counter()
    bits, _, t = kmer_oracle.kmer_errors(seq[:n], args.L, args.k, args.min_count)
    dt = time.perf_counter() - t0
    res.update(oracle_reads=n, oracle_s=round(dt, 3), oracle_windows_per_s=n * max(0, args.L - args.k + 1) / dt,
               oracle_min_count_used=t)
    if args.correct:
        # the walk's lookups depend on coverage and error rate: count them on a genome scaled to --oracle-reads reads
        g = max(args.L, args.genome * n // args.reads)
        s_seq, _, _, _ = synth.genome_reads(args.seed + 1, g, n, args.L, args.sub_rate)
        look = kmer_correct_oracle.kmer_correct_lookups(s_seq, args.L, args.k, args.min_count)
        res.update(correct_lookups_per_read=round(look / n, 2), correct_lookups_genome=g,
                   flag_lookups_per_read=max(0, args.L - args.k + 1))
    if not args.cpu_only:
        gpu_leg(args, seq, qual, err, second, res)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
