#!/usr/bin/env python3
"""`kbbq recalibrate -r` streamed: the sieved k-mer table next to the exact one, and a batch the single-batch path
refuses.  Prints one JSON line (and writes it to --out).

    python tools/kmer_stream_bench.py                               # both legs below
    python tools/kmer_stream_bench.py --big-reads 0                 # the 10 M leg only

Leg 1, --reads (10 M) x 150 bp of kbbq.synth.genome_reads (--genome 50 Mb, 1 % substitutions), k = 23, where both
paths fit: the device entry points on torch buffers, each call between CUDA events (one run, summed over chunks) -- sieve,
count-present, sieved histogram, flag -- with the table and filter kbbq_kmer_stream_plan gives from the free memory;
the keys of the sieved table against those of the exact table (kbbq_kmer_count); then kbbq_recalibrate_kmer_host and
the streamed session (batches of --batch reads from memory) by wall clock, and whether their qualities are the same
bytes.  Leg 2, --big-reads (48 M) x 150 bp of a --big-genome (240 Mb, 30x) genome: the single-batch call's refusal,
the device passes chunk by chunk (precision and recall of the flags against genome_reads' true errors, and
sum c h[c] = W), then the whole streamed session by wall clock.  The big leg's reads are generated in seeded blocks
of 1 M reads on all host cores (blocks_reads: genome_reads' sampling, one genome, block b drawn from the seed and b);
the run holds seq, qual and the true error mask in host memory, 3 bytes per base (22 GB at 48 M x 150 bp).  The card's
name, power limit and clock come from nvidia-smi in the same run; each leg's results are written to --out as soon as
it ends.  --correct runs both legs with the correcting walk (kbbq_kmer_correct, DESIGN.md §10) in place of the
boundary rule: the device pass, the single-batch call and the session.

--devices 0,1,2,3 (lists separated by ';' run in turn, e.g. "0;0,1;0,1,2,3") runs the big leg with the table split
by key across those GPUs (DESIGN.md §10, "Several GPUs"): per pass, the kernel time on each device (CUDA events on its
stream) and the wall time; the load of each partition; the bytes copied between devices; the map on the first device
reading every partition (the correcting walk with --correct); then the streamed session over the same devices, and
whether its qualities equal the first list's.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "kbbq-py_b200"), os.path.join(ROOT, "tools")]
sys.dont_write_bytecode = True


_GENOME = None


def _block(args):
    """Reads [lo, hi) of blocks_reads: genome_reads' sampling on the shared genome, drawn from (seed, lo)."""
    seed, lo, hi, L, sub_rate = args
    genome = _GENOME
    rng = np.random.default_rng([seed, lo])
    n = hi - lo
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    second = (np.arange(lo, hi) & 1).astype(np.uint8)
    pair = np.arange(lo, hi) >> 1
    npairs = int(pair[-1] - pair[0] + 1)
    frag = rng.integers(L, 2 * L + 1, npairs)
    start = rng.integers(0, genome.size - frag + 1)
    frag, start = frag[pair - pair[0]], start[pair - pair[0]]
    is2 = second.astype(bool)
    first = np.where(is2, start + frag - L, start)
    codes = genome[first[:, None] + np.arange(L)[None, :]]
    codes[is2] = 3 - codes[is2][:, ::-1]
    e = rng.random((n, L)) < sub_rate
    codes = np.where(e, (codes + rng.integers(1, 4, (n, L), dtype=np.uint8)) & 3, codes)
    q = np.where(e, rng.integers(2, 21, (n, L)), rng.integers(25, 41, (n, L))).astype(np.uint8)
    return lo, acgt[codes], q, e, second


def blocks_reads(seed, genome_len, n_reads, L, sub_rate=0.01, block=1 << 20):
    """genome_reads' reads (pairs from both strands of one random genome, iid substitutions), generated in seeded
    blocks on every host core -> seq, qual, err, second."""
    import multiprocessing as mp
    global _GENOME
    _GENOME = np.random.default_rng(seed).integers(0, 4, genome_len, dtype=np.uint8)
    seq = np.empty((n_reads, L), np.uint8)
    qual = np.empty((n_reads, L), np.uint8)
    err = np.empty((n_reads, L), bool)
    second = np.empty(n_reads, np.uint8)
    jobs = [(seed, lo, min(n_reads, lo + block), L, sub_rate) for lo in range(0, n_reads, block)]
    with mp.get_context("fork").Pool(min(len(jobs), os.cpu_count() or 1)) as pool:
        for lo, s_, q_, e_, sec in pool.imap_unordered(_block, jobs):
            hi = lo + s_.shape[0]
            seq[lo:hi], qual[lo:hi], err[lo:hi], second[lo:hi] = s_, q_, e_, sec
    _GENOME = None
    return seq, qual, err, second


def write(res, path):
    line = json.dumps(res)
    if path:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            f.write(line + "\n")
    return line


def session_run(seq, qual, second, L, k, batch, correct=False, devices=None):
    """The streamed path from memory (kbbq_session_kmer_*; devices: the table split across them) -> (out, t, hist,
    (filter_words, capacity), seconds)"""
    from kbbq import _native
    n = seq.shape[0]
    rg = np.zeros(n, np.uint16)
    spans = [(lo, min(batch, n - lo)) for lo in range(0, n, batch)]
    secs = {}
    t0 = time.perf_counter()
    with _native.Session(L, 1, 6, chunk_reads=batch, resident_reads=0, device=devices[0] if devices else None) as s:
        s.kmer_begin(k, n * max(0, L - k + 1), devices=devices)
        if correct:
            s.kmer_rule(_native.KMER_CORRECT)
        sizes = s.kmer_sizes()
        s.flush()
        secs["begin"] = time.perf_counter() - t0
        for name, step in (("sieve", lambda lo, m: s.kmer_sieve(seq[lo:lo + m])),
                           ("count", lambda lo, m: s.kmer_count(seq[lo:lo + m]))):
            t1 = time.perf_counter()
            for lo, m in spans:
                step(lo, m)
            s.flush()
            secs[name] = time.perf_counter() - t1
        t1 = time.perf_counter()
        t, hist = s.kmer_threshold()
        secs["threshold"] = time.perf_counter() - t1
        t1 = time.perf_counter()
        for lo, m in spans:
            s.build_chunk_kmer(seq[lo:lo + m], qual[lo:lo + m], rg[lo:lo + m], second[lo:lo + m])
        s.model()
        s.flush()
        secs["build_and_model"] = time.perf_counter() - t1
        t1 = time.perf_counter()
        out = np.empty(seq.shape, np.uint8)
        for lo, m in spans:
            s.apply_chunk(seq[lo:lo + m], qual[lo:lo + m], rg[lo:lo + m], second[lo:lo + m], out[lo:lo + m])
        s.sync()
        secs["apply"] = time.perf_counter() - t1
    secs["total"] = time.perf_counter() - t0
    return out, t, hist, sizes, {k_: round(v, 3) for k_, v in secs.items()}


class Passes:
    """Sieve / count-present / histogram / flag on torch buffers, chunk by chunk, timed with CUDA events."""

    def __init__(self, L, k, windows, correct=False):
        import torch
        from kbbq import _native
        self.torch, self.native, self.lib = torch, _native, _native.lib()
        self.L, self.k, self.correct = L, k, correct
        free, _ = torch.cuda.mem_get_info()
        self.F, self.cap = _native.kmer_stream_plan(windows, int(0.8 * free))
        self.filter = torch.zeros(self.F, dtype=torch.int64, device="cuda")
        self.table = torch.empty(2 * self.cap, dtype=torch.int64, device="cuda")
        self.status = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.windows = torch.zeros(1, dtype=torch.int64, device="cuda")
        self.hist = torch.zeros(256, dtype=torch.int64, device="cuda")
        self.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.ms = {"clear": 0.0, "sieve": 0.0, "count_present": 0.0, "histogram": 0.0,
                   "correct" if correct else "flag": 0.0}
        self.timed("clear", lambda: self.lib.kbbq_kmer_clear(self.p(self.table), self.cap, self.stream))

    def p(self, t):
        return C.c_void_p(t.data_ptr())

    def timed(self, name, call):
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        e0.record()
        self.native.check(call())
        e1.record()
        e1.synchronize()
        self.ms[name] += e0.elapsed_time(e1)

    def sieve(self, d_seq, n):
        self.timed("sieve", lambda: self.lib.kbbq_kmer_sieve(self.p(d_seq), n, self.L, self.k, self.p(self.filter), self.F,
                                                             self.p(self.table), self.cap, self.p(self.status), self.stream))

    def count(self, d_seq, n):
        self.timed("count_present", lambda: self.lib.kbbq_kmer_count_present(
            self.p(d_seq), n, self.L, self.k, self.p(self.table), self.cap, self.p(self.windows), self.p(self.status),
            self.stream))

    def histogram(self):
        self.timed("histogram", lambda: self.lib.kbbq_kmer_histogram_sieved(self.p(self.table), self.cap,
                                                                            self.p(self.windows), self.p(self.hist),
                                                                            self.stream))
        return self.hist.cpu().numpy().astype(np.uint64)

    def flag(self, d_seq, n, t, bits):
        fn = self.lib.kbbq_kmer_correct if self.correct else self.lib.kbbq_kmer_flag_sieved
        self.timed("correct" if self.correct else "flag",
                   lambda: fn(self.p(d_seq), n, self.L, self.k, self.p(self.table), self.cap, t, self.p(bits),
                              self.p(self.status), self.stream))

    def table_stats(self):
        """-> (keys in the table, of which count 1), a slice of slots at a time"""
        slots = self.table.view(-1, 2)
        keys = ones = 0
        for lo in range(0, self.cap, 1 << 28):
            s = slots[lo:lo + (1 << 28)]
            occupied = s[:, 0] != -1
            keys += int(occupied.sum())
            ones += int((occupied & (s[:, 1] == 1)).sum())
        return keys, ones


def run_passes(seq, L, k, chunk, err=None, correct=False):
    """The four passes over seq in chunks of `chunk` reads -> dict of results (and flags checked against err)."""
    import torch
    from kbbq.kmer import bits_to_mask
    n = seq.shape[0]
    W = n * max(0, L - k + 1)
    ps = Passes(L, k, W, correct)
    spans = [(lo, min(chunk, n - lo)) for lo in range(0, n, chunk)]
    for step in (ps.sieve, ps.count):
        for lo, m in spans:
            d = torch.from_numpy(seq[lo:lo + m].ravel()).cuda()
            step(d, m)
            del d
    hist = ps.histogram()
    t = ps.native.kmer_min_count(hist)
    keys, ones = ps.table_stats()
    res = dict(filter_words=ps.F, filter_bytes=8 * ps.F, capacity=ps.cap, table_bytes=16 * ps.cap, min_count_used=t,
               windows_valid=int(ps.windows.cpu()[0]), sum_c_hist=int(sum(c * int(hist[c]) for c in range(1, 256))),
               sieved_keys=keys, sieved_keys_count1=ones, distinct_keys=int(hist.sum()), singletons=int(hist[1]),
               false_positive_share=round(ones / max(1, int(hist[1])), 5))
    tp = flagged = errors = 0
    bits = torch.empty((chunk * L + 31) // 32 + 1, dtype=torch.int32, device="cuda")
    for lo, m in spans:
        d = torch.from_numpy(seq[lo:lo + m].ravel()).cuda()
        ps.flag(d, m, t, bits)
        if err is not None:
            got = bits_to_mask(bits.cpu().numpy().view(np.uint32), m, L)
            e = err[lo:lo + m]
            tp += int((got & e).sum())
            flagged += int(got.sum())
            errors += int(e.sum())
        del d
    res["status"] = int(ps.status.cpu()[0])
    res["pass_ms"] = {name: round(v, 2) for name, v in ps.ms.items()}
    if err is not None:
        res.update(flagged=flagged, precision=round(tp / max(1, flagged), 5), recall=round(tp / max(1, errors), 4))
    del ps
    torch.cuda.empty_cache()
    return res


class PartPasses:
    """Passes A and B of a table split across `devices` (kbbq_kmer_sieve_part / _count_present_part), the sieved
    histogram of each partition and the map (kbbq_kmer_flag_parts / _correct_parts) on devices[0], on torch buffers.
    Each partition has its own stream on its device; every chunk goes up to devices[0] and is copied to each other
    partition, as the session does.  Kernel time per device from CUDA events on its stream; wall time per pass from
    the host clock around the pass, which ends when every stream is done."""

    def __init__(self, L, k, windows, devices, correct=False):
        import torch
        from kbbq import _native
        self.torch, self.native, self.lib = torch, _native, _native.lib()
        self.L, self.k, self.correct, self.devices = L, k, correct, devices
        n = len(devices)
        budget = None
        for d in devices:   # as kbbq_session_kmer_begin_parts sizes them
            free, _ = torch.cuda.mem_get_info(d)
            b = 0.8 * free / devices.count(d)
            budget = b if budget is None else min(budget, b)
        self.F, self.cap = _native.kmer_stream_plan(-(-windows // n), int(budget))
        self.cap = min(self.cap, 1 << 32) if n > 1 else self.cap
        self.parts = []
        for d in devices:
            with torch.cuda.device(d):
                self.parts.append(dict(
                    device=d, stream=torch.cuda.Stream(d),
                    filter=torch.zeros(self.F, dtype=torch.int64, device=d),
                    table=torch.empty(2 * self.cap, dtype=torch.int64, device=d),
                    status=torch.zeros(1, dtype=torch.int32, device=d),
                    windows=torch.zeros(1, dtype=torch.int64, device=d),
                    hist=torch.zeros(256, dtype=torch.int64, device=d)))
        self.kernel_ms = {}   # pass -> per-partition milliseconds
        self.wall_ms = {}
        self.peer_bytes = 0
        self.timed_pass("clear", lambda q, p, d_seq, n_: self.lib.kbbq_kmer_clear(self.p(p["table"]), self.cap,
                                                                                   self.st(p)), [None])

    def p(self, t):
        return C.c_void_p(t.data_ptr())

    def st(self, part):
        return C.c_void_p(part["stream"].cuda_stream)

    def timed_pass(self, name, call, chunks):
        """call(q, part, d_seq, n) for every chunk (a device tensor of n reads on devices[0], or None) and partition"""
        torch = self.torch
        ms = self.kernel_ms.setdefault(name, [0.0] * len(self.parts))
        t0 = time.perf_counter()
        for chunk in chunks:
            d0, n = chunk if chunk is not None else (None, 0)
            ready = torch.cuda.Event()
            if d0 is not None:
                with torch.cuda.device(self.devices[0]):
                    ready.record(torch.cuda.current_stream(self.devices[0]))
            for q, part in enumerate(self.parts):
                with torch.cuda.device(part["device"]), torch.cuda.stream(part["stream"]):
                    part["stream"].wait_event(ready)
                    d = d0
                    if d0 is not None and q > 0:   # a copy even on the same device, as the session makes
                        d = torch.empty_like(d0, device=part["device"])
                        d.copy_(d0, non_blocking=True)
                        self.peer_bytes += d0.numel()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(part["stream"])
                    self.native.check(call(q, part, d, n))
                    e1.record(part["stream"])
                    part.setdefault("events", []).append((e0, e1))
                    if d is not None:
                        d.record_stream(part["stream"])
        for q, part in enumerate(self.parts):
            part["stream"].synchronize()
            ms[q] += sum(a.elapsed_time(b) for a, b in part.pop("events", []))
        self.wall_ms[name] = self.wall_ms.get(name, 0.0) + 1000 * (time.perf_counter() - t0)

    def sieve(self, chunks):
        n_parts = len(self.parts)
        self.timed_pass("sieve", lambda q, p, d, n: self.lib.kbbq_kmer_sieve_part(
            self.p(d), n, self.L, self.k, q, n_parts, self.p(p["filter"]), self.F, self.p(p["table"]), self.cap,
            self.p(p["status"]), self.st(p)), chunks)

    def count(self, chunks):
        n_parts = len(self.parts)
        self.timed_pass("count_present", lambda q, p, d, n: self.lib.kbbq_kmer_count_present_part(
            self.p(d), n, self.L, self.k, q, n_parts, self.p(p["table"]), self.cap, self.p(p["windows"]),
            self.p(p["status"]), self.st(p)), chunks)

    def histogram(self):
        self.timed_pass("histogram", lambda q, p, d, n: self.lib.kbbq_kmer_histogram_sieved(
            self.p(p["table"]), self.cap, self.p(p["windows"]), self.p(p["hist"]), self.st(p)), [None])
        return sum(p["hist"].cpu().numpy().astype(np.uint64) for p in self.parts)

    def flag(self, d_seq, n, t, bits):
        """the map on devices[0] only: one timed call"""
        torch = self.torch
        fn = self.lib.kbbq_kmer_correct_parts if self.correct else self.lib.kbbq_kmer_flag_parts
        tables = (C.c_void_p * len(self.parts))(*[p["table"].data_ptr() for p in self.parts])
        p0 = self.parts[0]
        name = "correct" if self.correct else "flag"
        with torch.cuda.device(p0["device"]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record(p0["stream"])
            self.native.check(fn(self.p(d_seq), n, self.L, self.k, tables, len(self.parts), self.cap, t, self.p(bits),
                                 self.p(p0["status"]), self.st(p0)))
            e1.record(p0["stream"])
            e1.synchronize()
        self.kernel_ms.setdefault(name, [0.0])[0] += e0.elapsed_time(e1)
        self.wall_ms[name] = self.wall_ms.get(name, 0.0) + 1000 * (time.perf_counter() - t0)

    def loads(self):
        """share of occupied slots of each partition, a slice of slots at a time"""
        out = []
        for p in self.parts:
            keys = p["table"].view(-1, 2)[:, 0]
            out.append(round(sum(int((keys[lo:lo + (1 << 28)] != -1).sum()) for lo in range(0, self.cap, 1 << 28))
                             / self.cap, 4))
        return out


def run_parts(seq, L, k, chunk, devices, err=None, correct=False):
    """The passes of a table split across `devices` over seq in chunks of `chunk` reads -> dict of results."""
    import torch
    from kbbq.kmer import bits_to_mask
    n = seq.shape[0]
    ps = PartPasses(L, k, n * max(0, L - k + 1), devices, correct)
    spans = [(lo, min(chunk, n - lo)) for lo in range(0, n, chunk)]
    for step in (ps.sieve, ps.count):
        for lo, m in spans:   # one chunk on the device at a time, as the session holds it
            with torch.cuda.device(devices[0]):
                d = torch.from_numpy(seq[lo:lo + m].ravel()).to(devices[0])
            step([(d, m)])
            del d
    hist = ps.histogram()
    t = ps.native.kmer_min_count(hist)
    res = dict(devices=devices, filter_words=ps.F, capacity=ps.cap, table_bytes_each=16 * ps.cap, min_count_used=t,
               partition_load=ps.loads(), windows_valid=int(sum(int(p["windows"].cpu()[0]) for p in ps.parts)),
               sum_c_hist=int(sum(c * int(hist[c]) for c in range(1, 256))))
    tp = flagged = errors = 0
    with torch.cuda.device(devices[0]):
        bits = torch.empty((chunk * L + 31) // 32 + 1, dtype=torch.int32, device=devices[0])
        for lo, m in spans:
            d = torch.from_numpy(seq[lo:lo + m].ravel()).to(devices[0])
            ps.flag(d, m, t, bits)
            if err is not None:
                got = bits_to_mask(bits.cpu().numpy().view(np.uint32), m, L)
                e = err[lo:lo + m]
                tp += int((got & e).sum())
                flagged += int(got.sum())
                errors += int(e.sum())
            del d
    res["status"] = [int(p["status"].cpu()[0]) for p in ps.parts]
    res["kernel_ms"] = {name: [round(v, 2) for v in ms] for name, ms in ps.kernel_ms.items()}
    res["wall_ms"] = {name: round(v, 2) for name, v in ps.wall_ms.items()}
    res["bytes_between_devices"] = ps.peer_bytes
    if err is not None:
        res.update(flagged=flagged, precision=round(tp / max(1, flagged), 5), recall=round(tp / max(1, errors), 4))
    del ps, bits
    torch.cuda.empty_cache()
    return res


def exact_keys(seq, L, k):
    """Distinct keys of the exact table (kbbq_kmer_count) of the whole batch."""
    import torch
    from kbbq import _native
    lib = _native.lib()
    n = seq.shape[0]
    cap = _native.kmer_table_bytes(n, L, k)[0]
    d = torch.from_numpy(seq.ravel()).cuda()
    table = torch.empty(2 * cap, dtype=torch.int64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())
    _native.check(lib.kbbq_kmer_clear(p(table), cap, st))
    _native.check(lib.kbbq_kmer_count(p(d), n, L, k, p(table), cap, p(status), st))
    keys = int((table.view(-1, 2)[:, 0] != -1).sum())
    del d, table
    torch.cuda.empty_cache()
    return cap, keys


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--genome", type=int, default=50_000_000)
    ap.add_argument("--big-reads", type=int, default=48_000_000)
    ap.add_argument("--big-genome", type=int, default=240_000_000)
    ap.add_argument("--L", type=int, default=150)
    ap.add_argument("--k", type=int, default=23)
    ap.add_argument("--batch", type=int, default=8_000_000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--correct", action="store_true", help="the correcting walk in place of the boundary rule")
    ap.add_argument("--devices", help="the table split across these GPUs, e.g. 0,1,2,3; lists separated by ';' run in "
                                      "turn; only the --big-reads leg runs")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    from kbbq import _native, synth
    from kmer_bench import card
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    L, k = args.L, args.k
    res = dict(card=card(), torch_device=torch.cuda.get_device_name(0), L=L, k=k, batch=args.batch,
               rule="correct" if args.correct else "boundaries")
    opt = {"correct": True} if args.correct else {}
    if args.devices:
        return devices_leg(args, res)

    t0 = time.perf_counter()
    seq, qual, err, second = synth.genome_reads(args.seed, args.genome, args.reads, L, 0.01)
    leg = dict(reads=args.reads, genome=args.genome, generate_s=round(time.perf_counter() - t0, 1))
    leg["exact_capacity"], leg["exact_keys"] = exact_keys(seq, L, k)
    leg.update(run_passes(seq, L, k, args.reads, err, args.correct))
    t0 = time.perf_counter()
    out_single, t_single = _native.recalibrate_kmer_host(seq, qual, None, second, L, 1, 6, k, **opt)
    leg["single_batch_s"] = round(time.perf_counter() - t0, 3)
    _native.lib().kbbq_host_release(_native.DEVICE)
    out_stream, t_stream, _, sizes, secs = session_run(seq, qual, second, L, k, args.batch, args.correct)
    leg.update(streamed_s=secs, streamed_sizes=sizes, same_threshold=t_single == t_stream,
               same_qualities=bool(np.array_equal(out_single, out_stream)))
    res["leg_10m"] = leg
    write(res, args.out)
    del seq, qual, err, second, out_single, out_stream

    if args.big_reads:
        t0 = time.perf_counter()
        seq, qual, err, second = blocks_reads(args.seed + 1, args.big_genome, args.big_reads, L, 0.01)
        leg = dict(reads=args.big_reads, genome=args.big_genome, generate_s=round(time.perf_counter() - t0, 1),
                   exact_rule_bytes=_native.kmer_table_bytes(args.big_reads, L, k)[1])
        try:
            _native.recalibrate_kmer_host(seq, qual, None, second, L, 1, 6, k, **opt)
            leg["single_batch"] = "ran"
        except _native.DoesNotFit as e:
            leg["single_batch"] = "refused: %s" % e
        leg.update(run_passes(seq, L, k, args.batch, err, args.correct))
        out, t, hist, sizes, secs = session_run(seq, qual, second, L, k, args.batch, args.correct)
        leg.update(streamed_s=secs, streamed_sizes=sizes, streamed_min_count=t,
                   streamed_sum_c_hist=int(sum(c * int(hist[c]) for c in range(1, 256))),
                   streamed_hist_255=int(hist[255]), windows=args.big_reads * max(0, L - k + 1), changed_qualities=int((out != qual).sum()))
        res["leg_48m"] = leg
    print(write(res, args.out))


def devices_leg(args, res):
    """The --big-reads leg with the table split across each device list of --devices: the passes on the device entry
    points (run_parts), then the streamed session; its qualities against those of the first list's session."""
    L, k = args.L, args.k
    t0 = time.perf_counter()
    seq, qual, err, second = blocks_reads(args.seed + 1, args.big_genome, args.big_reads, L, 0.01)
    res.update(reads=args.big_reads, genome=args.big_genome, generate_s=round(time.perf_counter() - t0, 1), legs=[])
    first = None
    for spec in args.devices.split(";"):
        devices = [int(x) for x in spec.split(",")]
        leg = run_parts(seq, L, k, args.batch, devices, err, args.correct)
        out, t, hist, sizes, secs = session_run(seq, qual, second, L, k, args.batch, args.correct, devices)
        first = out if first is None else first
        leg.update(streamed_s=secs, streamed_sizes=sizes, streamed_min_count=t,
                   same_qualities_as_first=bool(np.array_equal(out, first)))
        del out
        res["legs"].append(leg)
        write(res, args.out)
    print(write(res, args.out))


if __name__ == "__main__":
    main()
