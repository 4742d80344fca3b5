#!/usr/bin/env python3
"""bench.py -- throughput of the kbbq recalibration hot path (table build + model + apply).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--reads n --read-len L --read-groups R] [--layout auto|segmented|read-order]
                    [--scaling weak|strong --total-reads T] [--stream-batch B] [--dump-outputs DIR]

Metric (BASELINE.json): bases/sec recalibrated (table build + apply).  Workload:
  N = 1   BASELINE config 2: synthetic 10 M x 150 bp interleaved pairs, 1 read group, Q2-Q41, 1 % mismatches
  N > 1   BASELINE config 3: 100 M x 2 x 150 bp pairs, 8 read groups, sharded over 8 GPUs = 25 M reads per GPU
          (weak scaling: every rank holds its own 25 M-read shard of one global counter-based stream);
          --scaling strong splits --total-reads (default 200 M) over the ranks instead
`--reads / --read-len / --read-groups` select any other shape; config.workload always names what ran.

One step = one pass of the hot path over the batch resident in HBM: zero tables -> build -> (N > 1: ONE int64
all-reduce of the tables over NCCL) -> marginals + delta-Q model -> apply.  With several read groups the batch
is resident in the product's segmented layout (rows sorted by read group and mate, include/kbbq_b200.h), which
the host-buffer entry points produce on the device behind the PCIe copies; the same step on rows in read order
with rg[] per read (work-list gather) is measured next to it (`layouts`).  `e2e` is the pass through the
reference-facing host-buffer API from pinned host memory, copies (and the segmentation) inside the timed
region: kbbq_recalibrate_host at N = 1, kbbq.parallel.recalibrate_host_distributed (one session per rank, the
same all-reduce) at N > 1.  Batches (>= 4.5 GB in) are far larger than the 126 MB L2: no explicit flush.

At N = 1 the line also carries `configs` (BASELINE configs 3, 4 and 5 at full per-GPU size, measured after the
main timed region), `e2e_fastq` (FASTQ files on /dev/shm -> recalibrated FASTQ through
kbbq.recalibrate.recalibrate_fastq) and `cpu_baseline`; at N > 1 `parity_n` (rank 0 rebuilds every shard alone
and compares tables and output checksums with the N-rank result, outside the timed region).

`--impl reference` times the CPU restatement of the reference's algorithm (oracle/, all host threads) on a
bounded sample of the same workload; the Python reference itself is pure Python, cannot travel to the GPU box
and runs at ~0.26 Mbases/s/core (tools/reference_speed.py).

`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy (see dump_outputs): the inputs
are a pure function of the arguments, so two builds of the project can be compared output for output.

The benchmark runs from the tree as it was built and writes nothing there (no bytecode, no compiling).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

sys.dont_write_bytecode = True   # the tree may be read-only: leave no __pycache__ behind in it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "kbbq-py_b200"))

METRIC = "bases/sec recalibrated (table build + apply)"
UNIT = "bases/s"
ALGO_BYTES_BUILD = 3  # seq + qual + corrected read, per base
ALGO_BYTES_APPLY = 3  # seq + qual read, new qual written, per base
DTYPE = "u8 in/out, u32->int64 counts, f64 model"

# BASELINE.json configs (SURVEY.md section 8d): per-GPU shape and the seed of the counter-based stream
CONFIGS = {
    2: {"reads": 10_000_000, "read_len": 150, "read_groups": 1, "seed": 1002,
        "name": "BASELINE config 2: synthetic 10 M x 150 bp interleaved pairs, 1 read group"},
    3: {"reads": 25_000_000, "read_len": 150, "read_groups": 8, "seed": 1003,
        "name": "BASELINE config 3: synthetic 100 M x 2 x 150 bp pairs, 8 read groups, sharded over 8 GPUs (25 M reads per GPU)"},
    4: {"reads": 20_000_000, "read_len": 250, "read_groups": 32, "seed": 1004,
        "name": "BASELINE config 4: synthetic 20 M x 250 bp reads, 32 read groups"},
    5: {"reads": 500_000_000, "read_len": 150, "read_groups": 1, "seed": 1005, "batch": 32_000_000,
        "name": "BASELINE config 5: synthetic 500 M x 150 bp reads streamed in batches of 32 M"},
}


class Workload:
    def __init__(self, reads, L, R, seed, label, config=None):
        self.N, self.L, self.R, self.seed, self.label, self.config = reads, L, R, seed, label, config

    def describe(self, per="per GPU"):
        return "%s -- %d x %d bp reads %s, %d read group(s), Q2-Q41, 1%% mismatches, seed %d" % (
            self.label, self.N, self.L, per, self.R, self.seed)


def resolve_workload(args, world):
    """The workload of this run: an explicit shape, else config 2 on one GPU and config 3's shard on several."""
    explicit = args.reads is not None or args.read_len is not None or args.read_groups is not None
    base = CONFIGS[2 if world == 1 and args.scaling == "weak" else 3]   # strong scaling is config 3 at any N
    if args.stream_batch > 0 and not explicit:
        base = CONFIGS[5]
    N = args.reads if args.reads is not None else base["reads"]
    L = args.read_len if args.read_len is not None else base["read_len"]
    R = args.read_groups if args.read_groups is not None else base["read_groups"]
    if args.scaling == "strong":
        N = (args.total_reads // world) // 16 * 16
    cfg = None
    for k, c in CONFIGS.items():
        if (N, L, R) == (c["reads"], c["read_len"], c["read_groups"]) and (k != 5 or args.stream_batch > 0):
            cfg = k
    if cfg is not None:
        label = CONFIGS[cfg]["name"]
    elif args.scaling == "strong" and (L, R) == (150, 8):
        label = "BASELINE config 3 (strong scaling: %d reads in total split over %d GPU(s))" % (args.total_reads, world)
    else:
        label = "custom shape (not a BASELINE config)"
    seed = CONFIGS[cfg]["seed"] if cfg is not None else (1003 if R > 1 else 1002)
    return Workload(N, L, R, seed, label, cfg)


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML from a background thread (one
    sample per millisecond: the timed region is tens of milliseconds long), nvidia-smi -lms as fallback."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index):
        import threading
        self.proc, self.thread, self.stop_flag = None, None, threading.Event()
        self.sm, self.bits, self.smax, self.how = [], 0, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
            except Exception:
                pass
            handle = None
            if uuid:
                try:
                    handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
                except Exception:
                    handle = None
            if handle is None:
                handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM))
            reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self.stop_flag.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)))
                        self.bits |= int(reasons(handle))
                    except Exception:
                        pass
                    time.sleep(0.001)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.how = "nvml"
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.how = "nvidia-smi"
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            reasons = sorted(k for k, bit in self.REASONS.items() if self.bits & bit)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.smax,
                    "samples": len(self.sm), "reasons": reasons, "source": "nvml, 1 ms period, timed loops only"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


def cpu_port_throughput(n_reads, L, R, seed, target_s, threads=0):
    """Oracle (CPU port of the reference algorithm) on a bounded sample -> (bases/s, sample description)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle   # loads the libkbbq_oracle.so the build made; nothing is compiled here
    from kbbq import synth
    # every hardware thread this process may run on; torchrun exports OMP_NUM_THREADS=1 to its workers, which
    # omp_get_max_threads() would obey, so the count is passed explicitly (omp_set_num_threads in the oracle)
    threads = threads or len(os.sched_getaffinity(0)) or oracle.max_threads()
    probe = min(n_reads, 100_000)
    data = synth.synth_reads(seed, 0, probe, L, R)
    t0 = time.perf_counter()
    oracle.recalibrate(*data, L, R, threads=threads)
    rate = probe * L / max(time.perf_counter() - t0, 1e-6)
    sample = int(min(n_reads, max(probe, rate * target_s / L)))
    sample = min(sample, 4_000_000)  # bound host memory of the numpy generator
    if sample > probe:
        data = synth.synth_reads(seed, 0, sample, L, R)
    return oracle, data, sample, threads



def bind_to_gpu_cpus(gpu_index):
    """Several ranks on one host: run this rank (and first-touch its pinned buffers) on the CPUs NVML names
    as local to its GPU, so that the end-to-end copies do not cross sockets.  Returns the CPU count or None."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus and len(cpus) < len(os.sched_getaffinity(0)):
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None




def run_reference(args):
    """--impl reference: CPU restatement of the reference algorithm on the host cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = resolve_workload(args, world)
    L, R = wl.L, wl.R
    per_step = max(1.0, min(6.0, 150.0 / (args.steps + args.warmup)))
    oracle, data, sample, threads = cpu_port_throughput(wl.N, L, R, wl.seed, per_step)
    for _ in range(args.warmup):
        oracle.recalibrate(*data, L, R, threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle.recalibrate(*data, L, R, threads=threads)
    dt = time.perf_counter() - t0
    value = sample * L * args.steps / dt
    desc = "first %d reads x %d bp of the workload per step (oracle/kbbq_oracle.c, OpenMP)" % (sample, L)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int64/u8 (+f64/f80 model)",
        "data": "synthetic",
        "config": {"workload": wl.describe() + " (CPU arm: bounded sample)", "reads_per_step": sample, "read_len": L,
                   "read_groups": R, "seed": wl.seed},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "CPU port of the reference algorithm, not a tuned one (its table merge is a critical section and its "
                "delta step serial: 16 -> 32 threads gains nothing); the reference itself is pure Python, ~0.26 "
                "Mbases/s on one core (tools/reference_speed.py); host arrays in, host arrays out, no FASTQ parsing",
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# the hot path on a batch resident in HBM
# ------------------------------------------------------------------------------------------------------------

class HotPath:
    """One shard resident in HBM + the step over it.  layout "segmented": rows sorted by (read group, mate), the
    product's HBM layout with several read groups; "read-order": rows as the host has them, rg[] per read."""

    def __init__(self, wl, dev, first_read, layout):
        import torch
        from kbbq.device import DeviceRecalibrator, synth_reads
        self.torch, self.wl, self.dev, self.layout = torch, wl, dev, layout
        N, L, R = wl.N, wl.L, wl.R
        self.seq, self.qual, self.corr, self.rg, self.second = synth_reads(wl.seed, first_read, N, L, R, device=dev)
        self.rg_arg = self.rg if R > 1 else None
        self.rec = DeviceRecalibrator(L, R, max_reads=N + 64 * R, device=dev)
        self.sb = None
        if layout == "segmented":
            self.sb = self.rec.segment(self.seq, self.qual, self.corr, self.rg_arg, self.second)
            self.out = torch.empty(self.sb.rows_bound * L + 16, dtype=torch.uint8, device=dev)
            self.rec.check_status()
        else:
            self.out = torch.empty_like(self.qual)

    def drop_read_order_inputs(self):
        """segmented layout: the hot path no longer needs the arrays in read order"""
        self.corr = None

    def build(self):
        if self.sb is not None:
            self.rec.build_segmented(self.sb)
        else:
            self.rec.build(self.seq, self.qual, self.corr, self.rg_arg, self.second)

    def apply(self):
        if self.sb is not None:
            self.rec.apply_segmented(self.sb, self.out)
        else:
            self.rec.apply(self.seq, self.qual, self.out, self.rg_arg, self.second)

    def output_in_read_order(self):
        if self.sb is None:
            return self.out
        o = self.torch.empty_like(self.qual)
        self.rec.unsegment(self.sb, self.out, o)
        return o

    def step(self, ev=None):
        rec = self.rec
        rec.tables.zero_()
        if ev:
            ev[0].record()
        self.build()
        if ev:
            ev[1].record()
        rec.allreduce()
        rec.model()
        if ev:
            ev[2].record()
        self.apply()
        if ev:
            ev[3].record()


def time_hot_path(hp, K, W, world, barrier, use_graph=True, sampler_factory=None):
    """W warm-up steps, K timed steps (CUDA events, max over ranks), eager with per-phase events and -- the figure
    reported -- replayed from two CUDA graphs around the eager all-reduce.  Returns a dict."""
    import torch
    from kbbq import _native, parallel
    lib = _native.lib()
    dev, rec = hp.dev, hp.rec
    for _ in range(W):
        hp.step()
    rec.check_status()
    barrier()
    sampler = sampler_factory() if sampler_factory else None
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = lib.kbbq_launch_count()
    barrier()
    t0.record()
    for k in range(K):
        hp.step(evs[k])
    t1.record()
    barrier()
    launches = lib.kbbq_launch_count() - launches0
    eager_ms = parallel.max_over_ranks(t0.elapsed_time(t1), dev)
    graph_ms = None
    eager_phases = None
    if use_graph:
        # the collective stays outside the captures (NCCL inside a capture hung on this pool): one graph up to the
        # build, the eager all-reduce, one graph from the model on
        g1 = g2 = g3 = None
        try:
            g1, g2, g3 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1):
                rec.tables.zero_()
                hp.build()
            with torch.cuda.graph(g2):
                rec.model()
            with torch.cuda.graph(g3):
                hp.apply()
            torch.cuda.synchronize()
        except Exception as exc:  # capture not possible: the eager figure stands
            sys.stderr.write("bench.py: CUDA graph capture failed (%r); reporting the eager loop\n" % (exc,))
            g1 = g2 = g3 = None

        def replay(ev=None):
            if ev:
                ev[0].record()
            g1.replay()
            if ev:
                ev[1].record()
            rec.allreduce()
            g2.replay()
            if ev:
                ev[2].record()
            g3.replay()
            if ev:
                ev[3].record()

        if parallel.max_over_ranks(0.0 if g1 is not None else 1.0, dev) == 0.0:   # every rank replays or none does
            for _ in range(W):
                replay()
            barrier()
            gevs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
            t0.record()
            for k in range(K):
                replay(gevs[k])
            t1.record()
            barrier()
            graph_ms = parallel.max_over_ranks(t0.elapsed_time(t1), dev)
            rec.check_status()
            eager_phases = {"build_ms": statistics.mean(e[0].elapsed_time(e[1]) for e in evs),
                            "model_ms": statistics.mean(e[1].elapsed_time(e[2]) for e in evs),
                            "apply_ms": statistics.mean(e[2].elapsed_time(e[3]) for e in evs)}
            evs = gevs   # the per-phase times reported are those of the loop `value` comes from
    clocks = sampler.stop() if sampler else None   # sampled over both timed loops
    rec.check_status()
    build_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in evs)
    model_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in evs)
    apply_ms = statistics.mean(e[2].elapsed_time(e[3]) for e in evs)
    return {"K": K, "W": W, "eager_ms": eager_ms, "graph_ms": graph_ms, "build_ms": build_ms, "model_ms": model_ms,
            "apply_ms": apply_ms, "launches": int(launches), "clocks": clocks, "eager_phases": eager_phases}


def kernel_table(t, bases, peak):
    k = {"build_smem_kernel": {"ms": t["build_ms"], "algorithmic_bytes": ALGO_BYTES_BUILD * bases},
         "apply_smem_kernel": {"ms": t["apply_ms"], "algorithmic_bytes": ALGO_BYTES_APPLY * bases}}
    for v in k.values():
        v["gbs"] = v["algorithmic_bytes"] / (v["ms"] * 1e-3) / 1e9
        v["frac_of_peak"] = v["gbs"] / peak
    return k


def traffic_for(wl, layout, kernel):
    """DRAM bytes of one launch from the committed `ncu --set full` capture of this shape (profiles/traffic.json:
    bytes per base of dram__bytes_read.sum + dram__bytes_write.sum, scaled to this batch), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            t = json.load(fh)
        e = t["L%d_R%d_%s" % (wl.L, wl.R, layout)]
        return {"bytes": e[kernel]["bytes_per_base"] * wl.N * wl.L, "capture": e["capture"],
                "captured_reads": e["reads"]}
    except Exception:
        return None


def checksum(t, L):
    """Position-sensitive checksums of a u8 [n, L] tensor (device), as python ints."""
    import torch
    n = t.numel() // L
    t = t.reshape(-1)[:n * L].view(n, L)
    col = torch.arange(1, L + 1, device=t.device, dtype=torch.int64)
    s1 = s2 = s3 = 0
    step = 4_000_000
    for lo in range(0, n, step):
        x = t[lo:lo + step].to(torch.int32)
        rows = x.sum(1, dtype=torch.int64)
        s1 += int(rows.sum())
        s2 += int((x.to(torch.int64) * col).sum())
        ramp = (torch.arange(lo, lo + x.shape[0], device=t.device, dtype=torch.int64) % 65521) + 1
        s3 += int((rows * ramp).sum())
    return [s1, s2, s3]


DUMP_BYTES = 64_000_000


def dump_outputs(path, hp):
    """--dump-outputs: what a caller of the hot path holds after the last timed step, one DIR/<name>.npy per array.
    The tables and the model under the reference's names (meanq ... dinuc_total, rgdq ... dindq) as float64, exact
    for these int64 counts; the recalibrated qualities of a sample of reads drawn with the workload's seed as
    float32 [rows, L] (`out_qual`), with their read numbers in the batch (`out_qual_reads`).  DUMP_BYTES at most."""
    import numpy as np
    import torch
    rec, N, L = hp.rec, hp.wl.N, hp.wl.L
    fields = {"meanq": rec.meanq, "rg_errs": rec.rg_errs, "rg_total": rec.rg_total, "q_errs": rec.q_errs,
              "q_total": rec.q_total, "pos_errs": rec.pos_errs, "pos_total": rec.pos_total,
              "dinuc_errs": rec.din_errs, "dinuc_total": rec.din_total,
              "rgdq": rec.rgdq, "qdq": rec.qdq, "posdq": rec.posdq, "dindq": rec.dindq}
    arrays = {name: t.cpu().numpy().astype(np.float64) for name, t in fields.items()}
    room = DUMP_BYTES - (1 << 16) - sum(a.nbytes for a in arrays.values())   # 64 KB for the .npy headers
    rows = min(N, 1 << 16, room // (4 * L + 8))
    if rows <= 0:
        raise SystemExit("bench.py: the tables alone exceed the %d bytes of --dump-outputs" % DUMP_BYTES)
    idx = np.sort(np.random.default_rng(hp.wl.seed).choice(N, rows, replace=False))
    out = hp.output_in_read_order()
    arrays["out_qual"] = out[torch.from_numpy(idx).to(out.device)].cpu().numpy().astype(np.float32)
    arrays["out_qual_reads"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def link_rates(dev, barrier, world, nbytes=1 << 30):
    """Pinned H2D and D2H copy rates with every rank copying at once: the ceiling of the end-to-end step."""
    import torch
    from kbbq import parallel
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    h.fill_(1)
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = {}
    for name, fn in (("h2d", lambda: d.copy_(h, non_blocking=True)), ("d2h", lambda: h.copy_(d, non_blocking=True))):
        best = 1e9
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            best = min(best, parallel.max_over_ranks(time.perf_counter() - t0, dev))
        out[name + "_gbs_per_gpu"] = nbytes / best / 1e9
    out["n_gpus_copying"] = world
    return out


def measure_e2e(args, wl, dev, world, rank, local, barrier, first_read):
    """The same pass through the reference-facing host-buffer API, pinned host memory in and out."""
    import numpy as np
    import torch
    from kbbq import _native, parallel
    from kbbq.device import DeviceRecalibrator, synth_reads
    lib = _native.lib()
    L, R = wl.L, wl.R
    n = min(wl.N, args.e2e_reads)
    seq, qual, corr, rg, second = synth_reads(wl.seed, first_read, n, L, R, device=dev)
    h = {}
    for name, t in (("seq", seq), ("qual", qual), ("corr", corr), ("second", second), ("rg", rg)):
        h[name] = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h[name].copy_(t)
    h_out = torch.empty(qual.shape, dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize()
    a = {k: v.numpy() for k, v in h.items()}
    rg_host = a["rg"].view(np.uint16) if R > 1 else None
    out_np = h_out.numpy()
    traffic = {}
    if world == 1:
        def e2e_step():
            st = C.c_int(0)
            rc = lib.kbbq_recalibrate_host(_native.ptr(a["seq"].reshape(-1)), _native.ptr(a["qual"].reshape(-1)),
                                           _native.ptr(a["corr"].reshape(-1)), _native.ptr(rg_host),
                                           _native.ptr(a["second"]), n, L, R, 6, _native.ptr(out_np.reshape(-1)),
                                           None, None, C.byref(st), local)
            _native.check(rc, st.value)
        api = "kbbq_recalibrate_host (C ABI; pinned host buffers in, pinned host buffer out)"
    else:
        state = {"s": None}

        def e2e_step():
            state["s"] = parallel.recalibrate_host_distributed(a["seq"], a["qual"], a["corr"], rg_host, a["second"], L, R,
                                                               out_np, session=state["s"], device=dev)
        api = ("kbbq.parallel.recalibrate_host_distributed (one kbbq_session per rank fed from pinned host buffers; "
               "ONE NCCL all-reduce on the sessions' table buffers)")
    for _ in range(2):   # warm-up (allocations, first touch of the pinned buffers)
        e2e_step()
    # every step timed on its own (wall clock around the blocking call, max over ranks); the figure reported is the
    # MEDIAN step: on a freshly leased box the host side (page cache, memory bandwidth) is noisy for the first seconds
    ke = max(3, args.e2e_steps)
    times = []
    for _ in range(ke):
        barrier()
        t0 = time.perf_counter()
        e2e_step()
        torch.cuda.synchronize()
        times.append(parallel.max_over_ranks(time.perf_counter() - t0, dev))
    dt = statistics.median(times) * ke
    # check against the device API on the same reads (tables summed over the ranks alike)
    rec = DeviceRecalibrator(L, R, max_reads=n, device=dev)
    rg_arg = rg if R > 1 else None
    rec.build(seq, qual, corr, rg_arg, second)
    rec.allreduce()
    rec.model()
    want = torch.empty_like(qual)
    rec.apply(seq, qual, want, rg_arg, second)
    rec.check_status()
    if not torch.equal(h_out.to(dev), want):
        raise SystemExit("bench.py: host-buffer path and device path disagree")
    # what the library actually copied (counted by its sessions from the copies they issued) and in which form
    cpus = len(os.sched_getaffinity(0))
    mode = int(lib.kbbq_host_pack_mode(max(1, cpus // max(1, world))))
    if world > 1 and state["s"] is not None:
        h2d, _ = state["s"].traffic()
        state["s"].close()
    else:
        up = C.c_int64(0)
        _native.check(lib.kbbq_host_last_traffic(local, C.byref(up), None))
        h2d = up.value
    transport = {0: "reads, qualities and corrected reads cross PCIe as they are",
                 1: "corrected reads cross PCIe as a 1-bit mismatch map made by the host cores",
                 2: "reads + corrected reads cross PCIe as 4 bits per base (base code | mismatch) packed by the host "
                    "cores while the copy engine moves the qualities"}[mode]
    links = link_rates(dev, barrier, world)
    ideal = h2d / (links["h2d_gbs_per_gpu"] * 1e9) + n * L / (links["d2h_gbs_per_gpu"] * 1e9)
    return {"value": world * n * L * ke / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": n * L,
            "host_input_bytes_per_step": 3 * n * L + n + (2 * n if R > 1 else 0), "ms_per_step": 1e3 * dt / ke,
            "steps": ke, "ms_all_steps": [1e3 * x for x in times], "statistic": "median step", "reads_per_gpu": n, "api": api +
            "; " + transport +
            ("; chunks segmented by read group on the device" if R > 1 else ""),
            "link": links, "frac_of_link": ideal / (dt / ke),
            "frac_of_link_note": "(h2d_bytes / measured H2D rate + d2h_bytes / measured D2H rate) / step time: upload and "
                                 "download cannot overlap inside one call (build -> model -> apply)",
            "checked": "output bytes equal the device-API result on the same reads"}


def verify_parity_n(hp, wl, dev, world, rank):
    """N > 1, outside the timed region: rank 0 regenerates every rank's shard, builds all of them alone (rows in read
    order, the work-list kernels: a code path the N-rank run did not take) and compares the tables with the
    all-reduced ones of the N-rank step and the output checksums with those the ranks computed."""
    import torch
    import torch.distributed as dist
    from kbbq.device import DeviceRecalibrator, synth_reads
    L, R, N = wl.L, wl.R, wl.N
    mine = torch.tensor(checksum(hp.output_in_read_order(), L), dtype=torch.int64, device=dev)
    sums = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(sums, mine)
    ok = True
    detail = ""
    if rank == 0:
        solo = DeviceRecalibrator(L, R, max_reads=N, device=dev)
        for r in range(world):
            seq, qual, corr, rg, second = synth_reads(wl.seed, r * N, N, L, R, device=dev)
            solo.build(seq, qual, corr, rg if R > 1 else None, second)
            del seq, qual, corr, rg, second
        if not torch.equal(solo.tables, hp.rec.tables):
            ok, detail = False, "tables differ"
        solo.model()
        for r in range(world):
            seq, qual, corr, rg, second = synth_reads(wl.seed, r * N, N, L, R, device=dev)
            out = torch.empty_like(qual)
            solo.apply(seq, qual, out, rg if R > 1 else None, second)
            if checksum(out, L) != [int(x) for x in sums[r].tolist()]:
                ok, detail = False, detail or "output checksum of shard %d differs" % r
            del seq, qual, corr, rg, second, out
        solo.check_status()
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.broadcast(flag, 0)
    return "ok" if int(flag.item()) else "MISMATCH: " + detail


def run_streamed_config(wl, batch, dev, world, rank, barrier):
    """Batches that do not fit HBM at once (config 5, strong scaling on few GPUs): pass 1 builds the tables over
    every batch, one all-reduce + model, pass 2 applies batch by batch.  The batches are regenerated on the device
    (counter-based generator), which stands in for the host feeding them; only the hot-path calls are timed (CUDA
    events per batch, summed, max over ranks)."""
    import torch
    from kbbq import _native, parallel
    from kbbq.device import DeviceRecalibrator, synth_reads
    N, L, R = wl.N, wl.L, wl.R
    rec = DeviceRecalibrator(L, R, max_reads=batch + 64 * R, device=dev)
    lib = _native.lib()
    out = torch.empty(batch * L + 64 * R * L + 16, dtype=torch.uint8, device=dev)
    launches0 = lib.kbbq_launch_count()
    ms = {"build": 0.0, "model": 0.0, "apply": 0.0}

    def timed(key, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms[key] += e0.elapsed_time(e1)

    for phase in ("build", "apply"):
        for lo in range(0, N, batch):
            n = min(batch, N - lo)
            seq, qual, corr, rg, second = synth_reads(wl.seed, rank * N + lo, n, L, R, device=dev)
            if R > 1:   # batches arrive segmented (the host-buffer entry points do this per chunk, behind the copies)
                sb = rec.segment(seq, qual, corr if phase == "build" else None, rg, second)
                if phase == "build":
                    timed("build", lambda: rec.build_segmented(sb))
                else:
                    timed("apply", lambda: rec.apply_segmented(sb, out))
                del sb
            elif phase == "build":
                timed("build", lambda: rec.build(seq, qual, corr, None, second))
            else:
                timed("apply", lambda: rec.apply(seq, qual, out[:n * L], None, second))
            del seq, qual, corr, rg, second
        if phase == "build":
            timed("model", lambda: (rec.allreduce(), rec.model()))
    rec.check_status()
    total_ms = parallel.max_over_ranks(sum(ms.values()), dev)
    return {"total_ms": total_ms, "phase_ms": ms, "launches": int(lib.kbbq_launch_count() - launches0)}


def measure_fastq(args, local):
    """FASTQ -> recalibrated FASTQ through kbbq.recalibrate.recalibrate_fastq, files on /dev/shm (or TMPDIR)."""
    import tempfile
    from kbbq import recalibrate, synth
    n, L, R = args.fastq_reads, 150, 8
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    d = tempfile.mkdtemp(prefix="kbbq_bench_", dir=base)
    try:
        import numpy as np
        from kbbq.device import synth_reads
        data = [t.cpu().numpy() for t in synth_reads(1003, 0, n, L, R)]
        data[3] = data[3].view(np.uint16)
        fu, fc, fo = os.path.join(d, "reads.fq"), os.path.join(d, "corrected.fq"), os.path.join(d, "out.fq")
        synth.write_fastq_fast(fu, fc, *data, infer_rg=True)
        del data
        best, size_in = 1e9, os.path.getsize(fu) + os.path.getsize(fc)
        for rep in range(3):
            sys.stdout.flush()
            saved = os.dup(1)
            fd = os.open(fo, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
            os.dup2(fd, 1)
            try:
                t0 = time.perf_counter()
                recalibrate.recalibrate_fastq((fu, fc), infer_rg=True, devices=[local])
                sys.stdout.flush()
                dt = time.perf_counter() - t0
            finally:
                os.dup2(saved, 1)
                os.close(saved)
                os.close(fd)
            if rep:
                best = min(best, dt)
        size_out = os.path.getsize(fo)
        return {"value": n * L / best, "unit": UNIT, "reads": n, "read_len": L, "read_groups": R, "seconds": best,
                "input_bytes": size_in, "output_bytes": size_out,
                "api": "kbbq.recalibrate.recalibrate_fastq((reads.fq, corrected.fq), infer_rg=True) -> stdout; files on "
                       + ("/dev/shm" if base else "TMPDIR") + ", best of 2 after a warm-up run"}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def run_b200(args):
    import torch
    import torch.distributed as dist
    from kbbq import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (kbbq_b200 has no CPU path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_cpus(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    wl = resolve_workload(args, world)
    N, L, R = wl.N, wl.L, wl.R
    K, W = args.steps, max(args.warmup, 3)
    peak, peak_src = measured_peak_gbs()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    line = {"metric": METRIC, "unit": UNIT, "n_gpus": world, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic"}
    config = {"workload": wl.describe("per GPU" if args.scaling == "weak" else "per GPU (%d in total)" % (N * world)),
              "reads_per_gpu": N, "read_len": L, "read_groups": R, "seed": wl.seed,
              "l2": "inputs (%.1f GB per step and GPU) exceed the 126 MB L2; no explicit flush" % (4 * N * L / 1e9),
              "parallelism": "reads sharded by rank; one int64 all-reduce of the tables" if world > 1 else "single GPU"}
    if numa:
        config["host"] = "each rank bound to the %d CPUs local to its GPU (NVML affinity)" % numa

    # ---- batches that do not fit HBM at once: the two-pass streamed runner ----
    batch = args.stream_batch
    if batch <= 0 and N * L * (8 if R > 1 else 4) > 120e9:
        batch = 32_000_000 if R == 1 else 25_000_000
    if batch > 0:
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs needs the batch resident in HBM, not streamed in batches")
        sampler = ClockSampler(local) if rank == 0 else None
        r = run_streamed_config(wl, batch, dev, world, rank, barrier)
        clocks = sampler.stop() if sampler else None
        if rank == 0:
            ms = r["phase_ms"]
            gbs = 6 * N * L / ((ms["build"] + ms["apply"]) * 1e-3) / 1e9
            config["batch_reads"] = batch
            config["streamed"] = "two passes over batches regenerated on the device; hot-path calls only"
            line.update({"value": world * N * L / (r["total_ms"] * 1e-3), "steps": 1, "warmup": 0, "ms_per_step": r["total_ms"],
                         "config": config,
                         "roofline": {"bound": "hbm", "kernel": "build + apply", "achieved": gbs, "peak": peak, "unit": "GB/s",
                                      "frac": gbs / peak, "traffic": None, "peak_source": peak_src},
                         "phase_ms": ms, "gpu_launches": r["launches"], "clocks": clocks})
            print(json.dumps(line))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- main measurement: the shard resident in HBM in the product's layout ----
    layout = args.layout
    if layout == "auto":
        layout = "segmented" if R > 1 else "read-order"
    hp = HotPath(wl, dev, rank * N, layout)
    t = time_hot_path(hp, K, W, world, barrier, use_graph=not args.no_graph,
                      sampler_factory=(lambda: ClockSampler(local)) if rank == 0 else None)
    total_ms = t["graph_ms"] if t["graph_ms"] is not None else t["eager_ms"]
    config["layout"] = ("segmented: rows sorted by (read group, mate), spans padded to 16 rows -- the layout the host-buffer "
                        "entry points keep in HBM (segmentation: see `layouts` and `e2e`)") if layout == "segmented" else \
        "read order: rows as the host has them" + (", rg[] per read (work-list gather)" if R > 1 else "")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, hp)   # rank 0's shard starts at read 0 of the stream

    parity_n = None
    if world > 1 and not args.no_verify:
        hp.step()   # leaves the all-reduced tables and this rank's output behind
        parity_n = verify_parity_n(hp, wl, dev, world, rank)

    # ---- the other layout, for comparison (several read groups only) ----
    layouts = None
    if R > 1 and world == 1 and not args.no_configs:
        other = "read-order" if layout == "segmented" else "segmented"
        hp2 = HotPath(wl, dev, rank * N, other)
        t2 = time_hot_path(hp2, max(2, K // 4), 3, world, barrier, use_graph=False)
        seg_hp, ro_hp = (hp, hp2) if layout == "segmented" else (hp2, hp)
        ts = []
        for fn in (lambda: seg_hp.rec.segment(seg_hp.seq, seg_hp.qual, ro_hp.corr, seg_hp.rg_arg, seg_hp.second),
                   lambda: seg_hp.output_in_read_order()):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            fn()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        same = torch.equal(hp.rec.tables, hp2.rec.tables) and torch.equal(hp.output_in_read_order(), hp2.output_in_read_order())
        if not same:
            raise SystemExit("bench.py: the two layouts disagree")
        layouts = {}
        for name, tt in ((layout, t), (other, t2)):
            kt = kernel_table(tt, N * L, peak)
            layouts[name] = {"build_ms": tt["build_ms"], "apply_ms": tt["apply_ms"],
                             "build_frac": kt["build_smem_kernel"]["frac_of_peak"],
                             "apply_frac": kt["apply_smem_kernel"]["frac_of_peak"],
                             "eager_ms_per_step": tt["eager_ms"] / tt["K"]}
        layouts["segmentation"] = {"segment_3_arrays_ms": ts[0], "unsegment_output_ms": ts[1],
                                   "note": "one-off row permutation on the device (2 B moved per byte), inside `e2e`, "
                                           "outside `value`; tables and read-order output bytes of both layouts compared equal"}
        del hp2

    # ---- end to end through the host-buffer API ----
    e2e = None
    if not args.no_e2e:
        e2e = measure_e2e(args, wl, dev, world, rank, local, barrier, rank * N)

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    kernels = kernel_table(t, N * L, peak)
    dom = max(kernels, key=lambda n: kernels[n]["ms"])
    combined = (ALGO_BYTES_BUILD + ALGO_BYTES_APPLY) * N * L / ((t["build_ms"] + t["apply_ms"]) * 1e-3) / 1e9
    traffic = traffic_for(wl, layout, dom)
    line.update({
        "value": world * N * L * K / (total_ms * 1e-3), "steps": K, "warmup": W, "ms_per_step": total_ms / K,
        "config": config,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["gbs"], "peak": peak, "unit": "GB/s",
                     "frac": kernels[dom]["frac_of_peak"], "traffic": traffic["bytes"] if traffic else None,
                     "traffic_source": traffic, "peak_source": peak_src,
                     "timing": "CUDA events on the launching stream around the build phase (table reset, pre-pass kernels "
                               "< 1 %, kbbq_build*) and the apply phase of every step of the timed loop `value` comes "
                               "from" + (" (graph replay: one graph per phase)" if t["graph_ms"] is not None else " (eager)"),
                     "build_plus_apply_gbs": combined, "build_plus_apply_frac": combined / peak},
        "kernels": kernels,
        "phase_ms": {"build": t["build_ms"], "allreduce+model": t["model_ms"], "apply": t["apply_ms"]},
        "launch": {"mode": "CUDA graph replay" if t["graph_ms"] is not None else "eager",
                   "eager_ms_per_step": t["eager_ms"] / K,
                   "eager_phase_ms": ({"build": t["eager_phases"]["build_ms"], "allreduce+model": t["eager_phases"]["model_ms"],
                                       "apply": t["eager_phases"]["apply_ms"]} if t.get("eager_phases") else None),
                   "note": "`value`, `phase_ms`, `kernels` and `roofline` all come from the same timed loop: the step "
                           "replayed from one CUDA graph per phase (build | model | apply) around the eager all-reduce; "
                           "the eager launch loop is reported next to it"},
        "gpu_launches": t["launches"],
        "clocks": t["clocks"],
    })
    if layouts:
        line["layouts"] = layouts
    if parity_n is not None:
        line["parity_n"] = parity_n
    if e2e:
        line["e2e"] = e2e
    del hp
    torch.cuda.empty_cache()

    if world == 1 and not args.no_configs and wl.config == 2:
        # the other BASELINE configs at full per-GPU size, after the main timed region
        cfgs = {"2": {"workload": CONFIGS[2]["name"], "ms_per_step": total_ms / K, "value": line["value"],
                      "build_frac": kernels["build_smem_kernel"]["frac_of_peak"],
                      "apply_frac": kernels["apply_smem_kernel"]["frac_of_peak"], "layout": layout}}
        for c in (3, 4):
            cw = Workload(CONFIGS[c]["reads"], CONFIGS[c]["read_len"], CONFIGS[c]["read_groups"], CONFIGS[c]["seed"],
                          CONFIGS[c]["name"], c)
            entry = {"workload": cw.describe()}
            for lay in ("segmented", "read-order"):
                h = HotPath(cw, dev, 0, lay)
                tt = time_hot_path(h, 5, 3, 1, barrier, use_graph=True)   # both layouts from the graph replay: the eager
                #                                    loop of the work-list walk is at the mercy of the host's launch timing
                kt = kernel_table(tt, cw.N * cw.L, peak)
                ms = (tt["graph_ms"] if tt["graph_ms"] is not None else tt["eager_ms"]) / tt["K"]
                entry[lay] = {"ms_per_step": ms, "value": cw.N * cw.L / (ms * 1e-3),
                              "build_ms": tt["build_ms"], "apply_ms": tt["apply_ms"],
                              "build_frac": kt["build_smem_kernel"]["frac_of_peak"],
                              "apply_frac": kt["apply_smem_kernel"]["frac_of_peak"]}
                del h
                torch.cuda.empty_cache()
            cfgs[str(c)] = entry
        c5 = CONFIGS[5]
        cw = Workload(c5["reads"], c5["read_len"], c5["read_groups"], c5["seed"], c5["name"], 5)
        r5 = run_streamed_config(cw, c5["batch"], dev, 1, 0, barrier)
        gbs = 6 * cw.N * cw.L / ((r5["phase_ms"]["build"] + r5["phase_ms"]["apply"]) * 1e-3) / 1e9
        cfgs["5"] = {"workload": cw.describe(), "ms_per_step": r5["total_ms"], "value": cw.N * cw.L / (r5["total_ms"] * 1e-3),
                     "build_plus_apply_frac": gbs / peak, "phase_ms": r5["phase_ms"]}
        line["configs"] = cfgs
        torch.cuda.empty_cache()

    if world == 1 and not args.no_fastq:
        try:
            line["e2e_fastq"] = measure_fastq(args, local)
        except Exception as exc:   # a diagnostic figure: never lose the line over it
            line["e2e_fastq"] = {"error": repr(exc)}

    if world == 1 and not args.no_cpu:
        oracle, data, sample, threads = cpu_port_throughput(N, L, R, wl.seed, args.cpu_seconds)
        passes, t0 = 0, time.perf_counter()
        while passes == 0 or time.perf_counter() - t0 < args.cpu_seconds:
            oracle.recalibrate(*data, L, R, threads=threads)
            passes += 1
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": passes * sample * L / dt, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": "first %d reads x %d bp of the workload, %d pass(es) in %.1f s "
                                          "(oracle/kbbq_oracle.c, OpenMP)" % (sample, L, passes, dt)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads", type=int, default=None, help="reads per GPU (default: config 2 = 10 M on one GPU, config 3 = 25 M on several)")
    ap.add_argument("--read-len", type=int, default=None)
    ap.add_argument("--read-groups", type=int, default=None)
    ap.add_argument("--layout", default="auto", choices=["auto", "segmented", "read-order"],
                    help="HBM layout of the resident batch (auto: segmented with several read groups)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--total-reads", type=int, default=200_000_000, help="--scaling strong: reads split over the GPUs")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-reads", type=int, default=10_000_000, help="reads per GPU of the end-to-end measurement (pinned host memory: 6 B per base)")
    ap.add_argument("--fastq-reads", type=int, default=2_000_000)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--stream-batch", type=int, default=0,
                    help="stream --reads reads per GPU through the device in batches of this many (config 5)")
    ap.add_argument("--no-graph", action="store_true", help="time the eager launch loop instead of the CUDA-graph replay")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` / `layouts` blocks")
    ap.add_argument("--no-fastq", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="N > 1: skip the parity check against rank 0 alone")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the tables, the model and the qualities of a seeded sample of "
                         "reads that the last step computed to DIR/<name>.npy (float32 / float64, 64 MB at most)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
