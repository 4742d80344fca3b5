"""Kernel regimes that realistic data never reaches: every shared-memory plan the planner can pick (past the point
where every CTA's staging ring wraps), the tuning-hook plans, packed shared-memory counters driven to their flush
and fold bounds, every minscore, and bases outside ACGTN on the apply and BAM paths.

The expected answer is always the C oracle (oracle/kbbq_oracle.c) or a closed form, compared bit for bit: int64
tables, delta tables, output bytes, and the exception raised.  The host-only tests (planner) need no GPU.
"""
import concurrent.futures
import os
from functools import lru_cache

import numpy as np
import pytest

from conftest import DELTA_KEYS, TABLE_KEYS

SEG = 0x100          # kbbq_plan_info: arrays | KBBQ_PLAN_SEGMENTED = the plan of a segmented batch
ERR_UNIT = 65025     # build.cuh: a shared-memory counter holds total + 65025 * errors


def _native():
    from kbbq import _native as n
    return n


def _fits(p, L, minscore):
    """The fit assertions of test_host_logic.test_shared_memory_plans_fit_for_every_read_length, any minscore."""
    G, lanes, ng, threads, nprod, kps, stages, drep, total, table_bytes = (p[k] for k in (
        "G", "lanes", "ng", "threads", "nprod", "kps", "stages", "drep", "smem", "table_bytes"))
    assert total <= 232448 and table_bytes < total
    assert threads % 32 == 0 and threads + 32 * nprod <= 1024 and ng * lanes <= threads
    assert (G * L) % 4 == 0 and 1 <= kps <= 8 and stages >= 2 and drep in (8, 16, 32)
    rows, rs = 44 - minscore, (4 * ((L + 3) // 4) * 4 + 127) // 128 * 128
    assert table_bytes >= 2 * rows * rs + rows * 16 * drep * 4


@lru_cache(maxsize=None)
def plan_classes():
    """{(arrays, G, L % 4, kps, stages, drep, nprod): (smallest L, R)} over L = 4..288, R in {1, 3}, the build (3)
    and apply (2) kernels, in read order and segmented.  Computed from the planner, so it follows the planner."""
    n = _native()
    classes = {}
    for R in (1, 3):
        for L in range(4, 289):
            for arrays in (3, 2, 3 | SEG, 2 | SEG):
                p = n.plan_info(L, R, 6, arrays)
                if p is None:
                    continue
                key = (arrays, p["G"], L % 4, p["kps"], p["stages"], p["drep"], p["nprod"])
                if key not in classes or (L, R) < classes[key]:
                    classes[key] = (L, R)
    return classes


def _wrap_reads(L, R, sms):
    """Reads for which every CTA of every plan of (L, R) wraps its staging ring at least three times."""
    n = _native()
    need = 0
    for arrays in (3, 2, 3 | SEG, 2 | SEG):
        p = n.plan_info(L, R, 6, arrays)
        if p is not None:
            need = max(need, sms * (3 * p["stages"] + 1) * p["kps"] * p["ng"] * p["G"])
    return need


# ---------------------------------------------------------------------------------------------------------------
# CPU: the planner
# ---------------------------------------------------------------------------------------------------------------

def test_plan_classes_cover_read_order_and_segmented_plans():
    n = _native()
    classes = plan_classes()
    kinds = {k[0] for k in classes}
    assert kinds == {3, 2, 3 | SEG, 2 | SEG}
    for (arrays, G, lmod, kps, stages, drep, nprod), (L, R) in classes.items():
        p = n.plan_info(L, R, 6, arrays)
        _fits(p, L, 6)
        if arrays & SEG:   # a segmented span is one read group's geometry: power-of-two groups, one producer warp
            assert G & (G - 1) == 0 and nprod == 1, (arrays, L, R)
    # any other bit of `arrays` is a bad argument
    assert n.plan_info(150, 1, 6, 2 | 0x200) is None


def _plan_row(L):
    n = _native()
    lib = n.lib()
    rows = []
    for minscore in range(0, 43):
        for R in (1, 8):
            plans = {a: n.plan_info(L, R, minscore, a) for a in (3, 2, 3 | SEG, 2 | SEG)}
            rows.append((L, minscore, R, plans, bool(lib.kbbq_segmented_supported(L, R, minscore))))
    return rows


def test_plans_for_every_minscore():
    """Every L = 4..288, minscore = 0..42, R in {1, 8}: a plan that fits (the table has 44 - minscore rows) or
    None; kbbq_segmented_supported says yes exactly when both segmented plans exist; minscore 0 has no plan (row 0
    of the tables is the trash row) and minscore 43 none either."""
    n = _native()
    with concurrent.futures.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:   # ctypes drops the GIL
        results = [r for rows in ex.map(_plan_row, range(4, 289)) for r in rows]
    planned = 0
    for L, minscore, R, plans, seg_ok in results:
        if minscore == 0:
            assert all(p is None for p in plans.values()) and not seg_ok, (L, R)
            continue
        for arrays, p in plans.items():
            if p is not None:
                _fits(p, L, minscore)
                planned += 1
        assert seg_ok == (plans[3 | SEG] is not None and plans[2 | SEG] is not None), (L, minscore, R)
        # fewer rows never lose a plan: minscore 6 plans every length, so every larger minscore does too
        if minscore >= 6:
            assert plans[3] is not None and plans[2] is not None, (L, minscore, R)
    assert planned > 285 * 37 * 2 * 4
    for arrays in (3, 2, 3 | SEG, 2 | SEG):
        assert n.plan_info(150, 1, 43, arrays) is None


# ---------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    yield torch
    print("\npeak device memory of the module: %.1f GB" % (torch.cuda.max_memory_allocated() / 1e9))
    torch.cuda.empty_cache()


def _sms(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _dev(torch, *arrays):
    out = []
    for a in arrays:
        if a is None:
            out.append(None)
        elif a.dtype == np.uint16:
            out.append(torch.from_numpy(a.view(np.int16)).cuda())
        else:
            out.append(torch.from_numpy(np.ascontiguousarray(a)).cuda())
    return out


def _host(t):
    a = t.cpu().numpy()
    return a.view(np.uint16) if a.dtype == np.int16 else a


def _oracle_all(oracle, seq, qual, corr, rg, second, L, R, minscore=6):
    pe, pt, de, dt = oracle.build_tables(seq, qual, corr, rg, second, L, R, minscore, threads=os.cpu_count() or 1)
    tables = tuple(oracle.marginals(pe, pt)) + (pe, pt, de, dt)
    deltas = oracle.get_delta_qs(*tables)
    out = oracle.apply(seq, qual, rg, second, L, R, tables[0], *deltas, minscore=minscore)
    return tables, deltas, out


def _check(got_tables, got_deltas, got_out, want, what):
    tables, deltas, out = want
    for a, b, key in zip(got_tables, tables, TABLE_KEYS):
        assert np.array_equal(a, b), (key,) + what
    for a, b, key in zip(got_deltas, deltas, DELTA_KEYS):
        assert np.array_equal(a, b), (key,) + what
    assert np.array_equal(got_out.astype(np.int16), out), what


def _device_path(torch, d, L, R, path, minscore=6):
    """build -> model -> apply in read order through kbbq_build / kbbq_apply (path 0 / 1 / 2)."""
    from kbbq.device import DeviceRecalibrator
    s, q, c, g, sec = d
    rec = DeviceRecalibrator(L, R, max_reads=s.shape[0], minscore=minscore)
    rec.build(s, q, c, g, sec, path=path)
    tables, deltas = rec.covariate_arrays(), rec.delta_qs()
    out = torch.full_like(q, 255)
    rec.apply(s, q, out, g, sec, path=path)
    rec.check_status()
    return tables, deltas, out.cpu().numpy()


def _segmented_path(torch, d, L, R, minscore=6):
    from kbbq.device import DeviceRecalibrator
    s, q, c, g, sec = d
    rec = DeviceRecalibrator(L, R, max_reads=s.shape[0], minscore=minscore)
    sb = rec.segment(s, q, c, g, sec)
    rec.build_segmented(sb)
    tables, deltas = rec.covariate_arrays(), rec.delta_qs()
    out_seg = torch.full((sb.rows_bound * L + 16,), 255, dtype=torch.uint8, device=q.device)
    out = torch.full_like(q, 255)
    rec.apply_segmented(sb, out_seg)
    rec.unsegment(sb, out_seg, out)
    rec.check_status()
    return tables, deltas, out.cpu().numpy()


def _synth_mixed(torch, seed, N, L, R):
    """Device synth reads; unpaired (read groups and mates at random) half of the time; 10 % N bases and 10 %
    low qualities half of the time.  -> device tensors, host arrays."""
    from kbbq.device import synth_reads
    seq, qual, corr, rg, second = synth_reads(seed, 0, N, L, R)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    if seed % 2:
        rg = torch.randint(0, R, (N,), generator=gen, device="cuda", dtype=torch.int16)
        second = torch.randint(0, 2, (N,), generator=gen, device="cuda", dtype=torch.uint8)
    if seed % 4 < 2:
        seq[torch.rand(N, L, generator=gen, device="cuda") < 0.1] = ord("N")
        low = torch.rand(N, L, generator=gen, device="cuda") < 0.1
        qual = torch.where(low, torch.randint(0, 8, (N, L), generator=gen, device="cuda", dtype=torch.uint8), qual)
    d = (seq, qual, corr, rg, second)
    return d, tuple(_host(t) for t in d)


# ---------------------------------------------------------------------------------------------------------------
# A. every shared-memory plan, past ring wrap
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_every_plan_class_past_ring_wrap(torch_cuda, oracle_mod):
    """One representative (L, R) per plan class, sized so that every CTA wraps its staging ring (and flips the
    mbarrier phase) at least three times; read order through the shared-memory kernels (path 1) and segmented."""
    torch = torch_cuda
    n = _native()
    sms = _sms(torch)
    reps = sorted(set(plan_classes().values()))
    runs = {"build": 0, "apply": 0, "segmented": 0}
    for i, (L, R) in enumerate(reps):
        N = _wrap_reads(L, R, sms) + 2 * i + 1       # odd tail
        d, h = _synth_mixed(torch, 7000 + i, N, L, R)
        want = _oracle_all(oracle_mod, *h, L, R)
        _check(*_device_path(torch, d, L, R, 1), want, (L, R, N, "read order"))
        runs["build"] += 1
        runs["apply"] += 1
        if n.lib().kbbq_segmented_supported(L, R, 6):
            _check(*_segmented_path(torch, d, L, R), want, (L, R, N, "segmented"))
            runs["segmented"] += 1
        del d
    assert runs["segmented"] > 0
    print("plan classes: %d, representatives: %d, runs: %s" % (len(plan_classes()), len(reps), runs))


def _hook_combos():
    combos = []
    for L in (8, 75, 150, 251):
        for R in (1, 4):
            for kps in range(1, 9):
                for drep in (8, 16, 32):
                    for stages in (2, None):
                        combos.append((L, R, kps, drep, stages))
    return combos


def _set_hooks(monkeypatch, kps, drep, stages):
    monkeypatch.setenv("KBBQ_KPS", str(kps))
    monkeypatch.setenv("KBBQ_DREP", str(drep))
    if stages is None:
        monkeypatch.delenv("KBBQ_MIN_STAGES", raising=False)
        monkeypatch.delenv("KBBQ_MAX_STAGES", raising=False)
    else:
        monkeypatch.setenv("KBBQ_MIN_STAGES", str(stages))
        monkeypatch.setenv("KBBQ_MAX_STAGES", str(stages))


@pytest.mark.gpu
def test_tuning_hook_plans(torch_cuda, oracle_mod, monkeypatch):
    """KBBQ_KPS 1..8, KBBQ_DREP 8 / 16 / 32, a ring of 2 stages or the deepest that fits, at L = 8 / 75 / 150 / 251
    and R = 1 / 4: the plan obeys the hooks (checked through kbbq_plan_info) and every distinct plan computes the
    oracle's tables and qualities.  This runs build_smem_kernel / apply_smem_kernel instantiations 5..8 and 8 dinuc
    replicas, which the default planner never picks."""
    torch = torch_cuda
    n = _native()
    sms = _sms(torch)
    seen, ran, kps_run = set(), 0, set()
    for L, R, kps, drep, stages in _hook_combos():
        _set_hooks(monkeypatch, kps, drep, stages)
        pb, pa = n.plan_info(L, R, 6, 3), n.plan_info(L, R, 6, 2)
        if pb is None or pa is None:
            continue
        for p in (pb, pa):
            assert p["kps"] <= kps and p["drep"] <= drep, (L, R, kps, drep, p)
            if drep == 8:
                assert p["drep"] == 8
            if stages is not None:
                assert p["stages"] == stages
        key = (L, R, tuple(pb.values()), tuple(pa.values()))
        if key in seen:
            continue
        seen.add(key)
        N = sms * max((2 * p["stages"] + 1) * p["kps"] * p["ng"] * p["G"] for p in (pb, pa)) + 3
        d, h = _synth_mixed(torch, 9000 + ran, N, L, R)
        want = _oracle_all(oracle_mod, *h, L, R)
        _check(*_device_path(torch, d, L, R, 1), want, (L, R, kps, drep, stages))
        kps_run.update((pb["kps"], pa["kps"]))
        ran += 1
    assert kps_run >= set(range(1, 9)), kps_run
    print("tuning-hook plans run: %d" % ran)


# ---------------------------------------------------------------------------------------------------------------
# B. packed counters at their bounds
# ---------------------------------------------------------------------------------------------------------------

def _tiled_case(torch, oracle, B, L, R, M, rem, minscore=6):
    """A batch of M copies of block B (host arrays) plus its first `rem` reads, built on the device.  -> device
    tensors, want tables / deltas, want output of one copy of B, want output of the remainder."""
    seq, qual, corr, rg, second = B
    d = []
    for a in B:
        t = _dev(torch, a)[0]
        big = t.repeat((M,) + (1,) * (t.dim() - 1))
        d.append(torch.cat([big, t[:rem]]) if rem else big)
        del big
    tb = oracle.build_tables(seq, qual, corr, rg, second, L, R, minscore)
    tr = oracle.build_tables(seq[:rem], qual[:rem], corr[:rem], rg[:rem], second[:rem], L, R, minscore)
    pe, pt, de, dt = (M * a + b for a, b in zip(tb, tr))
    tables = tuple(oracle.marginals(pe, pt)) + (pe, pt, de, dt)
    deltas = oracle.get_delta_qs(*tables)
    out_b = oracle.apply(seq, qual, rg, second, L, R, tables[0], *deltas, minscore=minscore)
    return d, tables, deltas, out_b


def _check_tiled(torch, rec, out, tables, deltas, out_b, M, what):
    got = rec.covariate_arrays()
    for a, b, key in zip(got, tables, TABLE_KEYS):
        assert np.array_equal(a, b), (key,) + what
    for a, b, key in zip(rec.delta_qs(), deltas, DELTA_KEYS):
        assert np.array_equal(a, b), (key,) + what
    nb, L = out_b.shape
    want = torch.from_numpy(out_b.astype(np.uint8)).cuda()
    assert bool((out[:M * nb].view(M, nb, L) == want).all()), what
    rem = out.shape[0] - M * nb
    assert bool((out[M * nb:] == want[:rem]).all()), what


def _homopolymer_block(L, R, errors):
    nb = 64
    seq = np.empty((nb, L), np.uint8)
    seq[: nb // 2] = ord("A")                                     # every dinucleotide AA
    seq[nb // 2:] = np.frombuffer(b"AC" * L, np.uint8)[:L]        # AC / CA: other slots
    qual = np.full((nb, L), 30, np.uint8)
    corr = seq ^ 1 if errors else seq.copy()                      # a mismatch at every base, or none
    rg = ((np.arange(nb) // 2) % R).astype(np.uint16)
    rg[: nb // 2] = 0                                             # every AA read in read group 0
    second = (np.arange(nb) & 1).astype(np.uint8)
    return (seq, qual, corr, rg, second), nb


def _run_tiled(torch, oracle, B, nb, L, R, N, segmented, what):
    from kbbq.device import DeviceRecalibrator
    M, rem = N // nb, N % nb
    d, tables, deltas, out_b = _tiled_case(torch, oracle, B, L, R, M, rem)
    s, q, c, g, sec = d
    rec = DeviceRecalibrator(L, R, max_reads=s.shape[0])
    rec.build(s, q, c, g if R > 1 else None, sec, path=1)
    out = torch.empty_like(q)
    rec.model()
    rec.apply(s, q, out, g if R > 1 else None, sec, path=1)
    rec.check_status()
    _check_tiled(torch, rec, out, tables, deltas, out_b, M, what + ("read order",))
    del out
    if segmented:
        rec.reset()
        sb = rec.segment(s, q, c, g if R > 1 else None, sec)
        del s, c, g, sec, d
        rec.build_segmented(sb)
        rec.model()
        out_seg = torch.empty(sb.rows_bound * L + 16, dtype=torch.uint8, device=q.device)
        rec.apply_segmented(sb, out_seg)
        out = torch.empty_like(q)
        rec.unsegment(sb, out_seg, out)
        rec.check_status()
        del out_seg, sb
        _check_tiled(torch, rec, out, tables, deltas, out_b, M, what + ("segmented",))
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_dinuc_replicas_at_their_fold_bound(torch_cuda, oracle_mod, monkeypatch):
    """Homopolymer reads at one quality: half the reads, all of read group 0, put every base into dinucleotide AA of
    one row, so one
    replica cell of every CTA would take >= 3 * 65025 hits if the replicas were never folded (sized for 32
    replicas, the most the hits are spread over).  With a mismatch at every base the error field climbs to
    65024 * 65025 before each fold.  Every plan class, with and without errors, and 8 groups per stage on 8
    replicas (the most hits per replica and fold)."""
    torch = torch_cuda
    n = _native()
    sms = _sms(torch)
    cases = [(L, R, None) for L, R in sorted(set(plan_classes().values()))]
    cases += [(L, 1, (8, 8)) for L in (8, 75, 150, 251)]
    for L, R, hooks in cases:
        if hooks:
            monkeypatch.setenv("KBBQ_KPS", str(hooks[0]))
            monkeypatch.setenv("KBBQ_DREP", str(hooks[1]))
            assert n.plan_info(L, R, 6, 3)["drep"] == 8
        else:
            monkeypatch.delenv("KBBQ_KPS", raising=False)
            monkeypatch.delenv("KBBQ_DREP", raising=False)
        # hits on the AA cell of one replica of one CTA without folding: N / SMs * (L - 1) / 2 (half the reads)
        # / 32 (replicas) >= 3 * 65025
        N = -(-3 * ERR_UNIT * 32 * 2 * sms // (L - 1)) + 37
        seg = bool(n.lib().kbbq_segmented_supported(L, R, 6)) and hooks is None
        for errors in (True, False):
            B, nb = _homopolymer_block(L, R, errors)
            _run_tiled(torch, oracle_mod, B, nb, L, R, N, seg, (L, R, N, errors, hooks))


@pytest.mark.gpu
@pytest.mark.parametrize("L", [4, 37, 150])
def test_cycle_table_at_its_flush_bound(torch_cuda, oracle_mod, L):
    """One quality, all reads first of their pair, R = 2 in read order with one read group for all but the last
    16 reads: the work-list walk sees one long segment and every cycle cell takes one hit per read (no split over
    two table slots), so with N = SMs * 3 * 65025 reads a CTA's cells would pass 65025 three times without a
    flush.  The same batch in the segmented layout."""
    torch = torch_cuda
    sms = _sms(torch)
    R, nb = 2, 256
    rng = np.random.default_rng(L)
    seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (nb, L))]
    B = (seq, np.full((nb, L), 30, np.uint8), seq ^ 1, np.zeros(nb, np.uint16), np.zeros(nb, np.uint8))
    N = -(-3 * ERR_UNIT * sms // nb) * nb                       # whole copies of the block
    M = N // nb
    d, tables, deltas, out_b = _tiled_case(torch, oracle_mod, B, L, R, M, 0)
    # the last 16 reads are read group 1: tables move from group 0 to group 1 for them
    d[3][-16:] = 1
    tail = (seq[-16:], B[1][-16:], B[2][-16:], np.zeros(16, np.uint16), np.zeros(16, np.uint8))
    t0 = oracle_mod.build_tables(*tail, L, R)
    t1 = oracle_mod.build_tables(tail[0], tail[1], tail[2], np.ones(16, np.uint16), tail[4], L, R)
    pe, pt, de, dt = (a - b + c for a, b, c in zip(tables[5:], t0, t1))
    tables = tuple(oracle_mod.marginals(pe, pt)) + (pe, pt, de, dt)
    deltas = oracle_mod.get_delta_qs(*tables)
    out_b = oracle_mod.apply(B[0], B[1], B[3], B[4], L, R, tables[0], *deltas)
    out_t = oracle_mod.apply(tail[0], tail[1], np.ones(16, np.uint16), tail[4], L, R, tables[0], *deltas)
    from kbbq.device import DeviceRecalibrator
    s, q, c, g, sec = d
    rec = DeviceRecalibrator(L, R, max_reads=N)

    def check(out, what):
        got = rec.covariate_arrays()
        for a, b, key in zip(got, tables, TABLE_KEYS):
            assert np.array_equal(a, b), (key, L, what)
        want = torch.from_numpy(out_b.astype(np.uint8)).cuda()
        assert bool((out[:N - nb].view(M - 1, nb, L) == want).all()), (L, what)
        assert bool((out[N - nb:N - 16] == want[:-16]).all()), (L, what)
        assert np.array_equal(out[N - 16:].cpu().numpy().astype(np.int16), out_t), (L, what)

    rec.build(s, q, c, g, sec, path=1)
    rec.model()
    out = torch.empty_like(q)
    rec.apply(s, q, out, g, sec, path=1)
    rec.check_status()
    check(out, "read order")
    del out
    rec.reset()
    sb = rec.segment(s, q, c, g, sec)
    del s, c, g, sec, d
    torch.cuda.empty_cache()
    rec.build_segmented(sb)
    rec.model()
    out_seg = torch.empty(sb.rows_bound * L + 16, dtype=torch.uint8, device=q.device)
    rec.apply_segmented(sb, out_seg)
    out = torch.empty_like(q)
    rec.unsegment(sb, out_seg, out)
    rec.check_status()
    del out_seg, sb
    check(out, "segmented")
    print("L=%d: N=%d reads, %d hits per cycle cell per CTA without a flush" % (L, N, N // sms))
    del out, q, rec
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_calibration_counts_full_chunk(torch_cuda):
    """kbbq_calibration_counts over one full launch chunk (SMs * 3 CTAs * 256 threads * 2000 iterations * 32
    bases) plus 4 099 bases: every lane counter takes its 64 000 bases, every one an error, at one quality; with
    and without a skip mask on alternate bytes.  Closed form."""
    torch = torch_cuda
    from kbbq.device import calibration_counts
    sms = _sms(torch)
    n = sms * 3 * 256 * 2000 * 32 + 4099
    qual = torch.full((n,), 30, dtype=torch.uint8, device="cuda")
    err = torch.ones(n, dtype=torch.uint8, device="cuda")
    total, errs = calibration_counts(qual, err)
    want = np.zeros(256, np.int64)
    want[30] = n
    assert np.array_equal(total.cpu().numpy(), want) and np.array_equal(errs.cpu().numpy(), want)
    skip = torch.zeros(n, dtype=torch.uint8, device="cuda")
    skip[1::2] = 1
    total, errs = calibration_counts(qual, err, skip=skip)
    want[30] = n - n // 2
    assert np.array_equal(total.cpu().numpy(), want) and np.array_equal(errs.cpu().numpy(), want)
    del qual, err, skip
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------
# C. minscore
# ---------------------------------------------------------------------------------------------------------------

MINSCORES = [0, 1, 2, 5, 7, 20, 41, 42]


def _minscore_batch(m, L, R, seed):
    from kbbq import synth
    N = 2003
    seq, qual, corr, rg, second = synth.synth_reads(seed, 0, N, L, R)
    rng = np.random.default_rng(seed)
    pick = np.array([max(m - 1, 0), m, min(m + 1, 42), 0, 42], np.uint8)
    remap = rng.random((N, L)) < 0.7
    qual = np.where(remap, pick[rng.integers(0, 5, (N, L))], qual).astype(np.uint8)
    seq = np.where(rng.random((N, L)) < 0.05, np.uint8(ord("N")), seq)
    if seed % 2:
        rg = rng.integers(0, R, N).astype(np.uint16)
        second = rng.integers(0, 2, N).astype(np.uint8)
    return seq, qual, corr, rg, second


@pytest.mark.gpu
@pytest.mark.parametrize("m", MINSCORES)
def test_minscore_every_entry_point(torch_cuda, oracle_mod, m):
    """minscore drives the row arithmetic of the shared-memory kernels (44 - minscore rows, row 0 = trash), the
    apply's "row 0 holds minscore - 1" trick and the BAM canonical form's "quality 0 = skip" rule.  Every entry
    point against the oracle at that minscore; minscore 0 has no shared-memory plan: path 1 and the segmented
    layout refuse it, path 0 and the BAM entry points take the generic / direct kernels."""
    torch = torch_cuda
    n = _native()
    from kbbq.device import DeviceRecalibrator
    for L in (37, 100, 151):
        for R in (1, 3):
            h = _minscore_batch(m, L, R, 100 * m + L + R)
            want = _oracle_all(oracle_mod, *h, L, R, minscore=m)
            d = _dev(torch, *h)
            for path in (0, 1, 2):
                if m == 0 and path == 1:
                    with pytest.raises(n.KbbqNativeError):
                        _device_path(torch, d, L, R, path, minscore=m)
                    continue
                _check(*_device_path(torch, d, L, R, path, minscore=m), want, (m, L, R, path))
            if m == 0:
                assert not n.lib().kbbq_segmented_supported(L, R, m)
                with pytest.raises(n.KbbqNativeError):
                    _segmented_path(torch, d, L, R, minscore=m)
            elif n.lib().kbbq_segmented_supported(L, R, m):
                _check(*_segmented_path(torch, d, L, R, minscore=m), want, (m, L, R, "segmented"))
            # host-buffer entry point and a session
            # (it returns the four count tables, meanq and the deltas; the other marginals stay on the device)
            out, tabs, dqs = n.recalibrate_host(*h, L, R, minscore=m, want_tables=True)
            for a, b, key in zip(tabs, want[0][5:], TABLE_KEYS[5:]):
                assert np.array_equal(a, b), (key, m, L, R, "host")
            for a, b, key in zip(dqs, (want[0][0],) + tuple(want[1]), ("meanq",) + DELTA_KEYS):
                assert np.array_equal(a, b), (key, m, L, R, "host")
            assert np.array_equal(out.astype(np.int16), want[2]), (m, L, R, "host")
            with n.Session(L, R, m) as S:
                S.build_chunk(*h)
                S.model()
                out = np.zeros((h[0].shape[0], L), np.uint8)
                S.apply_chunk(h[0], h[1], h[3], h[4], out)
                S.sync()
                assert np.array_equal(out.astype(np.int16), want[2]), (m, L, R, "session")
            # BAM side: canonical form + shared-memory kernels (fast) and the direct kernels
            seq, qual, corr, rg, second = h
            rng = np.random.default_rng(m + L)
            err = (seq != corr).astype(np.uint8)
            skip = (rng.random((seq.shape[0], L)) < 0.05).astype(np.uint8)
            flags = rng.integers(0, 4, seq.shape[0]).astype(np.uint8)
            a0 = (rng.integers(0, 6, seq.shape[0]) * (rng.random(seq.shape[0]) < 0.4)).astype(np.uint16)
            a1 = (L - rng.integers(0, 6, seq.shape[0]) * (rng.random(seq.shape[0]) < 0.4)).astype(np.uint16)
            wt = oracle_mod.build_tables_bam(seq, qual, err, skip, rg, flags, a0, a1, L, R, minscore=m)
            for fast in (True, False):
                rec = DeviceRecalibrator(L, R, minscore=m)
                dd = _dev(torch, seq, qual, err, skip, rg, flags, a0, a1)
                rec.build_bam(*dd, fast=fast)
                tables = rec.covariate_arrays()
                rec.check_status()
                for key, a, b in zip(TABLE_KEYS[5:], tables[5:], wt):
                    assert np.array_equal(a, b), (key, m, L, R, fast)
                deltas = rec.delta_qs()
                out = torch.empty(seq.shape, dtype=torch.uint8, device="cuda")
                rec.apply_bam(dd[0], dd[1], out, dd[4], dd[5], fast=fast)
                rec.check_status()
                wo = oracle_mod.apply_bam(seq, qual, rg, flags, L, R, tables[0], *deltas, minscore=m)
                assert np.array_equal(out.cpu().numpy().astype(np.int16), wo), (m, L, R, fast)


@pytest.mark.gpu
def test_minscore_43_is_refused_everywhere(torch_cuda):
    """No quality reaches minscore 43: every entry point refuses it as a bad argument (KbbqNativeError)."""
    torch = torch_cuda
    n = _native()
    from kbbq import synth
    from kbbq.device import DeviceRecalibrator
    L, R = 37, 2
    h = synth.synth_reads(5, 0, 64, L, R)
    d = _dev(torch, *h)
    zeros = [np.zeros(s, np.int64) for s in ((R,), (R,), (R, 43), (R, 43, 2 * L), (R, 43, 17))]
    calls = [lambda p=p: _device_path(torch, d, L, R, p, minscore=43) for p in (0, 1, 2)]
    calls += [lambda: _segmented_path(torch, d, L, R, minscore=43),
              lambda: n.recalibrate_host(*h, L, R, minscore=43),
              lambda: n.Session(L, R, 43),
              lambda: n.build_host(*h, L, R, minscore=43),
              lambda: n.apply_host(h[0], h[1], h[3], h[4], L, R, *zeros, minscore=43)]
    err = (h[0] != h[2]).astype(np.uint8)
    for fast in (True, False):
        def bam_build(fast=fast):
            rec = DeviceRecalibrator(L, R, minscore=43)
            rec.build_bam(*_dev(torch, h[0], h[1], err), fast=fast)

        def bam_apply(fast=fast):
            rec = DeviceRecalibrator(L, R, minscore=43)
            rec.apply_bam(d[0], d[1], torch.empty_like(d[1]), d[3], None, fast=fast)
        calls += [bam_build, bam_apply]
    calls += [lambda: n.build_bam_host(h[0], h[1], err, None, h[3], None, None, None, L, R, minscore=43),
              lambda: n.apply_bam_host(h[0], h[1], h[3], None, L, R, *zeros, minscore=43)]
    for i, call in enumerate(calls):
        with pytest.raises(n.KbbqNativeError):
            call()


# ---------------------------------------------------------------------------------------------------------------
# D. bases outside ACGTN
# ---------------------------------------------------------------------------------------------------------------

BAD_BYTES = [ord("X"), ord("a"), ord("n"), ord("R"), ord("."), 0x00, 0xFF]
SITES = ["usable", "low_quality", "next_to_n"]


def _plant(seq, qual, r, pos, byte, site, minscore=6):
    L = seq.shape[1]
    seq[r, pos] = byte
    qual[r, pos] = 30 if site != "low_quality" else minscore - 4
    if site == "next_to_n":
        seq[r, pos - 1 if pos > 0 else pos + 1] = ord("N")


@pytest.fixture(scope="module")
def fastq_model(torch_cuda, oracle_mod):
    """A model built from clean reads: the apply-only entry points get reads that never went through a build."""
    from kbbq import synth
    L, R, N = 100, 2, 4000
    h = synth.synth_reads(31, 0, N, L, R)
    t = oracle_mod.covariate_arrays(*h, L, R)
    return L, R, h, t, oracle_mod.get_delta_qs(*t)


@pytest.mark.gpu
def test_fastq_apply_rejects_bases_outside_acgtn(torch_cuda, oracle_mod, fastq_model):
    """kbbq_apply (shared-memory, generic, segmented), kbbq_apply_host and compare_reads.recalibrate_fastq on
    reads with one byte outside ACGTN: TypeError, as the build and the host packer decide -- any such byte in the
    batch.  Afterwards the same recalibrator / entry point still works and matches the oracle."""
    torch = torch_cuda
    n = _native()
    from kbbq import compare_reads
    from kbbq.device import DeviceRecalibrator
    L, R, h, t, dq = fastq_model
    seq0, qual0, corr0, rg0, sec0 = (a[:512].copy() for a in h)
    rec = DeviceRecalibrator(L, R, max_reads=seq0.shape[0])
    for dst, src in zip((rec.meanq, rec.rgdq, rec.qdq, rec.posdq, rec.dindq), (t[0],) + tuple(dq)):
        dst.copy_(torch.from_numpy(src))
    want_clean = oracle_mod.apply(seq0, qual0, rg0, sec0, L, R, t[0], *dq)

    class Read:
        def __init__(self, s, q):
            self.sequence, self._q = s.tobytes().decode("latin-1"), q

        def get_quality_array(self):
            return self._q.tolist()

    failures = []
    for byte in BAD_BYTES:
        for pos in (0, L // 2, L - 1):
            for site in SITES:
                seq, qual = seq0.copy(), qual0.copy()
                r = 77
                _plant(seq, qual, r, pos, byte, site)
                s, q, g, sec = _dev(torch, seq, qual, rg0, sec0)
                for path in (1, 2, "segmented"):
                    rec.status.zero_()
                    out = torch.empty_like(q)
                    if path == "segmented":
                        sb = rec.segment(s, q, None, g, sec)
                        out_seg = torch.empty(sb.rows_bound * L + 16, dtype=torch.uint8, device="cuda")
                        rec.apply_segmented(sb, out_seg)
                    else:
                        rec.apply(s, q, out, g, sec, path=path)
                    try:
                        rec.check_status()
                        failures.append((byte, pos, site, path))
                    except TypeError:
                        pass
                try:
                    n.apply_host(seq, qual, rg0, sec0, L, R, t[0], *dq)
                    failures.append((byte, pos, site, "apply_host"))
                except TypeError:
                    pass
                g1 = int(rg0[r])
                if byte >= 0x80:   # not a one-character base of a FASTQ record's sequence string
                    continue
                try:
                    compare_reads.recalibrate_fastq(Read(seq[r], qual[r]), t[0], dq[0], dq[1], dq[2], dq[3], g1, None,
                                                    secondinpair=bool(sec0[r]))
                    failures.append((byte, pos, site, "recalibrate_fastq"))
                except TypeError:
                    pass
    assert not failures, "no TypeError for %d of %d cases, e.g. %s" % (
        len(failures), len(BAD_BYTES) * 3 * len(SITES) * 5 - 3 * len(SITES), failures[:8])
    # the recalibrator and the host entry point still work on clean reads
    s, q, g, sec = _dev(torch, seq0, qual0, rg0, sec0)
    for path in (1, 2):
        rec.status.zero_()
        out = torch.empty_like(q)
        rec.apply(s, q, out, g, sec, path=path)
        rec.check_status()
        assert np.array_equal(out.cpu().numpy().astype(np.int16), want_clean), path
    assert np.array_equal(n.apply_host(seq0, qual0, rg0, sec0, L, R, t[0], *dq).astype(np.int16), want_clean)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 3])
def test_apply_paths_agree_on_any_input(torch_cuda, fastq_model, R):
    """kbbq_apply path 1 (shared memory) and path 2 (generic): identical bytes and identical status word for
    arbitrary bytes in seq and qualities up to 127 (beyond that the call raises IndexError, and the byte-parallel
    arithmetic of the shared-memory kernel no longer keeps the qualities of neighbouring bytes apart)."""
    torch = torch_cuda
    from kbbq.device import DeviceRecalibrator
    L, _, h, t, dq = fastq_model
    rng = np.random.default_rng(R)
    N = 4096 + 5
    seq = np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, (N, L))]
    junk = rng.random((N, L)) < 0.01
    seq = np.where(junk, rng.integers(0, 256, (N, L)), seq).astype(np.uint8)
    qual = rng.integers(0, 43, (N, L)).astype(np.uint8)
    qual = np.where(rng.random((N, L)) < 0.002, rng.integers(43, 128, (N, L)), qual).astype(np.uint8)
    rg = rng.integers(0, R, N).astype(np.uint16)
    second = rng.integers(0, 2, N).astype(np.uint8)
    rec = DeviceRecalibrator(L, R, max_reads=N)
    for i in range(R):   # the clean model's first read group for every group
        rec.meanq[i], rec.rgdq[i] = int(t[0][0]), int(dq[0][0])
        rec.qdq[i].copy_(torch.from_numpy(dq[1][0]))
        rec.posdq[i].copy_(torch.from_numpy(dq[2][0]))
        rec.dindq[i].copy_(torch.from_numpy(dq[3][0]))
    for rows in (slice(0, N), slice(0, 4096)):   # with and without good bases only in some batches
        s, q, g, sec = _dev(torch, seq[rows], qual[rows], rg[rows], second[rows])
        res = []
        for path in (1, 2):
            rec.status.zero_()
            out = torch.full_like(q, 7)
            rec.apply(s, q, out, g if R > 1 else None, sec, path=path)
            res.append((out.cpu().numpy(), int(rec.status.item())))
        assert np.array_equal(res[0][0], res[1][0]), R
        assert res[0][1] == res[1][1] and res[0][1] & 3 == 3, (res[0][1], res[1][1])


def _bam_run(torch, oracle, h, L, R, fast, views=0):
    """build_bam -> model -> apply_bam; -> ("ok", tables, deltas, out) or the exception type raised."""
    from kbbq.device import DeviceRecalibrator
    seq, qual, err, skip, rg, flags, a0, a1 = h

    def dev(a):
        if a is None:
            return None
        t = _dev(torch, a)[0]
        if not views or a.ndim != 2:
            return t
        buf = torch.empty(t.numel() + 16, dtype=t.dtype, device="cuda")   # a view at a byte offset of 1..3
        v = buf[views:views + t.numel()].view(t.shape)
        v.copy_(t)
        return v
    rec = DeviceRecalibrator(L, R, minscore=6)
    try:
        dd = [dev(a) for a in h]
        rec.build_bam(*dd, fast=fast)
        tables = rec.covariate_arrays()
        rec.check_status()
        deltas = rec.delta_qs()
    except TypeError:
        return ("TypeError",)
    try:
        out = torch.empty(seq.shape, dtype=torch.uint8, device="cuda")
        rec.apply_bam(dd[0], dd[1], out, dd[4], dd[5], fast=fast)
        rec.check_status()
    except TypeError:
        return ("ok", tables, deltas, "TypeError")
    return ("ok", tables, deltas, out.cpu().numpy().astype(np.int16))


def _bam_oracle(oracle, h, L, R, tables=None, deltas=None):
    seq, qual, err, skip, rg, flags, a0, a1 = h
    try:
        wt = oracle.build_tables_bam(seq, qual, err, skip, rg, flags, a0, a1, L, R)
    except oracle.OracleError:
        return ("TypeError",)
    if tables is None:
        return ("ok", wt)
    try:
        wo = oracle.apply_bam(seq, qual, rg, flags, L, R, tables[0], *deltas)
    except oracle.OracleError:
        wo = "TypeError"
    return ("ok", wt, wo)


def _compare_bam(torch, oracle, h, L, R, what, views=0):
    fast = _bam_run(torch, oracle, h, L, R, True, views)
    direct = _bam_run(torch, oracle, h, L, R, False, views)
    assert fast[0] == direct[0], ("build", fast[0], direct[0]) + what
    want = _bam_oracle(oracle, h, L, R, *(direct[1:3] if direct[0] == "ok" else ()))
    assert want[0] == direct[0], ("oracle build", want[0], direct[0]) + what
    if direct[0] != "ok":
        return
    for key, a, b, c in zip(TABLE_KEYS[5:], fast[1][5:], direct[1][5:], want[1]):
        assert np.array_equal(a, b) and np.array_equal(b, c), (key,) + what
    for x, y in zip(fast[2], direct[2]):
        assert np.array_equal(x, y), what
    outs = (fast[3], direct[3], want[2])
    if any(isinstance(o, str) for o in outs):   # an exception: the same one everywhere
        assert all(isinstance(o, str) for o in outs), ("apply", [o if isinstance(o, str) else "ok" for o in outs]) + what
    else:
        assert np.array_equal(fast[3], direct[3]) and np.array_equal(direct[3], want[2]), ("apply",) + what


def _bam_batch(rng, N, L, R):
    from kbbq import synth
    seq, qual, corr, rg, second = synth.synth_reads(int(rng.integers(1, 1 << 30)), 0, N, L, R)
    err = (seq != corr).astype(np.uint8)
    skip = (rng.random((N, L)) < 0.05).astype(np.uint8)
    flags = rng.integers(0, 4, N).astype(np.uint8)
    a0 = (rng.integers(0, 4, N) * (rng.random(N) < 0.3)).astype(np.uint16)
    a1 = (L - rng.integers(0, 4, N) * (rng.random(N) < 0.3)).astype(np.uint16)
    return [seq, qual, err, skip, rg, flags, a0, a1]


@pytest.mark.gpu
def test_bam_fast_and_direct_agree_on_bases_outside_acgtn(torch_cuda, oracle_mod):
    """kbbq_build_bam / kbbq_apply_bam with and without a workspace on reads with one byte outside ACGTN at cycle 0,
    in the middle and at the end, at a usable site, a low-quality site and next to an N, forward and reverse: the
    reference's rule (TypeError for such a base in a usable dinucleotide of a forward read) on both paths, and the
    same tables and qualities when nothing is raised."""
    torch = torch_cuda
    rng = np.random.default_rng(404)
    L, R, N = 37, 2, 48
    base = _bam_batch(rng, N, L, R)
    base[3][:] = 0                         # no host skips: the planted byte is what decides
    base[6][:] = 0
    base[7][:] = L
    raised = 0
    for byte in BAD_BYTES:
        for pos in (0, L // 2, L - 1):
            for site in SITES:
                for reverse in (False, True):
                    h = [a.copy() for a in base]
                    r = 5
                    _plant(h[0], h[1], r, pos, byte, site)
                    h[5][r] = 2 if reverse else 0
                    _compare_bam(torch, oracle_mod, h, L, R, (byte, pos, site, reverse))
                    raised += _bam_oracle(oracle_mod, h, L, R)[0] == "TypeError"
    assert raised > 0


@pytest.mark.gpu
@pytest.mark.parametrize("L", [4, 5, 7, 37])
def test_bam_narrow_windows_and_offsets(torch_cuda, oracle_mod, L):
    """Aligned windows of 0 to 3 bases, windows reaching past the read, inverted ones, short reads, and source
    arrays at byte offsets 1 to 3: canonical form and direct kernels agree with the oracle.  pysam never returns a
    window past the read or an inverted one; for those the oracle states the library's documented rule (cut at L,
    empty), so they check that the paths agree with each other, not parity with the reference."""
    torch = torch_cuda
    rng = np.random.default_rng(L)
    N, R = 3001, 3
    h = _bam_batch(rng, N, L, R)
    kind = rng.integers(0, 4, N)
    start = rng.integers(0, L + 1, N)
    width = rng.integers(0, 4, N)
    a0 = np.where(kind == 0, start, h[6])
    a1 = np.where(kind == 0, np.minimum(start + width, L), h[7])
    a0 = np.where(kind == 1, rng.integers(0, L + 3, N), a0)          # past the read
    a1 = np.where(kind == 1, rng.integers(L, L + 5, N), a1)
    a0 = np.where(kind == 2, rng.integers(2, L + 2, N), a0)          # inverted
    a1 = np.where(kind == 2, a0 - rng.integers(1, 3, N), a1)
    h[6], h[7] = a0.clip(0, 65535).astype(np.uint16), a1.clip(0, 65535).astype(np.uint16)
    for views in (0, 1, 2, 3):
        _compare_bam(torch, oracle_mod, h, L, R, (L, views), views)


@pytest.mark.gpu
def test_bam_apply_only_rejects_like_the_direct_kernel(torch_cuda, oracle_mod, fastq_model):
    """kbbq_apply_bam on its own (a model from clean reads, reads that never went through kbbq_build_bam) with one
    byte outside ACGTN at cycle 0 / middle / last, at a usable site, a low-quality site and next to an N, forward
    and reverse: the canonical form (workspace) and the direct kernel raise the same exception, set the same status
    word and write the same bytes, and both agree with oracle_apply_bam."""
    torch = torch_cuda
    from kbbq.device import DeviceRecalibrator
    L, R, h, t, dq = fastq_model
    rng = np.random.default_rng(505)
    N = 64
    seq0, qual0 = h[0][:N].copy(), h[1][:N].copy()
    rg0 = h[3][:N].copy()
    flags0 = rng.integers(0, 4, N).astype(np.uint8)
    rec = DeviceRecalibrator(L, R)
    for dst, src in zip((rec.meanq, rec.rgdq, rec.qdq, rec.posdq, rec.dindq), (t[0],) + tuple(dq)):
        dst.copy_(torch.from_numpy(src))
    raised = 0
    for byte in BAD_BYTES:
        for pos in (0, L // 2, L - 1):
            for site in SITES:
                for reverse in (False, True):
                    seq, qual, flags = seq0.copy(), qual0.copy(), flags0.copy()
                    r = 9
                    _plant(seq, qual, r, pos, byte, site)
                    flags[r] = (flags[r] & 1) | (2 if reverse else 0)
                    s, q, g, f = _dev(torch, seq, qual, rg0, flags)
                    res = []
                    for fast in (True, False):
                        rec.status.zero_()
                        out = torch.full_like(q, 255)
                        rec.apply_bam(s, q, out, g, f, fast=fast)
                        res.append((int(rec.status.item()), out.cpu().numpy()))
                    what = (byte, pos, site, reverse)
                    assert res[0][0] == res[1][0], ("status", res[0][0], res[1][0]) + what
                    try:
                        want = oracle_mod.apply_bam(seq, qual, rg0, flags, L, R, t[0], *dq)
                    except oracle_mod.OracleError:
                        want = None
                    assert (want is None) == bool(res[1][0] & 2), ("oracle", want is None, res[1][0]) + what
                    if want is None:
                        raised += 1
                        continue
                    assert np.array_equal(res[0][1], res[1][1]), what
                    assert np.array_equal(res[1][1].astype(np.int16), want), what
    assert raised > 0


@pytest.mark.gpu
def test_apply_skips_the_base_check_only_for_batches_it_built(torch_cuda, oracle_mod):
    """DeviceRecalibrator.apply passes KBBQ_APPLY_BASES_CHECKED for the very tensor it built since the last reset,
    unchanged: the build has already flagged any base outside ACGTN in the same status word.  A batch written to
    since, or a reset in between, is checked again; with the flag the bytes are those of the checked apply."""
    torch = torch_cuda
    from kbbq import synth
    from kbbq.device import DeviceRecalibrator
    L, R, N = 100, 1, 4096
    h = synth.synth_reads(61, 0, N, L, R)
    s, q, c, g, sec = _dev(torch, *h)
    rec = DeviceRecalibrator(L, R, max_reads=N)
    rec.build(s, q, c, None, sec)
    rec.model()
    want = _oracle_all(oracle_mod, *h, L, R)[2]
    out = torch.empty_like(q)
    rec.apply(s, q, out, None, sec)
    rec.check_status()
    assert np.array_equal(out.cpu().numpy().astype(np.int16), want)
    # the same tensor, written to after the build: checked again
    s[17, 40] = ord("X")
    rec.apply(s, q, out, None, sec)
    with pytest.raises(TypeError):
        rec.check_status()
    # built with the bad base: the build raises, and so does the apply after it
    rec.reset()
    rec.build(s, q, c, None, sec)
    rec.apply(s, q, out, None, sec)
    with pytest.raises(TypeError):
        rec.check_status()
    # a reset forgets the build (and its status): the apply checks again
    rec.reset()
    rec.apply(s, q, out, None, sec)
    with pytest.raises(TypeError):
        rec.check_status()
    # the flag itself: no base check, the same bytes as the checked kernels
    for path in (1, 2):
        rec.status.zero_()
        o1, o2 = torch.empty_like(q), torch.empty_like(q)
        rec.apply(s, q, o1, None, sec, path=path)
        assert int(rec.status.item()) == 2, path
        rec.status.zero_()
        rec.apply(s, q, o2, None, sec, path=path | 0x10)
        assert int(rec.status.item()) == 0, path
        assert torch.equal(o1, o2), path
