"""The delta-Q model (csrc/model.cuh) at its numeric edges, bit for bit against exact and long-double references.

- meanq (marginals_rg_kernel) against an exact, rational p_to_q: single-quality read groups, random histograms, and
  read groups built from continued fractions whose mean error probability lies as close to a bucket boundary
  10^(-m/10) as totals up to 2^52 allow.  Inside a 2^-60 band around a boundary the oracle's long-double meanq may
  differ from the exact floor; the kernel gives the exact floor outside a 2^-96 band.
- The level kernels (delta_levels12_kernel, delta_level3_kernel) on planted tables: near ties at every level against
  the prior the earlier levels give, inconsistent cells (errs > tot), counts up to 2^45, R in {1, 3, 257},
  L in {1, 150, 300}, through kbbq_get_delta_qs_host and through a session; report-shaped calls (nq < 43, no cycle
  axis); the fold and the apply on the session's planted deltas.
- The real-prior posterior (posterior_q_real_kernel) against oracle_posterior_q_real.
- kbbq_marginals' read-group limit.
"""
import os
from decimal import Decimal, localcontext
from fractions import Fraction

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, load_case

NQ = 43
TIE = 2.0 ** -60        # the relative top-2 gap below which a cell counts as a near tie (as in test_gpu_parity)
BAND = 2.0 ** -60       # the relative distance from a p_to_q boundary inside which only the exact meanq is pinned
DD_BAND = 2.0 ** -96    # ... inside which not even that: the double-double mean may land on either side (DESIGN §4 K3)


# ---- exact meanq -------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def p_exact(oracle_mod):
    """KBBQ_P as exact rationals (the binary values of the doubles the kernel and the oracle use)."""
    return [Fraction(float(p)) for p in oracle_mod.constants()[0]]


def _mean_p(t, P):
    T = sum(int(x) for x in t)
    return None if T == 0 else sum(int(tq) * P[q] for q, tq in enumerate(t) if tq) / T


def exact_meanq(t, P):
    """p_to_q(sum_q t_q p_q / T) with no floating point: with P = num / den, P <= 10^(-m/10) <=> num^10 10^m <= den^10,
    and meanq = #{m in 1..42 : that holds} (the set is 1..meanq); T = 0 -> 0."""
    p = _mean_p(t, P)
    if p is None:
        return 0
    n10, d10 = p.numerator ** 10, p.denominator ** 10
    m = 0
    while m < NQ - 1 and n10 * 10 ** (m + 1) <= d10:
        m += 1
    return m


def _dec(f):
    return Decimal(f.numerator) / Decimal(f.denominator)


def boundary_margin(t, P):
    """Relative distance of the exact mean error probability from the nearest bucket boundary 10^(-m/10), m = 1..42."""
    p = _mean_p(t, P)
    if p is None:
        return float("inf")
    with localcontext() as ctx:
        ctx.prec = 60
        pd = _dec(p)
        return float(min(abs(pd - b) / b for b in _boundaries()))


_BOUNDS = []


def _boundaries():
    """10^(-m/10), m = 1..42, to 60 digits."""
    if not _BOUNDS:
        with localcontext() as ctx:
            ctx.prec = 60
            _BOUNDS.extend(Decimal(10) ** (Decimal(-m) / 10) for m in range(1, NQ))
    return _BOUNDS


def near_boundary_histograms(P, tmax=2 ** 40):
    """Read groups of two neighbouring qualities a < b around a boundary B = 10^(-m/10), m = 2..41, with p_a > B > p_b:
    their mean is B when t_a / t_b = x = (B - p_b) / (p_a - B), and the continued-fraction convergents h / k of x
    (h + k <= tmax) put it as close to B as such counts can.  -> int64 [n, 43] histograms."""
    out = []
    with localcontext() as ctx:
        ctx.prec = 100
        for m in range(2, 42):
            B = Decimal(10) ** (Decimal(-m) / 10)
            for a, b in ((m - 1, m), (m, m + 1), (m - 1, m + 1)):
                pa, pb = _dec(P[a]), _dec(P[b])
                if not pb < B < pa:
                    continue
                y = (B - pb) / (pa - B)
                h0, h1, k0, k1 = 0, 1, 1, 0
                for _ in range(80):
                    ai = int(y)
                    h0, h1, k0, k1 = h1, ai * h1 + h0, k1, ai * k1 + k0
                    if h1 + k1 > tmax:
                        break
                    if h1 and k1:
                        t = np.zeros(NQ, np.int64)
                        t[a], t[b] = h1, k1
                        out.append(t)
                    if y == ai:
                        break
                    y = 1 / (y - ai)
    return np.array(out)


def random_histograms(rng, n, tmax):
    """n read groups over 1..43 random qualities with counts up to tmax."""
    t = np.zeros((n, NQ), np.int64)
    for i in range(n):
        qs = rng.choice(NQ, rng.integers(1, NQ + 1), replace=False)
        t[i, qs] = (10 ** rng.uniform(0, np.log10(tmax), qs.size)).astype(np.int64)
    return t


def _single_quality(ts):
    """[q, t] single-quality read groups, q = 0..42, for every t in ts."""
    return np.array([np.eye(NQ, dtype=np.int64)[q] * t for t in ts for q in range(NQ)])


def _marginals_tables(t):
    """L = 1 tables whose read group r has t[r, q] observations of quality q (one error in each nonempty cell)."""
    pt = np.zeros((t.shape[0], NQ, 2), np.int64)
    pt[:, :, 1] = t
    return np.minimum(pt, 1), pt


# ---- planted tables ----------------------------------------------------------------------------------------------

EDGE_KINDS = ("errs = 0", "errs = tot", "tot = 0", "errs = tot + 1", "errs >= tot + 2")


def _edge_cells(rng, n, inconsistent):
    """inconsistent = 0: consistent kinds only; 1: also errs = tot + 1; 2: also errs >= tot + 2."""
    kind = rng.integers(0, 3 + inconsistent, n)
    tot = (10 ** rng.uniform(0, 13.5, n)).astype(np.int64)
    errs = np.where(kind == 1, tot, 0)
    tot[kind == 2] = 0
    errs = np.where(kind == 3, tot + 1, errs)
    errs = np.where(kind == 4, tot + 2 + rng.integers(0, 1000, n), errs)
    return errs, tot


def _cells(oracle, rng, priors, inconsistent, p_tie=0.5, p_edge=0.2, log10_hi=13.5):
    """Counts for cells with the given priors: near ties (oracle.near_tie_counts, 1e3 .. 10^log10_hi failures), edge
    cells and random cells with up to 2^45 observations.  The first cell is always a near tie."""
    priors = np.asarray(priors)
    pr = priors.ravel()
    n = pr.size
    kind = rng.choice(3, n, p=[p_tie, p_edge, 1 - p_tie - p_edge])
    kind[0] = 0
    tot = (10 ** rng.uniform(0, 13.5, n)).astype(np.int64)
    errs = np.rint(tot * 10 ** rng.uniform(-4.5, 0, n)).astype(np.int64)
    e, t = _edge_cells(rng, n, inconsistent)
    errs[kind == 1], tot[kind == 1] = e[kind == 1], t[kind == 1]
    sel = kind == 0
    e, t = oracle.near_tie_counts(pr[sel], int(rng.integers(1 << 30)), 3.0, log10_hi)
    errs[sel], tot[sel] = e, t
    return errs.reshape(priors.shape), tot.reshape(priors.shape)


def _chain(oracle, meanq, ge, gt, qe, qt):
    """The level-1 and level-2 priors the reference's get_delta_qs derives: meanq + rgdq, and + qdq."""
    nq = qt.shape[1]
    prior1 = meanq + oracle.gatk_delta_q(meanq, ge, gt)
    p1 = np.repeat(prior1[:, None], nq, 1)
    prior2 = p1 + oracle.gatk_delta_q(p1, qe, qt)
    return prior1, prior2


def plant_free_tables(oracle, R, L, seed, inconsistent=1):
    """Marginals and covariate tables planted independently (kbbq_get_delta_qs takes any tables): every level has
    near ties against the prior the levels above it give, edge cells and random cells.  -> the 9 tables."""
    rng = np.random.default_rng(seed)
    meanq = rng.integers(0, NQ, R)
    ge, gt = _cells(oracle, rng, meanq, inconsistent)
    prior1 = meanq + oracle.gatk_delta_q(meanq, ge, gt)
    qe, qt = _cells(oracle, rng, np.repeat(prior1[:, None], NQ, 1), inconsistent)
    _, prior2 = _chain(oracle, meanq, ge, gt, qe, qt)
    pe, pt = _cells(oracle, rng, np.repeat(prior2[:, :, None], 2 * L, 2), inconsistent)
    de, dt = _cells(oracle, rng, np.repeat(prior2[:, :, None], 16, 2), inconsistent)
    return meanq, ge, gt, qe, qt, pe, pt, de, dt


def plant_session_tables(oracle, R, L, seed, inconsistent=0):
    """Covariate tables whose marginals (what a session sums) carry near ties at every level.  Every (rg, q) has a
    dominant cycle-0 cell (1e11 .. 1e12 observations) that fixes its rate.  Read groups of kind 0 hold one quality
    only, so meanq is known and their one cell is a level-1 near tie; kind 1 has one 2^44-observation quality and
    level-2 near ties (1e6 .. 1e10 failures) in the others; kind 2 has level-3 near ties (1e3 .. 1e6 failures) in the
    other cycles.  Planted against the current chained priors and replanted where the cells moved them, until they
    hold.  Dinucleotide cells, outside the marginals, are planted against the final priors.  -> pe, pt, de, dt."""
    P = [Fraction(float(p)) for p in oracle.constants()[0]]
    rng = np.random.default_rng(seed)
    L2 = 2 * L
    pe, pt = np.zeros((R, NQ, L2), np.int64), np.zeros((R, NQ, L2), np.int64)
    pt[:, :, 0] = (10 ** rng.uniform(11, 12, (R, NQ))).astype(np.int64)
    pe[:, :, 0] = np.rint(pt[:, :, 0] * 10 ** rng.uniform(-4.2, -0.5, (R, NQ))).astype(np.int64)
    kind = np.arange(R) % 3
    q0 = rng.integers(0, NQ, R)
    for r in np.nonzero(kind == 0)[0]:
        pe[r], pt[r] = 0, 0
        mq = exact_meanq(np.eye(NQ, dtype=np.int64)[q0[r]], P)
        e, t = oracle.near_tie_counts([mq], int(rng.integers(1 << 30)), 3.0, 12.0)
        pe[r, q0[r], 0], pt[r, q0[r], 0] = e[0], t[0]
    k1 = np.nonzero(kind == 1)[0]
    pt[k1, q0[k1], 0] = 2 ** 44
    pe[k1, q0[k1], 0] = np.rint(2.0 ** 44 * 10 ** rng.uniform(-4.2, -0.5, k1.size)).astype(np.int64)
    other = np.ones((R, NQ), bool)
    other[np.arange(R), q0] = False
    lvl2 = (kind == 1)[:, None] & other                                 # (rg, q) cells holding level-2 near ties
    lvl3 = np.zeros((R, NQ, L2), bool)
    lvl3[kind == 2, :, 1:] = True                                       # cells holding level-3 near ties
    plant1 = np.full(R, -1)
    plant2 = np.full((R, NQ), -1)
    for _ in range(12):
        mq, ge, gt, qe, qt = oracle.marginals(pe, pt)
        prior1, prior2 = _chain(oracle, mq, ge, gt, qe, qt)
        redo2 = lvl2 & (plant1 != prior1)[:, None]
        redo3 = lvl3 & (plant2 != prior2)[:, :, None]
        if not redo2.any() and not redo3.any():
            break
        if redo2.any():
            e, t = oracle.near_tie_counts(np.broadcast_to(prior1[:, None], (R, NQ))[redo2],
                                          int(rng.integers(1 << 30)), 6.0, 10.0)
            pe[:, :, 0][redo2], pt[:, :, 0][redo2] = e, t
            plant1 = np.where(redo2.any(1), prior1, plant1)
        if redo3.any():
            e, t = _cells(oracle, rng, np.broadcast_to(prior2[:, :, None], (R, NQ, L2))[redo3], inconsistent,
                          p_tie=0.6, p_edge=0.1, log10_hi=6.0)
            t = np.minimum(t, 10 ** 7)                                   # the dominant cell keeps the rate of (rg, q)
            pe[redo3], pt[redo3] = np.minimum(e, t + inconsistent), t
            plant2 = np.where(redo3.any(2), prior2, plant2)
    de, dt = _cells(oracle, rng, np.repeat(prior2[:, :, None], 16, 2), inconsistent)
    return pe, pt, de, dt


def level_gaps(oracle, meanq, ge, gt, qe, qt, pe, pt, de, dt):
    """Relative top-2 gaps of every cell of levels 1, 2, 3 (cycle), 3 (dinucleotide) under the chained priors."""
    prior1, prior2 = _chain(oracle, meanq, ge, gt, qe, qt)
    gap = oracle.delta_q_top2_gap
    return (gap(meanq, ge, gt), gap(np.repeat(prior1[:, None], NQ, 1), qe, qt),
            gap(np.repeat(prior2[:, :, None], pt.shape[2], 2), pe, pt),
            gap(np.repeat(prior2[:, :, None], 16, 2), de, dt))


# ---- CPU: the references ------------------------------------------------------------------------------------------

def test_exact_meanq_single_quality_groups(oracle_mod, p_exact):
    """q -> p -> q: the exact floor, the oracle's long double and the reference's round trip agree on every quality."""
    s = load_case("scalars")
    t = _single_quality([1, 5, 2 ** 40, 10 ** 12])
    want = np.array([exact_meanq(x, p_exact) for x in t])
    assert np.array_equal(want, np.tile(s["p_to_q_roundtrip"], 4))
    assert np.array_equal(oracle_mod.marginals(*_marginals_tables(t))[0], want)
    assert exact_meanq(np.zeros(NQ, np.int64), p_exact) == 0


def test_exact_meanq_equals_oracle_off_the_boundaries(oracle_mod, p_exact):
    rng = np.random.default_rng(5)
    t = np.concatenate([random_histograms(rng, 1500, 2 ** 40), random_histograms(rng, 500, 2 ** 20)])
    t[:10] = 0
    t[:10, 0] = np.arange(10)                                         # all Q0 (p = 1), and one empty group
    margin = np.array([boundary_margin(x, p_exact) for x in t])
    keep = margin > BAND
    assert keep.sum() > 1900
    want = np.array([exact_meanq(x, p_exact) for x in t[keep]])
    assert np.array_equal(oracle_mod.marginals(*_marginals_tables(t[keep]))[0], want)
    assert len(set(want)) > 20


def test_near_boundary_histograms_sit_inside_the_band(oracle_mod, p_exact):
    """The continued-fraction read groups do come within 2^-60 of a boundary, and there the long-double oracle is no
    exact reference: it differs from the exact floor on some of them, and only inside the band.  With totals up to
    2^40 they stay outside the 2^-96 band of the double-double mean; up to 2^52 some come inside it."""
    t = near_boundary_histograms(p_exact)
    assert len(t) > 900
    margin = np.array([boundary_margin(x, p_exact) for x in t])
    assert (margin < BAND).sum() > 250 and 2.0 ** -90 < margin.min() < 2.0 ** -80
    t52 = near_boundary_histograms(p_exact, 2 ** 52)
    assert len(t52) > 1200 and (t52.sum(1) < 2 ** 53).all()
    assert sum(boundary_margin(x, p_exact) < DD_BAND for x in t52) > 100
    exact = np.array([exact_meanq(x, p_exact) for x in t])
    ld = oracle_mod.marginals(*_marginals_tables(t))[0]
    differ = ld != exact
    assert differ.sum() > 100
    assert (margin[differ] < BAND).all()


def test_double_double_boundaries_are_accurate():
    """KBBQ_BOUND_HI[m] + KBBQ_BOUND_LO[m] lies within 2^-104 (relative) of 10^(-m/10), m = 1..42: one term of the
    2^-96 band of meanq."""
    text = open(os.path.join(ROOT, "include", "kbbq_model_constants.h")).read()

    def table(name):
        body = text.split(name + "[KBBQ_NQ] = {")[1].split("}")[0]
        return [Decimal(float.fromhex(x.strip())) for x in body.split(",") if x.strip()]

    hi, lo = table("KBBQ_BOUND_HI"), table("KBBQ_BOUND_LO")
    assert len(hi) == len(lo) == NQ
    with localcontext() as ctx:
        ctx.prec = 60
        for m, b in enumerate(_boundaries(), start=1):
            assert abs(hi[m] + lo[m] - b) / b < Decimal(2) ** -104, m
            assert abs(lo[m]) <= Decimal(float.fromhex("0x1p-53")) * abs(hi[m])     # a canonical pair


def test_real_prior_oracle_at_integer_priors(oracle_mod):
    rng = np.random.default_rng(7)
    pq = rng.integers(0, NQ, 200_000)
    errs, tot = _cells(oracle_mod, rng, pq, inconsistent=2)
    want = oracle_mod.gatk_delta_q(pq, errs, tot) + pq
    assert np.array_equal(oracle_mod.posterior_q_real(pq.astype(np.float64), errs, tot), want)


@pytest.mark.parametrize("case,npz", [("tiny_r2", "tiny_r2"), ("tails_r2_second", "tails_r2_second"),
                                      ("sparse_r3", "report_sparse_r3")])
def test_real_prior_oracle_equals_golden_report(oracle_mod, case, npz):
    """The read-group table of a report the reference wrote: EmpiricalQuality = the real-prior posterior of
    EstimatedQReported (rounded to 5 decimals, kbbq/gatk/bqsr.py:289-297)."""
    from kbbq import recaltable
    from kbbq.gatk.bqsr import _estimated_q
    d = load_case(npz)
    est = _estimated_q(d["q_total"], d["rg_total"])
    post = oracle_mod.posterior_q_real(est, d["rg_errs"], d["rg_total"])
    keep = d["rg_total"] != 0
    table = recaltable.RecalibrationReport.fromfile(os.path.join(GOLDEN, "report_%s.txt" % case)).tables[2].data
    assert np.allclose(table["EstimatedQReported"].to_numpy(), est[keep], rtol=0, atol=5e-5)
    assert np.array_equal(table["EmpiricalQuality"].to_numpy(), post[keep].astype(np.float64))


@pytest.mark.parametrize("real", [False, True])
def test_near_tie_generator_for_given_priors(oracle_mod, real):
    """oracle.near_tie_counts builds, for the priors it is given, cells whose top-2 gap is below 2^-60, some of them
    exact ties of the 64-bit-significand sums (a blind random grid has none)."""
    rng = np.random.default_rng(11 + real)
    n = 1_200_000
    pq = np.round(rng.uniform(0, 42, n), 5) if real else rng.integers(0, NQ, n)
    errs, tot = oracle_mod.near_tie_counts(pq, 3, 10.0, 11.0)
    assert errs.shape == tot.shape == pq.shape and (errs >= 0).all() and (errs <= tot).all()
    _, gap = oracle_mod.posterior_q_real(pq.astype(np.float64), errs, tot, gap=True)
    if not real:
        assert np.array_equal(gap[:100_000], oracle_mod.delta_q_top2_gap(pq[:100_000], errs[:100_000], tot[:100_000]))
    assert (gap < TIE).sum() >= 8 and (gap == 0).sum() >= 5, ((gap < TIE).sum(), (gap == 0).sum())


def test_planted_tables_hold_near_ties_at_every_level(oracle_mod):
    """Both table planters put cells near a tie at every level under the priors the levels above actually give."""
    free = plant_free_tables(oracle_mod, 257, 4, 1, inconsistent=2)
    pe, pt, de, dt = plant_session_tables(oracle_mod, 257, 4, 2)
    sess = oracle_mod.marginals(pe, pt) + (pe, pt, de, dt)
    for tabs in (free, sess):
        for lvl, g in enumerate(level_gaps(oracle_mod, *tabs)):
            assert (g < 2.0 ** -30).sum() >= 10, (lvl, (g < 2.0 ** -30).sum())
    for g in level_gaps(oracle_mod, *free):
        assert (g < 2.0 ** -40).sum() >= 3
    # the counts reach 2^45, and the free tables hold every edge kind at every level
    assert max(int(a.max()) for a in free[1:]) >= 2 ** 44
    for e, t in zip(free[1::2], free[2::2]):
        assert (e == 0).any() and (e == t).any() and (t == 0).any() and (e == t + 1).any() and (e >= t + 2).any()


# ---- GPU: meanq ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_meanq_single_quality_groups_gpu():
    from kbbq import _native
    s = load_case("scalars")
    ts = [1, 5, 2 ** 40, 10 ** 12, 2 ** 52]
    mq, ge, gt, qe, qt = _native.marginals_host(*_marginals_tables(_single_quality(ts)))
    assert np.array_equal(mq, np.tile(s["p_to_q_roundtrip"], len(ts)))
    assert np.array_equal(gt, np.repeat(ts, NQ))


@pytest.mark.gpu
def test_meanq_random_histograms_gpu(oracle_mod, p_exact):
    """Random histograms, with counts up to 2^52 in the last ones: the kernel's two_prod (and the double of the
    total) is exact below 2^53, which bounds the counts a read group may hold for the exact floor."""
    from kbbq import _native
    rng = np.random.default_rng(21)
    t = np.concatenate([random_histograms(rng, 2000, 2 ** 40), random_histograms(rng, 300, 2 ** 46)])
    big = np.zeros((200, NQ), np.int64)
    for i in range(200):
        a, b = rng.choice(NQ, 2, replace=False)
        big[i, a], big[i, b] = rng.integers(1, 2 ** 51, 2)             # totals < 2^52
    t = np.concatenate([t, big, np.zeros((1, NQ), np.int64)])
    pe, pt = _marginals_tables(t)
    got = _native.marginals_host(pe, pt)
    want = oracle_mod.marginals(pe, pt)
    for a, b in zip(got[1:], want[1:]):
        assert np.array_equal(a, b)
    exact = np.array([exact_meanq(x, p_exact) for x in t])
    assert np.array_equal(got[0], exact)
    margin = np.array([boundary_margin(x, p_exact) for x in t])
    assert np.array_equal(got[0][margin > BAND], want[0][margin > BAND])


@pytest.mark.gpu
def test_meanq_near_boundaries_is_the_exact_floor(p_exact):
    """Continued-fraction read groups with totals up to 2^52: the kernel gives the exact floor on every one that lies
    outside the 2^-96 band its double-double mean allows (DESIGN.md §4 K3), hundreds of them inside the 2^-60 band
    where the long-double oracle is no reference.  The groups with T <= 2^40 are also scaled by an integer towards
    2^52: the same mean, with counts where the exactness of two_prod below 2^53 matters."""
    from kbbq import _native
    t = near_boundary_histograms(p_exact, 2 ** 52)
    small = t[t.sum(1) <= 2 ** 40]
    scale = np.maximum(1, (2 ** 52 - 1) // small.sum(1))
    t = np.concatenate([t, small * scale[:, None]])
    margin = np.array([boundary_margin(x, p_exact) for x in t])
    keep = margin > DD_BAND
    assert keep.sum() > 2000 and (margin[keep] < BAND).sum() > 500
    t = t[keep]
    got = _native.marginals_host(*_marginals_tables(t))[0]
    want = np.array([exact_meanq(x, p_exact) for x in t])
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, [(t[i].nonzero()[0].tolist(), t[i][t[i] > 0].tolist(), got[i], want[i]) for i in bad[:5]]


@pytest.mark.gpu
def test_marginals_read_group_limit():
    """R = 65535 is the largest grid the q marginals launch takes; R = 65536 is an argument error, refused before any
    copy or launch (the outputs stay as they were)."""
    from kbbq import _native
    lib = _native.lib()
    for R, rc_want in ((65535, 0), (65536, -1)):
        pe, pt = np.zeros((R, NQ, 2), np.int64), np.zeros((R, NQ, 2), np.int64)
        pt[:, 30, 0] = np.arange(R)
        pe[:, 30, 0] = np.arange(R) // 1000
        outs = [np.full((R, NQ), -7, np.int64), np.full((R, NQ), -7, np.int64)] + \
               [np.full(R, -7, np.int64) for _ in range(3)]
        rc = lib.kbbq_marginals_host(_native.ptr(pe), _native.ptr(pt), 1, R,
                                     *[_native.ptr(a) for a in (outs[0], outs[1], outs[2], outs[3], outs[4])],
                                     _native.DEVICE)
        assert rc == rc_want, (R, rc, lib.kbbq_strerror(rc).decode())
        if rc_want:
            assert all((a == -7).all() for a in outs)
        else:
            assert np.array_equal(outs[3], np.arange(R)) and np.array_equal(outs[2], np.arange(R) // 1000)
            assert outs[4][0] == 0 and (outs[4][1:] == load_case("scalars")["p_to_q_roundtrip"][30]).all()


# ---- GPU: the levels ----------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_inconsistent_cells_match_the_reference(oracle_mod):
    """errs >= tot + 2 (the reference scores candidate 0 at +inf: delta = -prior, posterior 0), errs = tot + 1,
    errs = tot and tot = 0, for every integer prior, through the cell kernel, the real-prior kernel and the levels."""
    from kbbq import _native
    pq = np.repeat(np.arange(NQ), 8)
    cells = [(7, 5), (5, 2), (2, 0), (10 ** 12, 10), (6, 5), (0, 0), (5, 5), (1, 0)]
    errs = np.tile([c[0] for c in cells], NQ).astype(np.int64)
    tot = np.tile([c[1] for c in cells], NQ).astype(np.int64)
    want = oracle_mod.gatk_delta_q(pq, errs, tot)
    assert (want[errs >= tot + 2] == -pq[errs >= tot + 2]).all()
    assert np.array_equal(_native.delta_q_host(pq, errs, tot), want)
    assert np.array_equal(_native.posterior_q_real_host(pq.astype(np.float64), errs, tot), want + pq)
    # the same cells at every level
    R = pq.size
    z = np.zeros((R, NQ, 2), np.int64)
    qe, qt = np.repeat(errs[:, None], NQ, 1), np.repeat(tot[:, None], NQ, 1)
    de, dt = np.repeat(qe[:, :, None], 16, 2), np.repeat(qt[:, :, None], 16, 2)
    tabs = (pq, errs, tot, qe, qt, z + qe[:, :, None], z + qt[:, :, None], de, dt)
    for a, b in zip(_native.get_delta_qs_host(*tabs), oracle_mod.get_delta_qs(*tabs)):
        assert np.array_equal(a, b)
    # planted tables holding every edge kind, through kbbq_get_delta_qs and through a session
    tabs = plant_free_tables(oracle_mod, 3, 150, 17, inconsistent=2)
    for a, b in zip(_native.get_delta_qs_host(*tabs), oracle_mod.get_delta_qs(*tabs)):
        assert np.array_equal(a, b)
    for R, L in ((3, 4), (3, 150)):
        pe, pt, de, dt = plant_session_tables(oracle_mod, R, L, 19 + R, inconsistent=2)
        assert (pe >= pt + 2).any() and (de >= dt + 2).any()
        marg = oracle_mod.marginals(pe, pt)
        with _native.Session(L, R) as s:
            s.set_tables(np.concatenate([pe.ravel(), pt.ravel(), de.ravel(), dt.ravel()]))
            got = s.model(want_deltas=True)
        for a, b in zip(got, (marg[0],) + oracle_mod.get_delta_qs(*marg, pe, pt, de, dt)):
            assert np.array_equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 3, 257])
@pytest.mark.parametrize("L", [1, 150, 300])
def test_levels_on_planted_tables(oracle_mod, R, L):
    """kbbq_get_delta_qs on independently planted marginals and covariate tables: near ties at every level against the
    chained priors, every edge kind, counts up to 2^45."""
    from kbbq import _native
    tabs = plant_free_tables(oracle_mod, R, L, 100 * R + L)
    got = _native.get_delta_qs_host(*tabs)
    want = oracle_mod.get_delta_qs(*tabs)
    for a, b, key in zip(got, want, ("rgdq", "qdq", "posdq", "dindq")):
        assert np.array_equal(a, b), (key, np.argwhere(a != b)[:5].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("R,L", [(1, 1), (3, 150), (257, 1), (3, 300)])
@pytest.mark.parametrize("inconsistent", [0, 1])
def test_session_model_on_planted_tables(oracle_mod, R, L, inconsistent):
    """Session.set_tables + model: the marginals, meanq and the four levels of planted covariate tables whose sums
    carry near ties at every level.  Without inconsistent cells, the session then applies one batch whose reads hit
    every (rg, q >= minscore, cycle, dinucleotide), which runs the fold on chained deltas no read-derived table gives."""
    from kbbq import _native
    pe, pt, de, dt = plant_session_tables(oracle_mod, R, L, 7 * R + L + inconsistent, inconsistent)
    marg = oracle_mod.marginals(pe, pt)
    want = oracle_mod.get_delta_qs(*marg, pe, pt, de, dt)
    with _native.Session(L, R) as s:
        s.set_tables(np.concatenate([pe.ravel(), pt.ravel(), de.ravel(), dt.ravel()]))
        meanq, *got = s.model(want_deltas=True)
        assert np.array_equal(meanq, marg[0])
        for a, b, key in zip(got, want, ("rgdq", "qdq", "posdq", "dindq")):
            assert np.array_equal(a, b), (key, np.argwhere(a != b)[:5].tolist())
        if inconsistent:
            return
        seq, qual, rg, second = _covering_batch(R, L, seed=R + L)
        out = np.full(qual.shape, 255, np.uint8)
        for lo in range(0, len(seq), s.chunk_reads):
            hi = lo + s.chunk_reads
            s.apply_chunk(seq[lo:hi], qual[lo:hi], rg[lo:hi], second[lo:hi], out[lo:hi])
        s.sync()
    ref = oracle_mod.apply(seq, qual, rg, second, L, R, marg[0], *want)
    # the apply writes the reference's integer sum as a byte
    assert np.array_equal(out, ref.astype(np.uint8)), np.argwhere(out != ref.astype(np.uint8))[:5].tolist()


DE_BRUIJN = np.frombuffer(b"AACAGATCCGCTGGTT", np.uint8)   # holds every dinucleotide once, read cyclically


def _covering_batch(R, L, seed, minscore=6):
    """Reads that hit every (rg, mate, q >= minscore, position, dinucleotide): for every (rg, mate, q), 16 reads of
    quality q throughout whose bases are the 16 rotations of DE_BRUIJN, so that at every position each dinucleotide
    ends in one of them, and one all-N read (no valid dinucleotide).  Then 512 random reads, qualities 0..42 (those
    below minscore pass through) and bases ACGTN."""
    assert len({DE_BRUIJN[i:i + 2].tobytes() for i in range(15)} | {DE_BRUIJN[[15, 0]].tobytes()}) == 16
    rng = np.random.default_rng(seed)
    g, sec, q, rot = [a.ravel() for a in np.meshgrid(np.arange(R), (0, 1), np.arange(minscore, NQ), np.arange(17),
                                                      indexing="ij")]
    seq = DE_BRUIJN[(np.arange(L)[None, :] + rot[:, None]) % 16]
    seq[rot == 16] = ord("N")
    qual = np.repeat(q.astype(np.uint8)[:, None], L, 1)
    nr = 512
    seq = np.concatenate([seq, np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, (nr, L), dtype=np.uint8)]])
    qual = np.concatenate([qual, rng.integers(0, NQ, (nr, L), dtype=np.uint8)])
    rg = np.concatenate([g, rng.integers(0, R, nr)]).astype(np.uint16)
    second = np.concatenate([sec, rng.integers(0, 2, nr)]).astype(np.uint8)
    return seq, qual, rg, second


@pytest.mark.gpu
def test_report_shaped_levels(oracle_mod):
    """The calls the report writer makes: nq < 43 qualities, no cycle axis, 16 dinucleotides; against gatk_delta_q
    chained level by level (the oracle's get_delta_qs assumes nq = 43)."""
    from kbbq import _native
    rng = np.random.default_rng(3)
    for R, nq in ((1, 1), (3, 7), (40, 42)):
        meanq = rng.integers(0, NQ, R)
        ge, gt = _cells(oracle_mod, rng, meanq, 1)
        prior1 = meanq + oracle_mod.gatk_delta_q(meanq, ge, gt)
        qe, qt = _cells(oracle_mod, rng, np.repeat(prior1[:, None], nq, 1), 1)
        qdq = oracle_mod.gatk_delta_q(np.repeat(prior1[:, None], nq, 1), qe, qt)
        prior2 = np.repeat((prior1[:, None] + qdq)[:, :, None], 16, 2)
        de, dt = _cells(oracle_mod, rng, prior2, 1)
        empty = np.zeros((R, nq, 0), np.int64)
        rgdq, q_got, pos_got, din_got = _native.get_delta_qs_host(meanq, ge, gt, qe, qt, empty, empty, de, dt)
        assert np.array_equal(rgdq, prior1 - meanq)
        assert np.array_equal(q_got, qdq)
        assert pos_got.shape == (R, nq, 0)
        assert np.array_equal(din_got[:, :, :16], oracle_mod.gatk_delta_q(prior2, de, dt))
        assert (din_got[:, :, 16] == 0).all()


# ---- GPU: the real prior ------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_real_prior_random_and_at_integers(oracle_mod):
    from kbbq import _native
    rng = np.random.default_rng(9)
    n = 300_000
    pr = np.round(rng.uniform(0, 42, n), 5)                           # as _estimated_q makes them
    errs, tot = _cells(oracle_mod, rng, pr, 1)
    assert np.array_equal(_native.posterior_q_real_host(pr, errs, tot), oracle_mod.posterior_q_real(pr, errs, tot))
    # integers: the real kernel equals the integer kernel
    pq = rng.integers(0, NQ, n)
    errs, tot = _cells(oracle_mod, rng, pq, 1)
    got = _native.posterior_q_real_host(pq.astype(np.float64), errs, tot)
    assert np.array_equal(got, _native.delta_q_host(pq, errs, tot) + pq)
    assert np.array_equal(got, oracle_mod.gatk_delta_q(pq, errs, tot) + pq)
    # just below and above an integer, where trunc(c - prior) steps
    k = rng.integers(0, NQ, n).astype(np.float64)
    eps = np.array([-1e-5, -1e-9, -1e-12, 1e-12, 1e-9, 1e-5])[rng.integers(0, 6, n)]
    near = k + eps
    ulp = rng.random(n) < 0.3
    near[ulp] = np.nextafter(k[ulp], np.where(eps[ulp] < 0, -np.inf, np.inf))
    near = np.clip(near, 0.0, 42.0)
    errs, tot = _cells(oracle_mod, rng, near, 1)
    assert np.array_equal(_native.posterior_q_real_host(near, errs, tot), oracle_mod.posterior_q_real(near, errs, tot))


@pytest.mark.gpu
def test_real_prior_near_ties_equal_long_double(oracle_mod):
    """A near-tie search with real priors (1e10 .. 1e11 failures): the kernel's x87-rounded sums against long double."""
    from kbbq import _native
    rng = np.random.default_rng(13)
    close = ties = 0
    for seed in range(2):
        pr = np.round(rng.uniform(0, 42, 2_000_000), 5)
        errs, tot = oracle_mod.near_tie_counts(pr, 200 + seed, 10.0, 11.0)
        want, gap = oracle_mod.posterior_q_real(pr, errs, tot, gap=True)
        got = _native.posterior_q_real_host(pr, errs, tot)
        assert np.array_equal(got, want), np.nonzero(got != want)[0][:5]
        close += int((gap < TIE).sum())
        ties += int((gap == 0).sum())
    assert close >= 10 and ties >= 5, (close, ties)
