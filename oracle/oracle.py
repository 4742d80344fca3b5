"""ctypes front end of the CPU parity oracle (oracle/kbbq_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs -- never by the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libkbbq_oracle.so")
NQ = 43

_lib = None


def build(force=False):
    src = os.path.join(HERE, "kbbq_oracle.c")
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", HERE, "-B", "libkbbq_oracle.so"])
    return LIB


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            build()
        _lib = C.CDLL(LIB)
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


class OracleError(Exception):
    pass


def _check(st):
    if st:
        raise OracleError({-1: "quality > 42", -2: "base outside ACGTN", -3: "rg >= R"}.get(st, st))


def constants():
    out = [np.zeros(NQ) for _ in range(4)]
    lib().oracle_constants(*[_p(a) for a in out])
    return out


def build_tables(seq, qual, corr, rg, second, L, R, minscore=6, threads=0):
    """-> pos_errs, pos_total [R,43,2L], din_errs, din_total [R,43,16] (int64)."""
    seq, qual, corr = _u8(seq).ravel(), _u8(qual).ravel(), _u8(corr).ravel()
    N = seq.size // L if L else 0
    rg = None if rg is None else np.ascontiguousarray(rg, dtype=np.uint16)
    second = None if second is None else _u8(second)
    tabs = [np.zeros((R, NQ, 2 * L), np.int64), np.zeros((R, NQ, 2 * L), np.int64),
            np.zeros((R, NQ, 16), np.int64), np.zeros((R, NQ, 16), np.int64)]
    args = [_p(seq), _p(qual), _p(corr), _p(rg), _p(second), C.c_int64(N), C.c_int(L), C.c_int(R),
            C.c_int(minscore)] + [_p(t) for t in tabs]
    if threads:
        st = lib().oracle_build_mt(*args, C.c_int(threads))
    else:
        st = lib().oracle_build(*args)
    _check(st)
    return tabs


def marginals(pos_errs, pos_total):
    """-> meanq, rg_errs, rg_total, q_errs, q_total (the first five of the reference's 9-tuple)."""
    R, _, L2 = pos_total.shape
    q_e, q_t = np.zeros((R, NQ), np.int64), np.zeros((R, NQ), np.int64)
    g_e, g_t, mq = np.zeros(R, np.int64), np.zeros(R, np.int64), np.zeros(R, np.int64)
    lib().oracle_marginals(_p(_i64(pos_errs)), _p(_i64(pos_total)), C.c_int(L2 // 2), C.c_int(R),
                           _p(q_e), _p(q_t), _p(g_e), _p(g_t), _p(mq))
    return mq, g_e, g_t, q_e, q_t


def covariate_arrays(seq, qual, corr, rg, second, L, R, minscore=6):
    """The reference's fastq_to_covariate_arrays 9-tuple (kbbq/recalibrate.py:121)."""
    pe, pt, de, dt = build_tables(seq, qual, corr, rg, second, L, R, minscore)
    mq, g_e, g_t, q_e, q_t = marginals(pe, pt)
    return mq, g_e, g_t, q_e, q_t, pe, pt, de, dt


def p_to_q(p):
    p = np.ascontiguousarray(p, dtype=np.float64)
    q = np.zeros(p.shape, np.int64)
    lib().oracle_p_to_q(_p(p), C.c_int64(p.size), _p(q))
    return q


def gatk_delta_q(prior_q, numerrs, numtotal):
    prior_q, numerrs, numtotal = _i64(prior_q), _i64(numerrs), _i64(numtotal)
    assert prior_q.shape == numerrs.shape == numtotal.shape
    out = np.zeros(prior_q.shape, np.int64)
    lib().oracle_gatk_delta_q(_p(prior_q), _p(numerrs), _p(numtotal), C.c_int64(prior_q.size), _p(out))
    return out


def delta_q_top2_gap(prior_q, numerrs, numtotal):
    """Relative gap between the two best posteriors of every cell (long double): how close to a tie."""
    prior_q, numerrs, numtotal = _i64(prior_q), _i64(numerrs), _i64(numtotal)
    out = np.zeros(prior_q.shape, np.float64)
    lib().oracle_delta_q_top2_gap(_p(prior_q), _p(numerrs), _p(numtotal), C.c_int64(prior_q.size), _p(out))
    return out


def near_tie_cells(n, seed, log10_lo=3.0, log10_hi=11.0):
    """Cells of gatk_delta_q whose two best candidates are as close as integer counts allow: for a random prior, a
    random adjacent candidate pair (c, c + 1) and a random failure count m, the error count that balances the two
    posteriors.  -> (prior, errs, total).  A blind random grid never comes near a tie; these do (with m >= 1e10 a
    few per million are exact ties of the 64-bit-significand sums)."""
    _, lnp, ln1mp, prior = constants()
    rng = np.random.default_rng(seed)
    pq = rng.integers(0, 43, n)
    c = rng.integers(1, 42, n)
    m = (10 ** rng.uniform(log10_lo, log10_hi, n)).astype(np.int64)
    d1, d2 = np.abs(c - pq), np.abs(c + 1 - pq)
    ok = (d1 < 19) & (d2 < 19)   # both priors finite
    pq, c, m, d1, d2 = pq[ok], c[ok], m[ok], d1[ok], d2[ok]
    k = np.rint(-((prior[d1] - prior[d2]) + m * (ln1mp[c] - ln1mp[c + 1])) / (lnp[c] - lnp[c + 1])).astype(np.int64)
    ok = k >= 1
    pq, m, k = pq[ok], m[ok], k[ok]
    return pq, k - 1, m + k - 2


def posterior_q_real(prior_q, numerrs, numtotal, gap=False):
    """gatk_delta_q(prior, ...) + prior for real priors (the read-group table of a recalibration report); with gap, also
    the relative gap between the two best posteriors of every cell."""
    prior_q = np.ascontiguousarray(prior_q, dtype=np.float64)
    numerrs, numtotal = _i64(numerrs), _i64(numtotal)
    assert prior_q.shape == numerrs.shape == numtotal.shape
    out = np.zeros(prior_q.shape, np.int64)
    rel = np.zeros(prior_q.shape, np.float64) if gap else None
    lib().oracle_posterior_q_real(_p(prior_q), _p(numerrs), _p(numtotal), C.c_int64(prior_q.size), _p(out), _p(rel))
    return (out, rel) if gap else out


def near_tie_counts(priors, seed, log10_lo=3.0, log10_hi=11.0):
    """near_tie_cells for the given priors (integer or real, in [0, 42]): for every prior, a random adjacent candidate
    pair (c, c + 1) within 18 of it and a random failure count m, the error count that balances the two posteriors by
    the same formula.  The candidate distance is |trunc(c - prior)|, as the real-prior posterior takes it.
    -> (errs, total), int64, shaped like priors."""
    _, lnp, ln1mp, prior = constants()
    rng = np.random.default_rng(seed)
    pq = np.asarray(priors, dtype=np.float64).ravel()
    errs, tot = np.zeros(pq.size, np.int64), np.zeros(pq.size, np.int64)
    todo = np.arange(pq.size)
    while todo.size:
        p = pq[todo]
        c = np.clip(np.floor(p).astype(np.int64) + rng.integers(-17, 18, todo.size), 1, 41)
        m = (10 ** rng.uniform(log10_lo, log10_hi, todo.size)).astype(np.int64)
        d1, d2 = np.abs(np.trunc(c - p)).astype(np.int64), np.abs(np.trunc(c + 1 - p)).astype(np.int64)
        ok = (d1 < 19) & (d2 < 19)   # both priors finite
        k = np.zeros(todo.size, np.int64)
        k[ok] = np.rint(-((prior[d1[ok]] - prior[d2[ok]]) + m[ok] * (ln1mp[c[ok]] - ln1mp[c[ok] + 1]))
                        / (lnp[c[ok]] - lnp[c[ok] + 1])).astype(np.int64)
        ok &= k >= 1
        errs[todo[ok]], tot[todo[ok]] = k[ok] - 1, m[ok] + k[ok] - 2
        todo = todo[~ok]
    shape = np.shape(priors)
    return errs.reshape(shape), tot.reshape(shape)


def get_delta_qs(meanq, rg_errs, rg_total, q_errs, q_total, pos_errs, pos_total, din_errs, din_total):
    R, _, L2 = pos_total.shape
    rgdq = np.zeros(R, np.int64)
    qdq = np.zeros((R, NQ), np.int64)
    posdq = np.zeros((R, NQ, L2), np.int64)
    dindq = np.zeros((R, NQ, 17), np.int64)
    ins = [_i64(a) for a in (meanq, rg_errs, rg_total, q_errs, q_total, pos_errs, pos_total,
                             din_errs, din_total)]
    lib().oracle_get_delta_qs(*[_p(a) for a in ins], C.c_int(L2 // 2), C.c_int(R),
                              _p(rgdq), _p(qdq), _p(posdq), _p(dindq))
    return rgdq, qdq, posdq, dindq


def apply(seq, qual, rg, second, L, R, meanq, rgdq, qdq, posdq, dindq, minscore=6):
    """-> int16 [N, L] recalibrated qualities (kbbq/compare_reads.py:320-328)."""
    seq, qual = _u8(seq).ravel(), _u8(qual).ravel()
    N = seq.size // L if L else 0
    rg = None if rg is None else np.ascontiguousarray(rg, dtype=np.uint16)
    second = None if second is None else _u8(second)
    out = np.zeros((N, L), np.int16)
    ins = [_i64(a) for a in (meanq, rgdq, qdq, posdq, dindq)]
    st = lib().oracle_apply(_p(seq), _p(qual), _p(rg), _p(second), C.c_int64(N), C.c_int(L),
                            C.c_int(R), C.c_int(minscore), *[_p(a) for a in ins], _p(out))
    _check(st)
    return out


def build_tables_bam(seq, qual, err, skip, rg, flags, aln_start, aln_end, L, R, minscore=6):
    """BAM-side tally (kbbq/gatk/bqsr.py:86-118) -> pos_errs, pos_total, din_errs, din_total."""
    seq, qual, err = _u8(seq).ravel(), _u8(qual).ravel(), _u8(err).ravel()
    skip = None if skip is None else _u8(skip).ravel()
    N = seq.size // L if L else 0
    u16 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.uint16)
    rg, aln_start, aln_end = u16(rg), u16(aln_start), u16(aln_end)
    flags = None if flags is None else _u8(flags)
    tabs = [np.zeros((R, NQ, 2 * L), np.int64), np.zeros((R, NQ, 2 * L), np.int64),
            np.zeros((R, NQ, 16), np.int64), np.zeros((R, NQ, 16), np.int64)]
    st = lib().oracle_build_bam(_p(seq), _p(qual), _p(err), _p(skip), _p(rg), _p(flags), _p(aln_start), _p(aln_end),
                                C.c_int64(N), C.c_int(L), C.c_int(R), C.c_int(minscore), *[_p(t) for t in tabs])
    _check(st)
    return tabs


def apply_bam(seq, qual, rg, flags, L, R, meanq, rgdq, qdq, posdq, dindq, minscore=6):
    """recalibrate_bamread (kbbq/gatk/applybqsr.py:65-78) -> int16 [N, L]."""
    seq, qual = _u8(seq).ravel(), _u8(qual).ravel()
    N = seq.size // L if L else 0
    rg = None if rg is None else np.ascontiguousarray(rg, dtype=np.uint16)
    flags = None if flags is None else _u8(flags)
    out = np.zeros((N, L), np.int16)
    ins = [_i64(a) for a in (meanq, rgdq, qdq, posdq, dindq)]
    st = lib().oracle_apply_bam(_p(seq), _p(qual), _p(rg), _p(flags), C.c_int64(N), C.c_int(L), C.c_int(R),
                                C.c_int(minscore), *[_p(a) for a in ins], _p(out))
    _check(st)
    return out


def recalibrate(seq, qual, corr, rg, second, L, R, minscore=6, threads=0):
    """Whole path on host buffers -> int16 [N, L]."""
    seq, qual, corr = _u8(seq).ravel(), _u8(qual).ravel(), _u8(corr).ravel()
    N = seq.size // L if L else 0
    rg = None if rg is None else np.ascontiguousarray(rg, dtype=np.uint16)
    second = None if second is None else _u8(second)
    out = np.zeros((N, L), np.int16)
    st = lib().oracle_recalibrate(_p(seq), _p(qual), _p(corr), _p(rg), _p(second), C.c_int64(N),
                                  C.c_int(L), C.c_int(R), C.c_int(minscore), _p(out),
                                  C.c_int(threads))
    _check(st)
    return out


def max_threads():
    return int(lib().oracle_max_threads())
