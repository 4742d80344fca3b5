// model.cuh -- K3: marginal tables, meanq and the hierarchical Bayesian delta-Q tables (fp64).
//
// Replaces the rg_* / q_* tallies and the meanq line of fastq_to_covariate_arrays
// (kbbq/recalibrate.py:111-115,120), compare_reads.gatk_delta_q (kbbq/compare_reads.py:235-260)
// and gatk.applybqsr.get_delta_qs (kbbq/gatk/applybqsr.py:80-103).  A few thousand cells x 43
// candidates: latency-bound, not a roofline kernel; it exists on the GPU so that the
// build -> model -> apply pipeline never leaves the device.
#pragma once
#include "common.cuh"

namespace kbbq {

__constant__ double c_lnp[NQ];
__constant__ double c_ln1mp[NQ];
__constant__ double c_prior[NQ];
__constant__ double c_p[NQ];
// 10^(-m/10) as unevaluated double-double sums (hi + lo), the p_to_q bucket boundaries
__constant__ double c_bound_hi[NQ];
__constant__ double c_bound_lo[NQ];

// ---- double-double helpers (error-free transforms; no contraction wanted, hence the _rn forms) --
struct dd { double hi, lo; };
__device__ __forceinline__ dd two_sum(double a, double b) {
    double s = __dadd_rn(a, b), bb = __dsub_rn(s, a);
    double e = __dadd_rn(__dsub_rn(a, __dsub_rn(s, bb)), __dsub_rn(b, bb));
    return {s, e};
}
__device__ __forceinline__ dd two_prod(double a, double b) {
    double p = __dmul_rn(a, b);
    return {p, __fma_rn(a, b, -p)};
}
__device__ __forceinline__ dd dd_add(dd a, dd b) {
    dd s = two_sum(a.hi, b.hi);
    double lo = __dadd_rn(s.lo, __dadd_rn(a.lo, b.lo));
    return two_sum(s.hi, lo);
}
__device__ __forceinline__ dd dd_div_d(dd a, double b) {  // a / b, b exact
    double q1 = __ddiv_rn(a.hi, b);
    dd p = two_prod(q1, b);
    double r = __dadd_rn(__dsub_rn(__dsub_rn(a.hi, p.hi), p.lo), a.lo);
    double q2 = __ddiv_rn(r, b);
    return two_sum(q1, q2);
}
__device__ __forceinline__ bool dd_le(dd a, double bh, double bl) {  // a <= (bh + bl)
    return a.hi < bh || (a.hi == bh && a.lo <= bl);
}

// ---- marginals ----------------------------------------------------------------------------------
// block (q, rg): q_errs/q_total[rg][q] = sum over the cycle axis
__global__ void marginals_q_kernel(const long long *pos_errs, const long long *pos_total, int L2,
                                   long long *q_errs, long long *q_total) {
    const int q = blockIdx.x, rg = blockIdx.y;
    const size_t base = ((size_t)rg * NQ + q) * L2;
    long long e = 0, t = 0;
    for (int c = threadIdx.x; c < L2; c += blockDim.x) { e += pos_errs[base + c]; t += pos_total[base + c]; }
    __shared__ long long se[32], st[32];
    for (int o = 16; o; o >>= 1) { e += __shfl_down_sync(0xFFFFFFFFu, e, o); t += __shfl_down_sync(0xFFFFFFFFu, t, o); }
    if ((threadIdx.x & 31) == 0) { se[threadIdx.x >> 5] = e; st[threadIdx.x >> 5] = t; }
    __syncthreads();
    if (threadIdx.x == 0) {
        e = 0; t = 0;
        for (int w = 0; w < (blockDim.x + 31) / 32; ++w) { e += se[w]; t += st[w]; }
        q_errs[rg * NQ + q] = e;
        q_total[rg * NQ + q] = t;
    }
}

// rg_* and meanq of every read group.
// expected_errs = sum_q q_total * p_q, p = expected / rg_total, meanq = trunc(-10 log10 p) clipped
// to [0, 42] (kbbq/compare_reads.py:262-267).  The reference does this in x87 long double; here the
// sum and the quotient are carried in double-double (~106 bits) and, since
// floor(-10 log10 p) = #{m in 1..42 : p <= 10^(-m/10)}, the logarithm is replaced by comparisons
// against double-double bucket boundaries, so no transcendental rounding is involved.
// One block per read group: the 86 counts are fetched by 43 threads at once (one thread walking them
// paid 43 dependent round trips, 13 us), then thread 0 adds them up in the order the reference does.
__global__ void marginals_rg_kernel(const long long *q_errs, const long long *q_total, int R,
                                    long long *rg_errs, long long *rg_total, long long *meanq) {
    const int rg = blockIdx.x;
    __shared__ long long s_e[NQ], s_t[NQ];
    if (threadIdx.x < NQ) {
        s_e[threadIdx.x] = q_errs[rg * NQ + threadIdx.x];
        s_t[threadIdx.x] = q_total[rg * NQ + threadIdx.x];
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    long long e = 0, t = 0;
    dd acc = {0.0, 0.0};
    for (int q = 0; q < NQ; ++q) {
        const long long tq = s_t[q];
        e += s_e[q];
        t += tq;
        if (tq) acc = dd_add(acc, two_prod((double)tq, c_p[q]));  // counts < 2^53 are exact
    }
    rg_errs[rg] = e;
    rg_total[rg] = t;
    long long mq = 0;
    if (t > 0) {
        if (acc.hi == 0.0) mq = NQ - 1;
        else {
            const dd p = dd_div_d(acc, (double)t);
            for (int m = 1; m < NQ; ++m) mq += dd_le(p, c_bound_hi[m], c_bound_lo[m]) ? 1 : 0;
        }
    }
    meanq[rg] = mq;  // t == 0: nan -> int -> clip gives 0 in the reference
}

// s = hi + lo exactly (two_sum).  The value an x87 extended-precision add returns for it: rounded to a 64-bit
// significand, ties to even, as a canonical (hi, lo) pair (hi = nearest double, lo = the rest), so that equal
// fp80 values give equal pairs and a lexicographic compare orders them as the fp80 values.
__device__ __forceinline__ dd round_to_x87(dd s) {
    if (s.lo == 0.0 || isinf(s.hi) || isnan(s.hi)) return s;
    int e;
    frexp(s.hi, &e);
    int eh = e - 1;  // floor(log2 |hi|)
    // hi a power of two and lo of the other sign: the sum lies in the binade below, with half the quantum
    if (fabs(s.hi) == ldexp(1.0, eh) && ((s.hi > 0.0) != (s.lo > 0.0))) eh -= 1;
    const int qe = eh - 63;  // exponent of the last of 64 significand bits
    // hi is a multiple of 2^11 quanta (even), so rounding the sum is rounding lo; rint = round half to even
    const double lo_r = ldexp(rint(ldexp(s.lo, -qe)), qe);
    const double h = __dadd_rn(s.hi, lo_r);
    return {h, __dadd_rn(__dsub_rn(s.hi, h), lo_r)};
}

// ---- gatk_delta_q -------------------------------------------------------------------------------
// posterior[c] = prior_dist[|c - prior|] + ((errs+1) ln p_c + (tot+1-errs) log1p(-p_c)); the
// reference adds the fp64 log-likelihood to an x87 long-double prior (kbbq/compare_reads.py:257-258), i.e.
// the sum is rounded to a 64-bit significand: the exact sum (two_sum) is rounded the same way and the
// candidates compared on that value.  First maximum wins (np.argmax); a +inf log-likelihood (errs >= tot + 2)
// gives candidate 0.
// `prior` is an integer quality, or (PRIOR = double: the read-group row of a recalibration report,
// kbbq/gatk/bqsr.py:293-297) a real one: the reference truncates candidate - prior towards zero
// before taking the absolute value (kbbq/compare_reads.py:245).  Returns the MAP candidate.
template <typename PRIOR>
__device__ __forceinline__ int posterior_q_cell(PRIOR prior, long long errs, long long tot) {
    const double k = (double)(errs + 1), mm = (double)((tot + 2) - (errs + 1));
    int best = 0;
    double bh = 0.0, bl = 0.0;
    bool have = false;
    for (int c = 0; c < NQ; ++c) {
        int d = (int)((PRIOR)c - prior);
        d = d < 0 ? -d : d;
        const double pr = d < NQ ? c_prior[d] : -KBBQ_INF;  // prior outside 0..42: IndexError in the reference
        const double a = __dmul_rn(k, c_lnp[c]);
        const double b = (mm == 0.0) ? 0.0 : __dmul_rn(mm, c_ln1mp[c]);
        const double ll = __dadd_rn(a, b);
        double h, l;
        if (isinf(pr) || isinf(ll)) {
            // ll = +inf only at c = 0 of an inconsistent cell (errs >= tot + 2: (negative) * log1p(-1)).  The
            // reference's binom.logpmf is -inf at every candidate there (k > n), so np.argmax gives candidate 0.
            if (ll > 0.0) return c;
            h = -KBBQ_INF; l = 0.0;
        }
        else { dd s = round_to_x87(two_sum(pr, ll)); h = s.hi; l = s.lo; }
        if (!have || h > bh || (h == bh && l > bl)) { best = c; bh = h; bl = l; have = true; }
    }
    return best;
}
__device__ __forceinline__ int delta_q_cell(int prior, long long errs, long long tot) {
    return posterior_q_cell<int>(prior, errs, tot) - prior;
}

__global__ void delta_q_kernel(const long long *prior, const long long *errs, const long long *tot,
                               long long n, long long *out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = delta_q_cell((int)prior[i], errs[i], tot[i]);
}

__global__ void posterior_q_real_kernel(const double *prior, const long long *errs, const long long *tot,
                                        long long n, long long *out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = posterior_q_cell<double>(prior[i], errs[i], tot[i]);
}

struct DeltaArgs {
    const long long *meanq, *rg_errs, *rg_total, *q_errs, *q_total, *pos_errs, *pos_total, *din_errs, *din_total;
    int R, nq, ncyc, ndin;
    long long *rgdq, *qdq, *posdq, *dindq;
};

// levels 1 and 2: block per read group
__global__ void delta_levels12_kernel(DeltaArgs a) {
    const int rg = blockIdx.x;
    __shared__ int s_prior1;
    if (threadIdx.x == 0) {
        const int mq = (int)a.meanq[rg];
        const int d = delta_q_cell(mq, a.rg_errs[rg], a.rg_total[rg]);
        a.rgdq[rg] = d;
        s_prior1 = mq + d;
    }
    __syncthreads();
    for (int q = threadIdx.x; q < a.nq; q += blockDim.x)
        a.qdq[rg * a.nq + q] = delta_q_cell(s_prior1, a.q_errs[rg * a.nq + q], a.q_total[rg * a.nq + q]);
}

// level 3: thread per (rg, q, covariate) cell; cycle cells first, then dinuc cells (+ zero pad)
__global__ void delta_level3_kernel(DeltaArgs a) {
    const long long ncell_pos = (long long)a.R * a.nq * a.ncyc;
    const long long ncell_din = (long long)a.R * a.nq * (a.ndin + 1);
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ncell_pos) {
        const long long gq = i / a.ncyc;
        const int rg = (int)(gq / a.nq);
        const int prior2 = (int)(a.meanq[rg] + a.rgdq[rg] + a.qdq[gq]);
        a.posdq[i] = delta_q_cell(prior2, a.pos_errs[i], a.pos_total[i]);
    } else if (i < ncell_pos + ncell_din) {
        i -= ncell_pos;
        const long long gq = i / (a.ndin + 1);
        const int d = (int)(i - gq * (a.ndin + 1));
        if (d == a.ndin) { a.dindq[i] = 0; return; }
        const int rg = (int)(gq / a.nq);
        const int prior2 = (int)(a.meanq[rg] + a.rgdq[rg] + a.qdq[gq]);
        a.dindq[i] = delta_q_cell(prior2, a.din_errs[gq * a.ndin + d], a.din_total[gq * a.ndin + d]);
    }
}

// ---- fold: reference-shaped int64 delta tables -> the two small tables the apply kernel gathers --
// With pad = dindq[rg][q][ndin1-1] (the column the dinuc index -1 gathers, kbbq/gatk/applybqsr.py:98-101):
// fold_cyc[rg][q][c2] = meanq + rgdq + qdq + posdq + pad      (q < nq, else 0)
// fold_din[rg][q][n]  = dindq[rg][q][ref(n)] - pad            for natural-order dinuc n < 16
// so an invalid dinucleotide contributes nothing on top of fold_cyc.
__global__ void fold_kernel(const long long *meanq, const long long *rgdq, const long long *qdq,
                            const long long *posdq, const long long *dindq, int R, int nq, int L2,
                            int ndin1, short *fold_cyc, short *fold_din) {
    const long long ncyc = (long long)R * NQ * L2, ndin = (long long)R * NQ * 16;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ncyc) {
        const long long gq = i / L2;
        const int c2 = (int)(i - gq * L2);
        const int rg = (int)(gq / NQ), q = (int)(gq - (long long)rg * NQ);
        long long v = 0;
        if (q < nq)
            v = meanq[rg] + rgdq[rg] + qdq[rg * nq + q] + posdq[((size_t)rg * nq + q) * L2 + c2] +
                dindq[((size_t)rg * nq + q) * ndin1 + ndin1 - 1];
        fold_cyc[i] = (short)v;
    } else if (i < ncyc + ndin) {
        i -= ncyc;
        const long long gq = i >> 4;
        const int n = (int)(i & 15);
        const int rg = (int)(gq / NQ), q = (int)(gq - (long long)rg * NQ);
        long long v = 0;
        if (q < nq) {
            const size_t row = ((size_t)rg * nq + q) * ndin1;
            v = dindq[row + nat_to_ref(n >> 2) * 4 + nat_to_ref(n & 3)] - dindq[row + ndin1 - 1];
        }
        fold_din[i] = (short)v;
    }
}

}  // namespace kbbq
