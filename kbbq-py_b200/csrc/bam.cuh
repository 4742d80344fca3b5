// bam.cuh -- the BAM side of the path (SURVEY.md section 8 row f3): the same tally and the same
// gather as the FASTQ kernels, for aligned reads.
//
// build_bam_kernel replaces the loop body of bqsr.bam_to_bqsr_covariates (kbbq/gatk/bqsr.py:86-118)
// with bamread_bqsr_cycle (:23-31) and bamread_bqsr_dinuc (:33-50) fused in: errors and sites to skip
// come from the host (CIGAR walk against the reference, known variant sites, adaptor trimming:
// compare_reads.find_read_errors, bqsr.trim_bamread) as one byte per base; the kernel adds the
// q < minscore and N skips (:94-96), numbers cycles inside the aligned part of the read, backwards
// on the reverse strand, and takes the dinucleotide from the reverse complement there.
// apply_bam_kernel replaces applybqsr.recalibrate_bamread (kbbq/gatk/applybqsr.py:65-78) with
// bamread_cycle_covariates / bamread_dinuc_covariates (:46-63): no clipping, whole read.
//
// One thread per base, 64-bit global reductions / gathers from the int64 delta tables: these reads
// arrive one BAM record at a time from a host parser, so the kernels are sized for correctness and
// streaming batches, not for the shared-memory machinery of build.cuh / apply.cuh.
#pragma once
#include "common.cuh"

namespace kbbq {

constexpr int BAM_FLAG_READ2 = 1;
constexpr int BAM_FLAG_REVERSE = 2;

// reference order A T G C -> 0 1 2 3 (kbbq/compare_reads.py:199), N -> 4, anything else -> 5
__device__ __forceinline__ int bam_code(uint8_t b) {
    return b == 'A' ? 0 : b == 'T' ? 1 : b == 'G' ? 2 : b == 'C' ? 3 : b == 'N' ? 4 : 5;
}

// Dinucleotide index of base i of a read whose covariate window is [lo, hi): -1 when there is no
// previous base in read direction, the quality is below minscore or either base is N.  On the
// reverse strand the window is reverse-complemented first (complement.get(x, 'N'): anything that is
// not ACGT becomes N, kbbq/gatk/bqsr.py:40, kbbq/gatk/applybqsr.py:56), so the previous base is the
// complement of the NEXT one in stored order.  *bad is set for a non-ACGTN base at a usable site of a
// forward read (TypeError in the reference).
__device__ __forceinline__ int bam_dinuc(const uint8_t *row, int i, int lo, int hi, bool reverse, unsigned int q,
                                         int minscore, bool *bad) {
    if ((int)q < minscore) return -1;
    int cur = bam_code(row[i]), prev;
    if (reverse) {
        if (i + 1 >= hi) return -1;
        prev = bam_code(row[i + 1]);
        if (cur >= 4 || prev >= 4) return -1;
        return 4 * (prev ^ 1) + (cur ^ 1);   // A <-> T, G <-> C
    }
    if (i - 1 < lo) return -1;
    prev = bam_code(row[i - 1]);
    if (cur == 4 || prev == 4) return -1;
    if (cur == 5 || prev == 5) { *bad = true; return -1; }
    return 4 * prev + cur;
}

// An aligned window reaching past the read is cut at its end, and an inverted one is empty (the canonical form
// does the same): query_alignment_start / _end never exceed the read length, so this only keeps bad input in bounds.
__device__ __forceinline__ void bam_clamp_window(int L, int *lo, int *hi) {
    if (*lo > L) *lo = L;
    if (*hi > L) *hi = L;
    if (*hi < *lo) *hi = *lo;
}

struct BuildBamArgs {
    const uint8_t *seq, *qual, *err, *skip;
    const uint16_t *rg;
    const uint8_t *flags;
    const uint16_t *aln_start, *aln_end;
    long long N;
    int L, R, minscore;
    unsigned long long *pos_errs, *pos_total, *din_errs, *din_total;
    int *status;
};

__global__ void build_bam_kernel(BuildBamArgs a) {
    const long long total = a.N * a.L;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx / a.L;
        const int i = (int)(idx - r * a.L);
        const unsigned int q = a.qual[idx];
        const uint8_t s = a.seq[idx];
        if (a.skip && a.skip[idx]) continue;
        if ((int)q < a.minscore || s == 'N') continue;           // kbbq/gatk/bqsr.py:94-96
        if (q > NQ - 1) { atomicOr(a.status, KBBQ_FLAG_QUAL_RANGE); continue; }
        const unsigned int g = a.rg ? a.rg[r] : 0;
        if (g >= (unsigned int)a.R) { atomicOr(a.status, KBBQ_FLAG_RG_RANGE); continue; }
        const int fl = a.flags ? a.flags[r] : 0;
        int lo = a.aln_start ? a.aln_start[r] : 0, hi = a.aln_end ? a.aln_end[r] : a.L;
        bam_clamp_window(a.L, &lo, &hi);
        const bool reverse = fl & BAM_FLAG_REVERSE;
        int cyc = 0, din = 0;                                     // clipped bases keep 0 (:24,:43)
        if (i >= lo && i < hi) {
            const int c = reverse ? hi - 1 - i : i - lo;
            cyc = (fl & BAM_FLAG_READ2) ? -(c + 1) : c;
            bool bad = false;
            din = bam_dinuc(a.seq + r * a.L, i, lo, hi, reverse, q, a.minscore, &bad);
            if (bad) atomicOr(a.status, KBBQ_FLAG_BAD_BASE);
        }
        const bool e = a.err[idx] != 0;
        const int c2 = cyc < 0 ? 2 * a.L + cyc : cyc;
        const size_t po = ((size_t)g * NQ + q) * (2 * a.L) + c2;
        atomicAdd(a.pos_total + po, 1ull);
        if (e) atomicAdd(a.pos_errs + po, 1ull);
        if (din >= 0) {
            const size_t d = ((size_t)g * NQ + q) * 16 + din;
            atomicAdd(a.din_total + d, 1ull);
            if (e) atomicAdd(a.din_errs + d, 1ull);
        }
    }
}

struct ApplyBamArgs {
    const uint8_t *seq, *qual;
    const uint16_t *rg;
    const uint8_t *flags;
    uint8_t *out;
    long long N;
    int L, R, minscore, nq, ndin1;
    const long long *meanq, *rgdq, *qdq, *posdq, *dindq;
    int *status;
};

__global__ void apply_bam_kernel(ApplyBamArgs a) {
    const long long total = a.N * a.L;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx / a.L;
        const int i = (int)(idx - r * a.L);
        const unsigned int q = a.qual[idx];
        if ((int)q < a.minscore) { a.out[idx] = (uint8_t)q; continue; }
        if ((int)q >= a.nq) { atomicOr(a.status, KBBQ_FLAG_QUAL_RANGE); a.out[idx] = (uint8_t)q; continue; }
        const unsigned int g = a.rg ? a.rg[r] : 0;
        if (g >= (unsigned int)a.R) { atomicOr(a.status, KBBQ_FLAG_RG_RANGE); a.out[idx] = (uint8_t)q; continue; }
        const int fl = a.flags ? a.flags[r] : 0;
        const bool reverse = fl & BAM_FLAG_REVERSE;
        const int c = reverse ? a.L - 1 - i : i;                  // kbbq/gatk/applybqsr.py:46-50
        const int c2 = (fl & BAM_FLAG_READ2) ? 2 * a.L - 1 - c : c;
        bool bad = false;
        int din = bam_dinuc(a.seq + r * a.L, i, 0, a.L, reverse, q, a.minscore, &bad);
        if (bad) atomicOr(a.status, KBBQ_FLAG_BAD_BASE);
        if (din < 0) din = a.ndin1 - 1;                           // index -1 gathers the last column
        const size_t gq = (size_t)g * a.nq + q;
        const long long v = a.meanq[g] + a.rgdq[g] + a.qdq[gq] + a.dindq[gq * a.ndin1 + din] +
                            a.posdq[gq * (2 * a.L) + c2];
        a.out[idx] = (uint8_t)v;
    }
}

// ---- canonical form: the BAM side on the FASTQ kernels --------------------------------------------
// The direct kernels above hit a few thousand hot cells of the global tables with atomics from every
// SM (215 ms for 10 M x 150 bp with one read group).  Everything that distinguishes an aligned read
// from a FASTQ read is a permutation and a mask, so one streaming pass rewrites a batch into reads the
// shared-memory kernels (build.cuh / apply.cuh) tally and recalibrate as they are:
//   position p of the rewritten read = cycle p: base lo + p of the aligned window, or hi - 1 - p and
//   complemented (anything but ACGT -> N) on the reverse strand; the rest of the row is N with quality 0;
//   quality 0 (below every minscore >= 1) for skipped bases and N bases, which the BAM tally leaves out
//   of BOTH tables while the FASTQ tally would count an N in the cycle table; corrected base = base ^ 1
//   where the host flagged an error; second = read 2.
// The previous base in read direction is then simply the previous byte, for either strand.  Bases
// outside the window that the host did NOT mark as skipped are tallied at cycle 0 / dinucleotide 0 as
// the reference does (kbbq/gatk/bqsr.py:24,43: the "full" arrays start as zeros); they are rare
// (find_read_errors skips every soft clip), so they take global atomics here.
struct BamCanonArgs {
    const uint8_t *seq, *qual, *err, *skip;
    const uint16_t *rg;
    const uint8_t *flags;
    const uint16_t *aln_start, *aln_end;
    long long N;
    int L, R, minscore, nq;   // nq: qualities the apply's delta tables hold (the build: 43)
    bool build;               // false: apply (whole read, qualities untouched, no corrected array)
    uint8_t *cseq, *cqual, *ccorr, *csecond;
    unsigned long long *pos_errs, *pos_total, *din_errs, *din_total;
    int *status;
};

__device__ __forceinline__ uint8_t bam_complement(uint8_t b) {
    return b == 'A' ? 'T' : b == 'T' ? 'A' : b == 'G' ? 'C' : b == 'C' ? 'G' : 'N';
}

// ---- the rewrite pass -------------------------------------------------------------------------------
// One thread produces one ALIGNED 32-bit word of every output array, i.e. four
// positions, from four source bytes fetched as two aligned words and a funnel shift (the source
// window starts at any byte, and runs backwards on the reverse strand: byte-reversed with one PRMT).
// Masks are byte-parallel as in build.cuh.  Words that reach outside the aligned window or the read
// (at most three per read) take the byte-wise path, which also does the reference's cycle-0 tally of
// unskipped bases outside the window.  One base per thread with byte accesses took 6.4 ms for
// 10 M x 150 bp (182 instructions per base); this form is bound by memory instead.
constexpr int BAM_WARPS = 8;  // warps per block of the canonical-form kernels

__device__ __forceinline__ uint32_t load4_any(const uint8_t *__restrict__ p) {
    const uintptr_t a = (uintptr_t)p;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(a & 3) * 8u;
    const uint32_t lo = w[0], hi = sh ? w[1] : 0u;  // nothing is read past the word that holds the last byte
    return __funnelshift_r(lo, hi, sh);
}
// 0xFF in every byte of x that is not zero
__device__ __forceinline__ uint32_t nonzero_mask(uint32_t x) {
    uint32_t m = (((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & H4, r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(m), "r"(0u), "r"(0xBA98u));  // sign of byte b -> byte b
    return r;
}
// complement.get(x, 'N') on four bases (kbbq/gatk/bqsr.py:40): A <-> T, C <-> G, anything else N
__device__ __forceinline__ uint32_t complement4(uint32_t w) {
    const uint32_t code3 = (w >> 1) & 0x07070707u;          // A 0, C 1, T 2, G 3, N 7
    const uint32_t y = code3 | (code3 >> 4);
    const uint32_t sel = __byte_perm(y, 0u, 0x4420u) & 0x7777u;
    const uint32_t self = __byte_perm(0x47544341u /* A C T G */, 0x4E000000u /* . . . N */, sel);
    const uint32_t comp = __byte_perm(0x43414754u /* T G A C */, 0x4E4E4E4Eu, sel);
    const uint32_t bad = nonzero_mask(self ^ w);              // a byte that is not the base its code stands for
    return (comp & ~bad) | (0x4E4E4E4Eu & bad);
}
// 0xFF in every byte of w that is not one of A, C, G, T, N
__device__ __forceinline__ uint32_t nonacgtn_mask(uint32_t w) {
    const uint32_t code3 = (w >> 1) & 0x07070707u;
    const uint32_t y = code3 | (code3 >> 4);
    const uint32_t sel = __byte_perm(y, 0u, 0x4420u) & 0x7777u;
    return nonzero_mask(__byte_perm(0x47544341u /* A C T G */, 0x4E000000u /* . . . N */, sel) ^ w);
}

// One thread per aligned output word (`wmax` word slots per read, r0 = first read of this launch), so
// that nothing waits for anything: a warp-per-read loop was bound by its chain of round trips.
__global__ void __launch_bounds__(BAM_WARPS * 32) bam_canon_kernel(BamCanonArgs a, long long r0, unsigned int wmax) {
    const unsigned int t = blockIdx.x * (unsigned int)(BAM_WARPS * 32) + threadIdx.x;
    const unsigned int rl = t / wmax;
    const int k = (int)(t - rl * wmax);
    const long long r = r0 + rl;
    if (r >= a.N) return;
    const uint8_t *__restrict__ seq = a.seq, *__restrict__ qual = a.qual, *__restrict__ errp = a.err,
                  *__restrict__ skipp = a.skip;
    const int fl = a.flags ? a.flags[r] : 0;
    const bool reverse = fl & BAM_FLAG_REVERSE;
    int lo = 0, hi = a.L;
    if (a.build) {
        lo = a.aln_start ? a.aln_start[r] : 0;
        hi = a.aln_end ? a.aln_end[r] : a.L;
        bam_clamp_window(a.L, &lo, &hi);
    }
    const int alen = hi - lo;
    const long long row = r * a.L;
    // output words are aligned in memory: word k holds positions 4 k - ao .. 4 k - ao + 3 (the three
    // canonical arrays share their alignment: carve_bam_workspace)
    const int ao = (int)((uintptr_t)(a.cseq + row) & 3);
    if (k == 0) a.csecond[r] = (uint8_t)(fl & BAM_FLAG_READ2);
    if (k >= ((ao + a.L + 3) >> 2)) return;
    const int p0 = 4 * k - ao;
    // four positions inside the window: word path -- unless a forward-strand base of the word, or the one before it,
    // lies outside ACGTN: the byte-wise path writes those as N and applies the reference's rule to them
    if (p0 >= 0 && p0 + 3 < alen &&
        (reverse || (!nonacgtn_mask(load4_any(seq + row + lo + p0)) && (p0 == 0 || bam_code(seq[row + lo + p0 - 1]) != 5)))) {
        const long long s = row + (reverse ? hi - 4 - p0 : lo + p0);
        uint32_t ws = load4_any(seq + s), wq = load4_any(qual + s), we = 0u, wk = 0u;
        if (a.build) {
            we = load4_any(errp + s);
            if (skipp) wk = load4_any(skipp + s);
        }
        if (reverse) {
            ws = __byte_perm(ws, 0u, 0x0123u);
            wq = __byte_perm(wq, 0u, 0x0123u);
            we = __byte_perm(we, 0u, 0x0123u);
            wk = __byte_perm(wk, 0u, 0x0123u);
        }
        const uint32_t b4 = reverse ? complement4(ws) : ws;
        uint32_t q4 = wq;
        if (a.build) {
            const uint32_t is_n = ~nonzero_mask(ws ^ 0x4E4E4E4Eu);      // the ORIGINAL base is N (:96)
            q4 &= ~(is_n | nonzero_mask(wk));
            *reinterpret_cast<uint32_t *>(a.ccorr + row + p0) = b4 ^ (nonzero_mask(we) & ONE4);
        }
        *reinterpret_cast<uint32_t *>(a.cseq + row + p0) = b4;
        *reinterpret_cast<uint32_t *>(a.cqual + row + p0) = q4;
        return;
    }
    for (int j = 0; j < 4; ++j) {  // a word at an edge of the window or of the read: byte by byte
        const int p = p0 + j;
        if (p < 0 || p >= a.L) continue;
        // every position reads exactly one source base: inside the window the one that lands here,
        // outside it one clipped base ([0, lo) then [hi, L))
        const bool inside = p < alen;
        const int kk = p - alen;
        const long long i = row + (inside ? (reverse ? hi - 1 - p : lo + p) : (kk < lo ? kk : hi + (kk - lo)));
        const uint8_t s = seq[i];
        const unsigned int qq = qual[i];
        const bool e = a.build && errp[i] != 0;
        const bool sk = a.build && skipp && skipp[i] != 0;
        uint8_t b = 'N', q = 0, c = 'N';
        if (inside) {
            // a forward-strand base outside ACGTN: N in the canonical read, which leaves out its dinucleotides as the
            // reference does where it does not raise; where it raises (bam_dinuc), the flag is set here
            b = reverse ? bam_complement(s) : bam_code(s) == 5 ? (uint8_t)'N' : s;
            if (!reverse && p > 0 && (a.build ? !sk : true)) {
                const int cc = bam_code(s), pc = bam_code(seq[i - 1]);
                const unsigned int g = a.rg ? a.rg[r] : 0;
                if ((int)qq >= a.minscore && (int)qq < a.nq && g < (unsigned int)a.R && cc != 4 && pc != 4 &&
                    (cc == 5 || pc == 5))
                    atomicOr(a.status, KBBQ_FLAG_BAD_BASE);
            }
            q = (a.build && (sk || s == 'N')) ? (uint8_t)0 : (uint8_t)qq;
            c = e ? (uint8_t)(b ^ 1) : b;
        } else if (a.build && !sk && (int)qq >= a.minscore && s != 'N') {
            const unsigned int g = a.rg ? a.rg[r] : 0;
            if (qq > NQ - 1) atomicOr(a.status, KBBQ_FLAG_QUAL_RANGE);
            else if (g >= (unsigned int)a.R) atomicOr(a.status, KBBQ_FLAG_RG_RANGE);
            else {
                const size_t po = ((size_t)g * NQ + qq) * (2 * a.L), d = ((size_t)g * NQ + qq) * 16;
                atomicAdd(a.pos_total + po, 1ull);
                atomicAdd(a.din_total + d, 1ull);
                if (e) { atomicAdd(a.pos_errs + po, 1ull); atomicAdd(a.din_errs + d, 1ull); }
            }
        }
        a.cseq[row + p] = b;
        a.cqual[row + p] = q;
        if (a.build) a.ccorr[row + p] = c;
    }
}

// out[r][i] = canonical out[r][p(i)]: flips the reverse-strand reads back (apply only); aligned output words
__global__ void __launch_bounds__(BAM_WARPS * 32) bam_uncanon_kernel(const uint8_t *__restrict__ cout, const uint8_t *flags,
                                                                    long long N, int L, uint8_t *__restrict__ out,
                                                                    long long r0, unsigned int wmax) {
    const unsigned int t = blockIdx.x * (unsigned int)(BAM_WARPS * 32) + threadIdx.x;
    const unsigned int rl = t / wmax;
    const int k = (int)(t - rl * wmax);
    const long long r = r0 + rl;
    if (r >= N) return;
    const bool reverse = flags && (flags[r] & BAM_FLAG_REVERSE);
    const long long row = r * L;
    const int ao = (int)((uintptr_t)(out + row) & 3);
    if (k >= ((ao + L + 3) >> 2)) return;
    const int i0 = 4 * k - ao;
    if (i0 >= 0 && i0 + 3 < L) {
        uint32_t w = load4_any(cout + row + (reverse ? L - 4 - i0 : i0));
        if (reverse) w = __byte_perm(w, 0u, 0x0123u);
        *reinterpret_cast<uint32_t *>(out + row + i0) = w;
        return;
    }
    for (int j = 0; j < 4; ++j) {
        const int i = i0 + j;
        if (i >= 0 && i < L) out[row + i] = cout[row + (reverse ? L - 1 - i : i)];
    }
}

}  // namespace kbbq
