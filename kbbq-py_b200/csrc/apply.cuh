// apply.cuh -- K2: recalibration apply kernel.
//
// Replaces compare_reads.recalibrate_fastq (kbbq/compare_reads.py:320-328) over a packed batch:
//   out = q < minscore ? q : meanq[rg] + rgdq[rg] + qdq[rg,q] + dindq[rg,q,dinuc] + posdq[rg,q,cycle]
// Every term is an integer, so the five-term sum is folded (model.cuh: fold_kernel) into two small
// tables per read group:
//   fold_cyc[q][cycle] = meanq + rgdq + qdq[q] + posdq[q][cycle] + dindq[q][last]   (last = the column an
//                        invalid dinucleotide, index -1, gathers)
//   fold_din[q][dinuc] = dindq[q][dinuc] - dindq[q][last]
// so that an invalid dinucleotide simply reads a zero row, and the kernel does two shared-memory
// gathers per base instead of five global ones.
//
// Roofline: HBM, 3 B/base (seq + qual in, new qual out).  Same thread mapping, TMA staging ring,
// byte-parallel row index and IDP.4A address arithmetic as the build kernel (build.cuh): the cycle
// table is gathered at consecutive banks by consecutive lanes and the dinuc table is replicated per
// lane, so both gathers are bank-conflict free.
#pragma once
#include "build.cuh"
#include "common.cuh"
#include "stage.cuh"

namespace kbbq {

struct ApplyArgs {
    const uint8_t *seq, *qual;
    uint8_t *out;
    long long total_bytes;  // N * L
    Geom g;
    TableCfg t;
    StageLayout sl;
    int R, nq;
    int nsub, segmode;  // see BuildArgs
    const entry_t *entries;
    const unsigned int *seg;
    const unsigned int *uni;  // see BuildArgs
    const short *fold_cyc;  // [R][43][2L]
    const short *fold_din;  // [R][43][16]   natural dinuc order (code = (base >> 1) & 3)
    int *status;
};

static_assert((offsetof(ApplyArgs, t) + offsetof(TableCfg, ohe)) % 16 == 0,
              "ApplyArgs: TableCfg::ohe has to be 16-byte aligned in the kernel parameters (build.cuh); pad Geom");

// bytes of shared memory the apply tables take
__host__ __device__ inline int apply_table_bytes(const TableCfg &t) { return t.table_bytes; }

// Consumer side of the apply kernel; UNI as in build_consume (build.cuh).  VALIDATE: flag a base outside ACGTN as the
// build does (off when the caller vouches for the bases: KBBQ_APPLY_BASES_CHECKED, kbbq_b200.cu).
template <int KPS, bool UNI, bool VALIDATE>
__device__ __forceinline__ void apply_consume(const ApplyArgs &a, unsigned char *smem_raw, uint32_t lo, uint32_t hi,
                                              uint32_t uni_flo, uint32_t uni_fhi) {
    const Geom &g = a.g;
    const TableCfg &t = a.t;
    const StageLayout &sl = a.sl;
    const int nconsumers = g.threads;
    const uint32_t bar0 = pin(smem_u32(smem_raw + sl.bar_off));
    const ThreadMap m = make_thread_map(g, t, UNI, true);
    const int lane = threadIdx.x & 31;
    const uint32_t pos_base = smem_addr(smem_raw + t.pos_off);
    const uint32_t din_base = pin(smem_addr(smem_raw + t.din_off) + (lane & (t.drep - 1)) * 4);
    uint32_t aeff[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) aeff[b] = pos_base + m.cell[b];
    uint32_t cur_flag = 1;
    const uint32_t selv = pin(m.selv), seln = pin(m.seln);
    const uint32_t rowsel = m.row >= 0 ? (uint32_t)m.row : 0u;
    const uint32_t lanemask = pin(m.row >= 0 ? 0xFFu : 0u);
    const uint32_t rowmask = pin(m.rowmask);
    const bool live = m.row >= 0;
    const uint32_t kgrp = g.ng * g.gbytes;
    // how this thread's word is written back: whole (0), one aligned half (1, the usual partial
    // word: reads of even length start 2-byte aligned) or byte by byte (2)
    const bool half_lo = m.rowmask == 0x0000FFFFu, half_hi = m.rowmask == 0xFFFF0000u;
    const bool st32 = m.rowmask == 0xFFFFFFFFu, st16 = half_lo || half_hi, st8 = !st32 && !st16 && m.rowmask != 0u;
    const uint32_t wshift = pin(half_hi ? 16u : 0u);
    unsigned long long outp = (unsigned long long)(a.out + m.toff + (half_hi ? 2 : 0));
    asm volatile("" : "+l"(outp));
    const uint32_t data0 = pin(smem_u32(smem_raw + sl.data_off) + m.toff + (UNI ? m.grp * g.gbytes : 0));
    const uint32_t hdr0 = pin(smem_u32(smem_raw + sl.hdr_off) + m.grp * 16);
    const uint32_t stage_bytes = pin(sl.narr * sl.abytes), abytes = pin(sl.abytes), hdr_stride = sl.ngs * 16, krec = g.ng * 16;
    const uint32_t nstages = pin(sl.stages), ngs = pin(sl.ngs);
    const uint32_t revoff = t.revoff, addq = t.addq, gbytes = g.gbytes;
    const uint32_t addnq = (uint32_t)(128 - a.nq) * ONE4;  // q + this has bit 7 set iff q >= nq (q < 128)
    const uint32_t one = pin(1u);                          // see add_fma (build.cuh)
    const uint32_t lut_lo = pin(0x43014101u), lut_hi = pin(0x474E0154u);  // base validation LUT (build.cuh)
    uint32_t stage = 0, phase = 0;
    uint32_t qgood = 0xFFFFFFFFu, bbad = 0;

    int cur_rg = -1, cur_sub = -1;
    int hs0 = 0, hs1 = 1;   // half of the cycle axis each table slot holds (build.cuh)
    if (UNI && !a.segmode) {
        hs0 = (int)((uni_flo & 0xFFu) >> 1);
        hs1 = (int)(((uni_flo >> 8) & 0xFFu) >> 1);
    }
    for (int sub = 0; sub < a.nsub; ++sub) {
        uint32_t s_lo = a.seg[sub], s_hi = a.seg[sub + 1];
        if (s_hi <= lo) continue;
        if (s_lo >= hi) break;
        if (s_lo < lo) s_lo = lo;
        if (s_hi > hi) s_hi = hi;
        if (s_lo >= s_hi) continue;
        const int rg = a.segmode ? sub >> 1 : sub;

        // stage this read group's folded tables; row 0 = "leave the quality alone": the dinuc table holds 0
        // there (invalid dinucs of any quality land on it), the cycle tables hold minscore - 1, the only
        // quality that reaches row 0 with its byte selected.  In a span of a segmented batch both slots hold
        // the span's half of the cycle axis, so the tables are staged again whenever the span changes.
        if (rg != cur_rg || (a.segmode && sub != cur_sub)) {
            cur_rg = rg;
            cur_sub = sub;
            if (a.segmode) hs0 = hs1 = sub & 1;
            consumer_sync(nconsumers);
            for (int i = threadIdx.x; i < apply_table_bytes(t) / 4; i += nconsumers)
                reinterpret_cast<int *>(smem_raw)[i] = i * 4 < t.din_off && (i * 4) % t.revoff < t.rs ? g.minscore - 1 : 0;
            consumer_sync(nconsumers);
            const int L = g.L, L2 = 2 * g.L;
            const short *fc = a.fold_cyc + (size_t)rg * NQ * L2;
            for (int i = threadIdx.x; i < 2 * (t.nrows - 1) * L; i += nconsumers) {
                const int slot = i >= (t.nrows - 1) * L, j = i - slot * (t.nrows - 1) * L;
                const int r = j / L + 1, c = j - (r - 1) * L;
                const int half = slot ? hs1 : hs0;
                int *p = reinterpret_cast<int *>(smem_raw + t.pos_off + slot * t.revoff + r * t.rs) + ((c & 3) * t.sj + (c >> 2));
                *p = fc[(size_t)(r + g.minscore - 1) * L2 + (half ? L2 - 1 - c : c)];
            }
            const short *fd = a.fold_din + (size_t)rg * NQ * DIN_SLOTS;
            for (int i = threadIdx.x; i < (t.nrows - 1) * DIN_SLOTS * t.drep; i += nconsumers) {
                const int cell = i / t.drep, r = cell / DIN_SLOTS + 1, s = cell & (DIN_SLOTS - 1);
                int *p = reinterpret_cast<int *>(smem_raw + t.din_off + r * t.dq + s * (t.drep * 4)) + (i & (t.drep - 1));
                *p = fd[(r + g.minscore - 1) * DIN_SLOTS + s];
            }
            consumer_sync(nconsumers);
        }

        for (uint32_t first = s_lo; first < s_hi; first += ngs) {
            mbar_wait(bar0 + stage * 8, phase);
            const uint32_t shdr = pin(hdr0 + stage * hdr_stride);
            uint32_t sdata = data0 + stage * stage_bytes;
            uint32_t nlive = sl.ngs;
            if (UNI) {
                sdata += (uint32_t)((unsigned long long)first * g.gbytes) & 15u;
                nlive = s_hi - first;
            }
            sdata = pin(sdata);
            // one (row, word) of one group: four qualities of one read
            auto apply_word = [&](const uint32_t wa, const uint32_t hgrp) {
                uint32_t sw, qw, pb;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(sw) : "r"(wa));
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(qw) : "r"(wa + abytes));
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(pb) : "r"(wa - 1));

                const uint32_t nu = ~add_fma(qw, one, addnq);  // bit 7 clear <=> q >= nq: IndexError in the reference
                const uint32_t w5 = add_fma(qw, one, addq);
                qgood &= nu & ~qw;
                const uint32_t vraw = w5 & nu & ~qw;
                const uint32_t vm8 = prmt(vraw, 0u, selv);  // 0xFF for owned bytes with minscore - 1 <= q < nq
                const uint32_t qrow4 = w5 & vm8 & 0x3F3F3F3Fu;
                const uint32_t pw = prmt(pb, sw, 0x6540u);
                const uint32_t d4 = (pw & 0x06060606u) * 4u + (sw & 0x06060606u);
                const uint32_t nm8 = prmt((sw | pw) * 16u, 0xFFFFFFFFu, seln);
                const uint32_t qd = qrow4 & ~nm8;
                const uint32_t x01 = prmt(d4, qd, 0x5140u), x23 = prmt(d4, qd, 0x7362u);  // see build.cuh
                if (VALIDATE) {
                    // base validation as in the build: rebuild each byte from its 3-bit code, any difference = a base
                    // outside ACGTN (foreign bytes are masked off by rowmask at the end)
                    const uint32_t code3 = sw & 0x07070707u;
                    const uint32_t vsel = __dp2a_hi(t.val16[1], code3, __dp2a_lo(t.val16[0], code3, 0u));
                    bbad |= prmt(lut_lo, lut_hi, vsel) ^ sw;
                }

                uint32_t v[4];
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const uint32_t pa = (b & 2) ? __dp2a_hi(t.cyc16[b & 1], qrow4, aeff[b]) : __dp2a_lo(t.cyc16[b & 1], qrow4, aeff[b]);
                    const uint32_t xb = (b & 2) ? x23 : x01;
                    const uint32_t da = (b & 1) ? __dp2a_hi(t.din16, xb, din_base) : __dp2a_lo(t.din16, xb, din_base);
                    uint32_t x, y;
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(x) : "r"(pa));
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(y) : "r"(da));
                    v[b] = x + y;
                }
                // low byte of every sum; qualities that do not pass vm8 stay as they are.  q == minscore - 1
                // passes vm8 with row 0, whose cycle table holds minscore - 1 and whose dinuc table holds 0.
                const uint32_t sum4 = __byte_perm(__byte_perm(v[0], v[1], 0x0040), __byte_perm(v[2], v[3], 0x0040), 0x5410);
                const uint32_t res = (sum4 & vm8) | (qw & ~vm8);
                // group base + this thread's offset inside the group (64-bit multiply-add, one instruction)
                const unsigned long long dst = outp + (unsigned long long)hgrp * gbytes;
                if (UNI) {
                    // uniform walk: a live thread owns its whole word (make_thread_map) -- one predicated store
                    if (st32) asm volatile("st.global.u32 [%0], %1;" ::"l"(dst), "r"(res) : "memory");
                    return;
                }
                // work-list walk: a word that straddles two rows has two owners -- whole word, one aligned half, or bytes
                if (st32) asm volatile("st.global.u32 [%0], %1;" ::"l"(dst), "r"(res) : "memory");
                if (st16) asm volatile("st.global.u16 [%0], %1;" ::"l"(dst), "h"((unsigned short)(res >> wshift)) : "memory");
                if (st8) {
#pragma unroll
                    for (int b = 0; b < 4; ++b)
                        if ((rowmask >> (8 * b)) & 1u)
                            asm volatile("st.global.u8 [%0], %1;" ::"l"(dst + b), "r"(res >> (8 * b)) : "memory");
                }
            };
            if (UNI && nlive >= sl.ngs) {
                // a full stage of a uniform batch, the usual case: no per-word predicates (padding lanes own no byte
                // and store nothing)
#pragma unroll
                for (int k = 0; k < KPS; ++k) apply_word(sdata + k * kgrp, first + m.grp + k * g.ng);
            } else {
#pragma unroll
                for (int k = 0; k < KPS; ++k) {
                    uint32_t soff, hgrp;
                    if (UNI) {
                        if (!live || (uint32_t)(m.grp + k * g.ng) >= nlive) continue;
                        soff = k * kgrp;
                        hgrp = first + m.grp + k * g.ng;
                    } else {
                        uint32_t flo, fhi;
                        if (g.contig) {   // the identity list, read where it lies; past the span: no rows
                            const uint32_t e = first + (uint32_t)m.grp + (uint32_t)(k * g.ng);
                            const uint4 rec = e < s_hi ? __ldg(a.entries + e) : make_uint4(0u, 0u, 0u, 0u);
                            soff = rec.x; hgrp = rec.y; flo = rec.z; fhi = rec.w;
                        } else {
                            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                                         : "=r"(soff), "=r"(hgrp), "=r"(flo), "=r"(fhi)
                                         : "r"(shdr + k * krec));
                        }
                        // cycle-table addresses are kept for the last row flag seen (see build.cuh)
                        const uint32_t flag = prmt(flo, fhi, rowsel) & lanemask;
                        if (flag != cur_flag) {
                            if (!flag) continue;
                            const uint32_t delta = ((flag >> 1) - (cur_flag >> 1)) * revoff;
#pragma unroll
                            for (int b = 0; b < 4; ++b) aeff[b] += delta;
                            cur_flag = flag;
                        }
                    }
                    apply_word(sdata + soff, hgrp);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar0 + (nstages + stage) * 8);
            if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
    }
    if (~qgood & rowmask & H4) atomicOr(a.status, KBBQ_FLAG_QUAL_RANGE);
    if (VALIDATE && (bbad & rowmask)) atomicOr(a.status, KBBQ_FLAG_BAD_BASE);
}


template <int KPS, bool VALIDATE>
__global__ void __launch_bounds__(MAX_THREADS, 1) apply_smem_kernel(const __grid_constant__ ApplyArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const Geom &g = a.g;
    const StageLayout &sl = a.sl;
    const int nconsumers = g.threads;

    const unsigned long long E = a.seg[a.nsub];
    const uint32_t lo = (uint32_t)(E * blockIdx.x / gridDim.x), hi = (uint32_t)(E * (blockIdx.x + 1) / gridDim.x);
    const bool contig = a.R == 1 || a.segmode;
    const bool uniform = contig && a.uni[0] == 0u;

    const uint32_t bar0 = smem_u32(smem_raw + sl.bar_off);
    if (threadIdx.x == 0) {
        for (int s = 0; s < sl.stages; ++s) {
            mbar_init(bar0 + s * 8, 1);
            mbar_init(bar0 + (sl.stages + s) * 8, nconsumers / 32);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if ((int)threadIdx.x >= nconsumers) {  // ---- producer warp ----
        ProducerArgs p;
        p.arr[0] = a.seq; p.arr[1] = a.qual; p.arr[2] = nullptr;
        p.entries = a.entries; p.seg = a.seg; p.nsub = a.nsub; p.contig = contig; p.lo = lo; p.hi = hi;
        p.gbytes = g.gbytes; p.ng = sl.ngs; p.total_bytes = a.total_bytes;
        p.pw = ((int)threadIdx.x - nconsumers) >> 5; p.nprod = g.nprod;
        p.uniform = uniform;
        producer_loop(p, sl, smem_raw);
        return;
    }

    if (uniform) apply_consume<KPS, true, VALIDATE>(a, smem_raw, lo, hi, a.uni[1], a.uni[2]);
    else apply_consume<KPS, false, VALIDATE>(a, smem_raw, lo, hi, 0u, 0u);
}

// Generic path (any L): one thread per base, folded tables gathered from global memory (L1/L2).
struct ApplyGenericArgs {
    const uint8_t *seq, *qual;
    const uint16_t *rg;
    const uint8_t *second;
    uint8_t *out;
    long long N;
    int L, R, minscore, nq;
    const short *fold_cyc, *fold_din;
    int *status;
    bool validate;   // see apply_consume
};

__global__ void apply_generic_kernel(ApplyGenericArgs a) {
    const long long total = a.N * a.L;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / a.L;
        const int c = (int)(i - r * a.L);
        const unsigned int q = a.qual[i];
        const uint8_t s = a.seq[i];
        if (a.validate && base_code_ref(s) == 5) atomicOr(a.status, KBBQ_FLAG_BAD_BASE);   // the build's rule: any byte outside ACGTN
        if ((int)q < a.minscore) { a.out[i] = (uint8_t)q; continue; }
        if ((int)q >= a.nq) { atomicOr(a.status, KBBQ_FLAG_QUAL_RANGE); a.out[i] = (uint8_t)q; continue; }
        const unsigned int g = a.rg ? a.rg[r] : 0;
        if (g >= (unsigned int)a.R) { atomicOr(a.status, KBBQ_FLAG_RG_RANGE); a.out[i] = (uint8_t)q; continue; }
        const int c2 = (a.second && a.second[r]) ? 2 * a.L - 1 - c : c;
        const size_t gq = (size_t)g * NQ + q;
        int v = a.fold_cyc[gq * (2 * a.L) + c2];
        if (c > 0) {
            // as the shared-memory kernel: a byte with bit 3 set (of ACGTN only N) has no dinucleotide term
            const uint8_t ps = a.seq[i - 1];
            if (!((s | ps) & 8u)) v += a.fold_din[gq * DIN_SLOTS + ((((ps >> 1) & 3) << 2) | ((s >> 1) & 3))];
        }
        a.out[i] = (uint8_t)v;
    }
}

}  // namespace kbbq
