// kbbq_b200.cu -- the C ABI of libkbbq_b200.so (see include/kbbq_b200.h).
// One translation unit: kernels live in the .cuh files, this file validates arguments, picks the
// kernel configuration and enqueues.  Compiled for sm_100a only.
#include <algorithm>
#include <mutex>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "apply.cuh"
#include "bam.cuh"
#include "build.cuh"
#include "calib.cuh"
#include "common.cuh"
#include "model.cuh"
#include "prepare.cuh"
#include "segment.cuh"
#include "synth.cuh"

namespace kbbq {

std::atomic<long long> g_launches{0};
char g_last_cuda_error[256] = "";

// per-device __constant__ images of the model tables; a failed upload is retried by the next call
static std::mutex g_const_mu;
static bool g_const_done[64];

static int upload_constants(int device) {
    std::lock_guard<std::mutex> lock(g_const_mu);
    if (device >= 0 && device < 64 && g_const_done[device]) return KBBQ_OK;
    KBBQ_CUDA(cudaMemcpyToSymbol(c_lnp, KBBQ_LN_P, sizeof(double) * NQ));
    KBBQ_CUDA(cudaMemcpyToSymbol(c_ln1mp, KBBQ_LN_1MP, sizeof(double) * NQ));
    KBBQ_CUDA(cudaMemcpyToSymbol(c_prior, KBBQ_PRIOR, sizeof(double) * NQ));
    KBBQ_CUDA(cudaMemcpyToSymbol(c_p, KBBQ_P, sizeof(double) * NQ));
    KBBQ_CUDA(cudaMemcpyToSymbol(c_bound_hi, KBBQ_BOUND_HI, sizeof(double) * NQ));
    KBBQ_CUDA(cudaMemcpyToSymbol(c_bound_lo, KBBQ_BOUND_LO, sizeof(double) * NQ));
    if (device >= 0 && device < 64) g_const_done[device] = true;
    return KBBQ_OK;
}

static int current_device_info(int *device, int *sms, int *max_smem) {
    KBBQ_CUDA(cudaGetDevice(device));
    static std::atomic<int> s_sms[64], s_smem[64];   // several host threads (one per device) come through here
    if (*device < 64 && s_sms[*device].load()) {
        *sms = s_sms[*device].load();
        *max_smem = s_smem[*device].load();
        return KBBQ_OK;
    }
    KBBQ_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, *device));
    KBBQ_CUDA(cudaDeviceGetAttribute(max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, *device));
    if (*sms <= 0) *sms = KBBQ_SM_COUNT_FALLBACK;
    if (*device < 64) { s_smem[*device].store(*max_smem); s_sms[*device].store(*sms); }
    return KBBQ_OK;
}

static bool misaligned(const void *p, size_t a) { return ((uintptr_t)p & (a - 1)) != 0; }

// Shared-memory plan of a kernel: table geometry + staging ring.  Barrier traffic is paid per stage,
// so with 32 dinuc replicas (conflict free; 16 if that does not fit) take as many groups per
// thread-group and stage (kps <= 4, at most 32 groups per stage: one per producer lane) as still
// leave a ring of 3 stages; failing that, whatever ring of at least 2 stages fits.
// Measured on 10M x 150 bp: build kps 1 / drep 32 1.51 ms, kps 2 / drep 32 1.24 ms, kps 4 / drep 16 1.30 ms.
static bool plan_smem(const Geom &g, int narr, int max_smem, TableCfg *tc, StageLayout *sl) {
    const char *e = getenv("KBBQ_KPS");  // tuning / test hooks
    const int kmax = e ? std::max(1, std::min(8, atoi(e))) : 4;
    const char *d = getenv("KBBQ_DREP");
    const int dmax = d ? atoi(d) : 32;
    const char *w = getenv("KBBQ_MIN_STAGES");
    const int want = w ? std::max(2, std::min(8, atoi(w))) : 2;
    const char *ms = getenv("KBBQ_MAX_STAGES");
    const int smax = ms ? std::max(want, std::min(MAX_STAGES, atoi(ms))) : MAX_STAGES;
    // Measured (tools/kps_sweep.sh and the shape runs in DESIGN.md): more groups per barrier round win
    // -- four groups x two stages beats two x four by 5 % in the 150 bp build -- as long as the stages
    // behind the one being consumed hold the bandwidth-delay product of an SM (~30 B/clk x ~1400 clk);
    // below that a deeper ring of smaller stages is faster (250 bp).  Both matter more than
    // conflict-free dinuc replicas.
    // (Round 2: the build kernel spends fewer instructions per stage than it did when the 40 KB rule was found, and a
    // deeper ring of smaller stages now wins there as long as a thread-group still takes two groups per barrier
    // round -- 150 bp: kps 2 x 4 stages 0.898 ms, kps 4 x 2 stages 0.912 ms; 76 bp: kps 3 x 3 0.866 ms, kps 4 x 2
    // 0.945 ms; but 250 bp: kps 1 x 7 1.339 ms, kps 2 x 3 0.989 ms -- while the apply kernel still prefers four
    // groups per round: 0.809 against 0.889 ms with two.)  So: rules in order of preference, each a minimum of bytes
    // in flight behind the stage being consumed, a minimum of groups per round and a number of dinuc replicas; 0 bytes
    // = whatever fits.
    struct Rule { int in_flight, kmin, drep; };
    // Conflict-free dinuc replicas (32) before the ring rules (16 replicas cost 10 % at 150 bp), but two groups per
    // round with 16 replicas before one group per round with 32 (250 bp rows in read order, apply: 4.79 against 5.18 ms)
    const Rule build_rules[] = {{60000, 2, 32}, {40000, 2, 32}, {0, 2, 32}, {40000, 2, 16}, {0, 2, 16},
                                {40000, 1, 32}, {0, 1, 32}, {40000, 1, 16}, {0, 1, 16}, {0, 1, 8}};
    const Rule apply_rules[] = {{40000, 2, 32}, {0, 2, 32}, {40000, 2, 16}, {0, 2, 16},
                                {40000, 1, 32}, {0, 1, 32}, {40000, 1, 16}, {0, 1, 16}, {0, 1, 8}};
    const Rule *rules = narr == 3 ? build_rules : apply_rules;
    const int nrules = narr == 3 ? 10 : 9;
    const char *f = getenv("KBBQ_IN_FLIGHT");   // tuning hook: replaces the first rule's bytes
    for (int r = 0; r < nrules; ++r) {
        const int drep = rules[r].drep;
        if (drep > dmax || (drep == 8 && dmax > 8)) continue;   // 8 replicas only on request
        const int in_flight_min = (r == 0 && f) ? std::max(0, atoi(f)) : rules[r].in_flight;
        for (int k = kmax; k >= rules[r].kmin; --k) {
            if (!g.contig && g.ng * k > 32) continue;  // gathered groups: one producer lane per group of a stage
            if (!make_table_cfg(g, k, drep, narr == 2, tc)) return false;   // narr 2: the apply kernel
            for (int s = smax; s >= want; --s) {
                // several producer warps take the iterations round-robin: a stage must always be
                // refilled by the same warp (its waits are only one phase deep), so the ring
                // depth has to be a multiple of their number
                if (s % g.nprod) continue;
                *sl = make_stage_layout(g, narr, s, k, tc->table_bytes);
                if (sl->total > max_smem) continue;
                if ((s - 1) * narr * sl->abytes < in_flight_min) break;  // deepest ring that fits is too shallow
                return true;
            }
        }
    }
    return false;
}

// Geometry + shared-memory plan; with several read groups the producer-warp count falls back from 8
// when a ring of that many stages does not fit.
static bool plan_kernel(int L, int R, int minscore, int narr, int max_smem, Geom *g, TableCfg *tc, StageLayout *sl,
                        bool segmode = false) {
    int first = 8;
    if (const char *e = getenv("KBBQ_NPROD")) first = std::max(1, std::min(8, atoi(e)));  // tuning hook
    const bool single = R == 1 || segmode;  // contiguous spans: the one-read-group geometry
    for (int nprod = (single ? 1 : first); nprod >= 1; nprod >>= 1) {
        if (!make_geom(L, minscore, single, nprod, g, segmode)) return false;
        if (g->row < 65536 && plan_smem(*g, narr, max_smem, tc, sl)) return true;
    }
    return false;
}

template <int KPS>
static int launch_build_kps(const BuildArgs &a, int grid, size_t smem, cudaStream_t st) {
    auto kern = build_smem_kernel<KPS, true>;
    KBBQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, a.g.threads + 32 * a.g.nprod, smem, st>>>(a);  // + the producer warp(s)
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}
static int launch_build_smem(const BuildArgs &a, int grid, size_t smem, cudaStream_t st) {
    switch (a.sl.kps) {
    case 8: return launch_build_kps<8>(a, grid, smem, st);
    case 7: return launch_build_kps<7>(a, grid, smem, st);
    case 6: return launch_build_kps<6>(a, grid, smem, st);
    case 5: return launch_build_kps<5>(a, grid, smem, st);
    case 4: return launch_build_kps<4>(a, grid, smem, st);
    case 3: return launch_build_kps<3>(a, grid, smem, st);
    case 2: return launch_build_kps<2>(a, grid, smem, st);
    default: return launch_build_kps<1>(a, grid, smem, st);
    }
}

template <int KPS>
static int launch_apply_kps(const ApplyArgs &a, bool validate, int grid, size_t smem, cudaStream_t st) {
    auto kern = validate ? apply_smem_kernel<KPS, true> : apply_smem_kernel<KPS, false>;
    KBBQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, a.g.threads + 32 * a.g.nprod, smem, st>>>(a);  // + the producer warp(s)
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}
static int launch_apply_smem(const ApplyArgs &a, bool validate, int grid, size_t smem, cudaStream_t st) {
    switch (a.sl.kps) {
    case 8: return launch_apply_kps<8>(a, validate, grid, smem, st);
    case 7: return launch_apply_kps<7>(a, validate, grid, smem, st);
    case 6: return launch_apply_kps<6>(a, validate, grid, smem, st);
    case 5: return launch_apply_kps<5>(a, validate, grid, smem, st);
    case 4: return launch_apply_kps<4>(a, validate, grid, smem, st);
    case 3: return launch_apply_kps<3>(a, validate, grid, smem, st);
    case 2: return launch_apply_kps<2>(a, validate, grid, smem, st);
    default: return launch_apply_kps<1>(a, validate, grid, smem, st);
    }
}

}  // namespace kbbq

using namespace kbbq;

extern "C" {

int kbbq_abi_version(void) { return 1; }

const char *kbbq_strerror(int code) {
    switch (code) {
    case KBBQ_OK: return "ok";
    case KBBQ_E_ARG: return "bad argument";
    case KBBQ_E_CUDA: return "CUDA runtime error";
    case KBBQ_E_WORKSPACE: return "workspace too small";
    case KBBQ_E_DATA: return "input data error (see status flags)";
    case KBBQ_E_IO: return "FASTQ file could not be opened, read or written";
    case KBBQ_E_FORMAT: return "malformed FASTQ (4-line records expected)";
    case KBBQ_E_RAGGED: return "reads of unequal length";
    case KBBQ_E_NAME_FIELD: return "read name has no read-group field";
    case KBBQ_E_NAME_RG: return "read-group field does not start with RG";
    case KBBQ_E_NAME_MISMATCH: return "corrected read name does not start with the read name";
    case KBBQ_E_PEER: return "multi-GPU: peer access between the devices is not available";
    case KBBQ_E_UNSUPPORTED: return "not handled by this entry point (use the chunked driver)";
    default: return "unknown error";
    }
}

const char *kbbq_last_cuda_error(void) { return g_last_cuda_error; }

int64_t kbbq_pos_table_elems(int L, int R) { return (int64_t)R * NQ * 2 * L; }
int64_t kbbq_din_table_elems(int R) { return (int64_t)R * NQ * 16; }
int64_t kbbq_launch_count(void) { return g_launches.load(); }

int kbbq_plan_info(int L, int R, int minscore, int arrays, int max_smem, int *out) {
    const bool segmode = (arrays & KBBQ_PLAN_SEGMENTED) != 0;
    arrays &= ~KBBQ_PLAN_SEGMENTED;
    if (!out || L < 1 || R < 1 || (arrays != 2 && arrays != 3)) return KBBQ_E_ARG;
    Geom g;
    TableCfg tc;
    StageLayout sl;
    if (!plan_kernel(L, R, minscore, arrays, max_smem > 0 ? max_smem : 232448, &g, &tc, &sl, segmode))
        return KBBQ_E_ARG;  // the generic kernels would be used
    const int v[10] = {g.G, g.lanes, g.ng, g.threads, g.nprod, sl.kps, sl.stages, tc.drep, sl.total, tc.table_bytes};
    for (int i = 0; i < 10; ++i) out[i] = v[i];
    return KBBQ_OK;
}

int kbbq_workspace_bytes(int64_t N, int L, int R, size_t *bytes) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || !bytes) return KBBQ_E_ARG;
    *bytes = carve_workspace(nullptr, N, L, R).bytes;
    return KBBQ_OK;
}

// kbbq_build / kbbq_build_segmented.  seg_rows != NULL: a segmented batch of at most N rows (segment.cuh).
static int build_impl(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
                      const uint8_t *second, int64_t N, int L, int R, int minscore, int64_t *pos_errs,
                      int64_t *pos_total, int64_t *din_errs, int64_t *din_total, void *workspace,
                      size_t workspace_bytes, int *status, int path, void *stream, const unsigned int *seg_rows) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || minscore < 0 || minscore >= NQ) return KBBQ_E_ARG;
    if (!pos_errs || !pos_total || !din_errs || !din_total || !status) return KBBQ_E_ARG;
    if (N == 0) return KBBQ_OK;
    if (!seq || !qual || !corr) return KBBQ_E_ARG;
    const bool segmode = seg_rows != nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;

    Geom g;
    TableCfg tc;
    StageLayout sl;
    const bool smem_ok = path != 2 && !misaligned(seq, 16) && !misaligned(qual, 16) && !misaligned(corr, 16) &&
                         plan_kernel(L, R, minscore, 3, max_smem, &g, &tc, &sl, segmode) &&
                         (uint64_t)((N + g.G - 1) / g.G) < 0xFFFFFFFFull;
    if (!smem_ok) {
        if (path == 1 || segmode) return KBBQ_E_ARG;
        BuildGenericArgs a = {seq, qual, corr, rg, second, N, L, R, minscore,
                              (unsigned long long *)pos_errs, (unsigned long long *)pos_total,
                              (unsigned long long *)din_errs, (unsigned long long *)din_total, status};
        build_generic_kernel<<<sms * 8, 256, 0, st>>>(a);
        KBBQ_LAUNCHED();
        return KBBQ_OK;
    }
    Workspace w = carve_workspace(workspace, N, L, R);
    if (!workspace || workspace_bytes < w.bytes) return KBBQ_E_WORKSPACE;
    if (segmode) {
        seg_prepare_kernel<<<1, 256, 0, st>>>(seg_rows, 2 * R, g.G, (unsigned long long)N, w.seg, w.uni, status);
        KBBQ_LAUNCHED();
    } else {
        // One read group: a partial last group would be the only one with untallied rows and cost the
        // whole batch its header-free fast path; its few reads go through the generic kernel instead.
        const int64_t tail = (R == 1 && N > g.G) ? N % g.G : 0;
        if (tail) {
            const int64_t n0 = N - tail;
            BuildGenericArgs ga = {seq + n0 * L, qual + n0 * L, corr + n0 * L, rg ? rg + n0 : nullptr,
                                   second ? second + n0 : nullptr, tail, L, R, minscore,
                                   (unsigned long long *)pos_errs, (unsigned long long *)pos_total,
                                   (unsigned long long *)din_errs, (unsigned long long *)din_total, status};
            build_generic_kernel<<<1, 256, 0, st>>>(ga);
            KBBQ_LAUNCHED();
            N = n0;
        }
        rc = run_prepare(rg, second, N, g.G, R, w, status, sms, sl.ngs, g.gbytes, sl.slot, st);
        if (rc) return rc;
    }

    BuildArgs a;
    a.seq = seq; a.qual = qual; a.corr = corr; a.total_bytes = N * L; a.g = g; a.t = tc; a.R = R;
    a.nsub = segmode ? 2 * R : R; a.segmode = segmode ? 1 : 0;
    a.sl = sl;
    a.entries = w.entries; a.seg = w.seg; a.uni = w.uni;
    a.pos_errs = (unsigned long long *)pos_errs; a.pos_total = (unsigned long long *)pos_total;
    a.din_errs = (unsigned long long *)din_errs; a.din_total = (unsigned long long *)din_total;
    a.status = status;
    return launch_build_smem(a, sms, a.sl.total, st);
}

int kbbq_build(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
               const uint8_t *second, int64_t N, int L, int R, int minscore, int64_t *pos_errs,
               int64_t *pos_total, int64_t *din_errs, int64_t *din_total, void *workspace,
               size_t workspace_bytes, int *status, int path, void *stream) {
    return build_impl(seq, qual, corr, rg, second, N, L, R, minscore, pos_errs, pos_total, din_errs, din_total,
                      workspace, workspace_bytes, status, path, stream, nullptr);
}

int kbbq_build_segmented(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint32_t *seg,
                         int64_t rows_bound, int L, int R, int minscore, int64_t *pos_errs, int64_t *pos_total,
                         int64_t *din_errs, int64_t *din_total, void *workspace, size_t workspace_bytes, int *status,
                         void *stream) {
    if (!seg || rows_bound % SEG_ALIGN) return KBBQ_E_ARG;
    return build_impl(seq, qual, corr, nullptr, nullptr, rows_bound, L, R, minscore, pos_errs, pos_total, din_errs,
                      din_total, workspace, workspace_bytes, status, 1, stream, seg);
}

int kbbq_marginals(const int64_t *pos_errs, const int64_t *pos_total, int L, int R, int64_t *q_errs,
                   int64_t *q_total, int64_t *rg_errs, int64_t *rg_total, int64_t *meanq, void *stream) {
    if (L < 1 || R < 1 || !pos_errs || !pos_total || !q_errs || !q_total || !rg_errs || !rg_total || !meanq)
        return KBBQ_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int device;
    KBBQ_CUDA(cudaGetDevice(&device));
    int rc = upload_constants(device);
    if (rc) return rc;
    marginals_q_kernel<<<dim3(NQ, R), 128, 0, st>>>((const long long *)pos_errs, (const long long *)pos_total,
                                                   2 * L, (long long *)q_errs, (long long *)q_total);
    KBBQ_LAUNCHED();
    marginals_rg_kernel<<<R, 64, 0, st>>>((const long long *)q_errs, (const long long *)q_total, R,
                                                      (long long *)rg_errs, (long long *)rg_total, (long long *)meanq);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_delta_q(const int64_t *prior_q, const int64_t *numerrs, const int64_t *numtotal, int64_t n,
                 int64_t *delta, void *stream) {
    if (n < 0 || (n > 0 && (!prior_q || !numerrs || !numtotal || !delta))) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    int device;
    KBBQ_CUDA(cudaGetDevice(&device));
    int rc = upload_constants(device);
    if (rc) return rc;
    delta_q_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        (const long long *)prior_q, (const long long *)numerrs, (const long long *)numtotal, n, (long long *)delta);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_posterior_q_real(const double *prior_q, const int64_t *numerrs, const int64_t *numtotal, int64_t n,
                          int64_t *posterior, void *stream) {
    if (n < 0 || (n > 0 && (!prior_q || !numerrs || !numtotal || !posterior))) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    int device;
    KBBQ_CUDA(cudaGetDevice(&device));
    int rc = upload_constants(device);
    if (rc) return rc;
    posterior_q_real_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        prior_q, (const long long *)numerrs, (const long long *)numtotal, n, (long long *)posterior);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

// Workspace of the BAM-side entry points: the canonical copies of the batch (bam.cuh) followed by the
// workspace of kbbq_build / kbbq_apply.
struct BamWorkspace {
    uint8_t *cseq, *cqual, *cthird, *csecond;  // third array: corrected reads (build) / canonical output (apply)
    void *inner;
    size_t inner_bytes, bytes;
};
static BamWorkspace carve_bam_workspace(void *base, long long N, int L, int R) {
    BamWorkspace w = {};
    char *p = (char *)base;
    size_t off = 0;
    const size_t nb = align_up((size_t)N * L + 16, 256);
    w.cseq = (uint8_t *)(p + off); off += nb;
    w.cqual = (uint8_t *)(p + off); off += nb;
    w.cthird = (uint8_t *)(p + off); off += nb;
    w.csecond = (uint8_t *)(p + off); off += align_up((size_t)N + 16, 256);
    w.inner = p + off;
    w.inner_bytes = carve_workspace(nullptr, N, L, R).bytes;
    w.bytes = off + w.inner_bytes;
    return w;
}

// one thread per output word; 32-bit thread indices, so very large batches take several launches
static int launch_bam_canon(const BamCanonArgs &c, cudaStream_t st) {
    const unsigned int wmax = (unsigned int)((3 + c.L + 3) >> 2);
    const long long per = std::max<long long>(1, (long long)(0x7FFFFFFFu / wmax) / 256 * 256);
    for (long long r0 = 0; r0 < c.N; r0 += per) {
        const long long n = std::min<long long>(per, c.N - r0);
        bam_canon_kernel<<<(unsigned)((n * wmax + BAM_WARPS * 32 - 1) / (BAM_WARPS * 32)), BAM_WARPS * 32, 0, st>>>(c, r0, wmax);
        KBBQ_LAUNCHED();
    }
    return KBBQ_OK;
}

int kbbq_bam_workspace_bytes(int64_t N, int L, int R, size_t *bytes) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || !bytes) return KBBQ_E_ARG;
    *bytes = carve_bam_workspace(nullptr, N, L, R).bytes;
    return KBBQ_OK;
}

int kbbq_build_bam(const uint8_t *seq, const uint8_t *qual, const uint8_t *err, const uint8_t *skip, const uint16_t *rg,
                   const uint8_t *flags, const uint16_t *aln_start, const uint16_t *aln_end, int64_t N, int L, int R,
                   int minscore, int64_t *pos_errs, int64_t *pos_total, int64_t *din_errs, int64_t *din_total,
                   void *workspace, size_t workspace_bytes, int *status, void *stream) {
    if (N < 0 || L < 1 || L > 32767 || R < 1 || R > 65535 || minscore < 0 || minscore >= NQ) return KBBQ_E_ARG;
    if (!pos_errs || !pos_total || !din_errs || !din_total || !status) return KBBQ_E_ARG;
    if (N == 0) return KBBQ_OK;
    if (!seq || !qual || !err) return KBBQ_E_ARG;
    int device, sms = KBBQ_SM_COUNT_FALLBACK;
    KBBQ_CUDA(cudaGetDevice(&device));
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    cudaStream_t st = (cudaStream_t)stream;
    const long long blocks = std::min<long long>(((long long)N * L + 255) / 256, (long long)sms * 16);
    if (workspace && minscore >= 1) {  // canonical form + the shared-memory build kernel
        BamWorkspace w = carve_bam_workspace(workspace, N, L, R);
        if (workspace_bytes < w.bytes) return KBBQ_E_WORKSPACE;
        BamCanonArgs c = {seq, qual, err, skip, rg, flags, aln_start, aln_end, N, L, R, minscore, NQ, true,
                          w.cseq, w.cqual, w.cthird, w.csecond,
                          (unsigned long long *)pos_errs, (unsigned long long *)pos_total,
                          (unsigned long long *)din_errs, (unsigned long long *)din_total, status};
        { const int rc_ = launch_bam_canon(c, st); if (rc_) return rc_; }
        return kbbq_build(w.cseq, w.cqual, w.cthird, rg, w.csecond, N, L, R, minscore, pos_errs, pos_total, din_errs,
                          din_total, w.inner, w.inner_bytes, status, 0, stream);
    }
    // no workspace (or minscore 0, where no quality can mean "skip"): direct kernel, global atomics
    BuildBamArgs a = {seq, qual, err, skip, rg, flags, aln_start, aln_end, N, L, R, minscore,
                      (unsigned long long *)pos_errs, (unsigned long long *)pos_total,
                      (unsigned long long *)din_errs, (unsigned long long *)din_total, status};
    build_bam_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_apply_bam(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *flags, int64_t N, int L,
                   int R, int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                   const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual, void *workspace,
                   size_t workspace_bytes, int *status, void *stream) {
    if (N < 0 || L < 1 || L > 32767 || R < 1 || R > 65535 || minscore < 0 || minscore >= NQ || nq < 1 || nq > 256 ||
        ndin1 != 17)
        return KBBQ_E_ARG;
    if (!meanq || !rgdq || !qdq || !posdq || !dindq || !status) return KBBQ_E_ARG;
    if (N == 0) return KBBQ_OK;
    if (!seq || !qual || !out_qual) return KBBQ_E_ARG;
    int device, sms = KBBQ_SM_COUNT_FALLBACK;
    KBBQ_CUDA(cudaGetDevice(&device));
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    cudaStream_t st = (cudaStream_t)stream;
    const long long blocks = std::min<long long>(((long long)N * L + 255) / 256, (long long)sms * 16);
    if (workspace && minscore >= 1 && nq <= NQ) {  // canonical form + the shared-memory apply kernel + flip back
        BamWorkspace w = carve_bam_workspace(workspace, N, L, R);
        if (workspace_bytes < w.bytes) return KBBQ_E_WORKSPACE;
        BamCanonArgs c = {seq, qual, nullptr, nullptr, rg, flags, nullptr, nullptr, N, L, R, minscore, nq, false,
                          w.cseq, w.cqual, nullptr, w.csecond, nullptr, nullptr, nullptr, nullptr, status};
        { const int rc_ = launch_bam_canon(c, st); if (rc_) return rc_; }
        // the canonical reads hold A, C, G, T, N only: bam_canon_kernel has already applied the reference's rule
        int rc = kbbq_apply(w.cseq, w.cqual, rg, w.csecond, N, L, R, minscore, meanq, rgdq, qdq, posdq, dindq, nq, ndin1,
                            w.cthird, w.inner, w.inner_bytes, status, KBBQ_APPLY_BASES_CHECKED, stream);
        if (rc) return rc;
        {
            const unsigned int wmax = (unsigned int)((3 + L + 3) >> 2);
            const long long per = std::max<long long>(1, (long long)(0x7FFFFFFFu / wmax) / 256 * 256);  // reads per launch
            for (long long r0 = 0; r0 < N; r0 += per) {
                const long long n = std::min<long long>(per, N - r0);
                bam_uncanon_kernel<<<(unsigned)((n * wmax + BAM_WARPS * 32 - 1) / (BAM_WARPS * 32)), BAM_WARPS * 32, 0, st>>>(
                    w.cthird, flags, N, L, out_qual, r0, wmax);
                KBBQ_LAUNCHED();
            }
        }
        return KBBQ_OK;
    }
    ApplyBamArgs a = {seq, qual, rg, flags, out_qual, N, L, R, minscore, nq, ndin1, (const long long *)meanq,
                      (const long long *)rgdq, (const long long *)qdq, (const long long *)posdq,
                      (const long long *)dindq, status};
    apply_bam_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_calibration_counts(const uint8_t *qual, const uint8_t *err, const uint8_t *seq, const uint8_t *corr,
                            const uint8_t *skip, int64_t n, int64_t *total, int64_t *errs, void *stream) {
    if (n < 0 || !total || !errs) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    if (!qual || (!err && (!seq || !corr))) return KBBQ_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int device, sms = KBBQ_SM_COUNT_FALLBACK;
    KBBQ_CUDA(cudaGetDevice(&device));
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    auto misaligned = [](const void *p) { return p && ((uintptr_t)p & 15u); };
    CalibArgs a = {qual, err, seq, corr, skip, n, (unsigned long long *)total, (unsigned long long *)errs};
    if (misaligned(qual) || misaligned(err) || misaligned(skip) || (!err && (misaligned(seq) || misaligned(corr)))) {
        const long long chunk = 1ll << 31;  // a CTA counter is u32
        for (long long o = 0; o < n; o += chunk) {
            CalibArgs c = a;
            c.qual += o; if (err) c.err += o; else { c.seq += o; c.corr += o; } if (skip) c.skip += o;
            c.n = std::min<long long>(chunk, n - o);
            calibration_scalar_kernel<<<sms * 8, CAL_THREADS, 0, st>>>(c);
            KBBQ_LAUNCHED();
        }
        return KBBQ_OK;
    }
    const int grid = sms * 3;  // 3 CTAs of 64 KB shared memory per SM
    const long long chunk = (long long)grid * CAL_THREADS * CAL_MAX_ITERS * 32;  // multiple of 16
    auto kern = err ? (skip ? calibration_kernel<true, true> : calibration_kernel<true, false>)
                    : (skip ? calibration_kernel<false, true> : calibration_kernel<false, false>);
    KBBQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, CAL_SMEM));
    for (long long o = 0; o < n; o += chunk) {
        CalibArgs c = a;
        c.qual += o; if (err) c.err += o; else { c.seq += o; c.corr += o; } if (skip) c.skip += o;
        c.n = std::min<long long>(chunk, n - o);
        kern<<<grid, CAL_THREADS, CAL_SMEM, st>>>(c);
        KBBQ_LAUNCHED();
    }
    return KBBQ_OK;
}

int kbbq_get_delta_qs(const int64_t *meanq, const int64_t *rg_errs, const int64_t *rg_total,
                      const int64_t *q_errs, const int64_t *q_total, const int64_t *pos_errs,
                      const int64_t *pos_total, const int64_t *din_errs, const int64_t *din_total, int R,
                      int nq, int ncyc, int ndin, int64_t *rgdq, int64_t *qdq, int64_t *posdq,
                      int64_t *dindq, void *stream) {
    if (R < 1 || nq < 1 || ncyc < 0 || ndin < 0) return KBBQ_E_ARG;
    if (!meanq || !rg_errs || !rg_total || !q_errs || !q_total || !rgdq || !qdq) return KBBQ_E_ARG;
    if ((ncyc && (!pos_errs || !pos_total || !posdq)) || !dindq || (ndin && (!din_errs || !din_total)))
        return KBBQ_E_ARG;
    int device;
    KBBQ_CUDA(cudaGetDevice(&device));
    int rc = upload_constants(device);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    DeltaArgs a = {(const long long *)meanq, (const long long *)rg_errs, (const long long *)rg_total,
                   (const long long *)q_errs, (const long long *)q_total, (const long long *)pos_errs,
                   (const long long *)pos_total, (const long long *)din_errs, (const long long *)din_total,
                   R, nq, ncyc, ndin, (long long *)rgdq, (long long *)qdq, (long long *)posdq, (long long *)dindq};
    delta_levels12_kernel<<<R, 64, 0, st>>>(a);
    KBBQ_LAUNCHED();
    const long long cells = (long long)R * nq * (ncyc + ndin + 1);
    delta_level3_kernel<<<(unsigned)((cells + 127) / 128), 128, 0, st>>>(a);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

static int apply_impl(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second, int64_t N,
                      int L, int R, int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                      const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual,
                      void *workspace, size_t workspace_bytes, int *status, int path, void *stream,
                      const unsigned int *seg_rows) {
    const bool segmode = seg_rows != nullptr;
    const bool validate = !(path & KBBQ_APPLY_BASES_CHECKED);
    path &= ~KBBQ_APPLY_BASES_CHECKED;
    if (N < 0 || L < 1 || R < 1 || R > 65535 || minscore < 0 || minscore >= NQ) return KBBQ_E_ARG;
    if (nq < 1 || nq > NQ || ndin1 < 16 || ndin1 > 64) return KBBQ_E_ARG;
    if (!meanq || !rgdq || !qdq || !posdq || !dindq || !status) return KBBQ_E_ARG;
    if (N == 0) return KBBQ_OK;
    if (!seq || !qual || !out_qual) return KBBQ_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    Workspace w = carve_workspace(workspace, N, L, R);
    if (!workspace || workspace_bytes < w.bytes) return KBBQ_E_WORKSPACE;

    const long long fold_cells = (long long)R * NQ * (2 * L + 16);
    fold_kernel<<<(unsigned)((fold_cells + 255) / 256), 256, 0, st>>>(
        (const long long *)meanq, (const long long *)rgdq, (const long long *)qdq, (const long long *)posdq,
        (const long long *)dindq, R, nq, 2 * L, ndin1, w.fold_cyc, w.fold_din);
    KBBQ_LAUNCHED();

    Geom g;
    TableCfg tc;
    StageLayout sl;
    const bool smem_ok = path != 2 && !misaligned(seq, 16) && !misaligned(qual, 16) && !misaligned(out_qual, 4) &&
                         plan_kernel(L, R, minscore, 2, max_smem, &g, &tc, &sl, segmode) &&
                         (uint64_t)((N + g.G - 1) / g.G) < 0xFFFFFFFFull;
    if (!smem_ok) {
        if (path == 1 || segmode) return KBBQ_E_ARG;
        ApplyGenericArgs a = {seq, qual, rg, second, out_qual, N, L, R, minscore, nq, w.fold_cyc, w.fold_din, status, validate};
        apply_generic_kernel<<<sms * 8, 256, 0, st>>>(a);
        KBBQ_LAUNCHED();
        return KBBQ_OK;
    }
    const int64_t tail = (!segmode && R == 1 && N > g.G) ? N % g.G : 0;  // see kbbq_build
    if (tail) {
        const int64_t n0 = N - tail;
        ApplyGenericArgs ga = {seq + n0 * L, qual + n0 * L, rg ? rg + n0 : nullptr, second ? second + n0 : nullptr,
                               out_qual + n0 * L, tail, L, R, minscore, nq, w.fold_cyc, w.fold_din, status, validate};
        apply_generic_kernel<<<1, 256, 0, st>>>(ga);
        KBBQ_LAUNCHED();
        N = n0;
    }
    if (segmode) {
        seg_prepare_kernel<<<1, 256, 0, st>>>(seg_rows, 2 * R, g.G, (unsigned long long)N, w.seg, w.uni, status);
        KBBQ_LAUNCHED();
    } else {
        rc = run_prepare(rg, second, N, g.G, R, w, status, sms, sl.ngs, g.gbytes, sl.slot, st);
        if (rc) return rc;
    }
    ApplyArgs a;
    a.nsub = segmode ? 2 * R : R; a.segmode = segmode ? 1 : 0;
    a.seq = seq; a.qual = qual; a.out = out_qual; a.total_bytes = N * L; a.g = g; a.t = tc; a.R = R; a.nq = nq;
    a.sl = sl;
    a.entries = w.entries; a.seg = w.seg; a.uni = w.uni; a.fold_cyc = w.fold_cyc; a.fold_din = w.fold_din; a.status = status;
    return launch_apply_smem(a, validate, sms, a.sl.total, st);
}

int kbbq_apply(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second, int64_t N,
               int L, int R, int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
               const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual,
               void *workspace, size_t workspace_bytes, int *status, int path, void *stream) {
    return apply_impl(seq, qual, rg, second, N, L, R, minscore, meanq, rgdq, qdq, posdq, dindq, nq, ndin1, out_qual,
                      workspace, workspace_bytes, status, path, stream, nullptr);
}

int kbbq_apply_segmented_flags(const uint8_t *seq, const uint8_t *qual, const uint32_t *seg, int64_t rows_bound, int L,
                               int R, int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                               const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual,
                               void *workspace, size_t workspace_bytes, int *status, int flags, void *stream) {
    if (!seg || rows_bound % SEG_ALIGN || (flags & ~KBBQ_APPLY_BASES_CHECKED)) return KBBQ_E_ARG;
    return apply_impl(seq, qual, nullptr, nullptr, rows_bound, L, R, minscore, meanq, rgdq, qdq, posdq, dindq, nq, ndin1,
                      out_qual, workspace, workspace_bytes, status, 1 | flags, stream, seg);
}

int kbbq_apply_segmented(const uint8_t *seq, const uint8_t *qual, const uint32_t *seg, int64_t rows_bound, int L, int R,
                         int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                         const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual,
                         void *workspace, size_t workspace_bytes, int *status, void *stream) {
    return kbbq_apply_segmented_flags(seq, qual, seg, rows_bound, L, R, minscore, meanq, rgdq, qdq, posdq, dindq, nq, ndin1,
                                      out_qual, workspace, workspace_bytes, status, 0, stream);
}

// ---- segmented batch layout (segment.cuh) ----

int64_t kbbq_segment_rows_bound(int64_t N, int R) {
    if (N < 0 || R < 1) return -1;
    return (N + SEG_ALIGN - 1) / SEG_ALIGN * SEG_ALIGN + (int64_t)2 * R * SEG_ALIGN;
}

int64_t kbbq_segment_table_elems(int R) { return R < 1 ? -1 : (int64_t)6 * R + 1; }

int kbbq_segmented_supported(int L, int R, int minscore) {
    if (L < 1 || R < 1 || R > 65535) return 0;
    Geom g;
    TableCfg tc;
    StageLayout sl;
    return plan_kernel(L, R, minscore, 3, 232448, &g, &tc, &sl, true) && plan_kernel(L, R, minscore, 2, 232448, &g, &tc, &sl, true);
}

int kbbq_segment_plan(const uint16_t *rg, const uint8_t *second, int64_t N, int R, uint32_t *seg, uint32_t *dest,
                      int *status, void *stream) {
    if (N < 0 || R < 1 || R > 65535 || !seg || !status || (N > 0 && !dest)) return KBBQ_E_ARG;
    if (kbbq_segment_rows_bound(N, R) >= 0xFFFFFFFFll) return KBBQ_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int nkeys = 2 * R;
    SegPlanArgs a = {rg, second, N, R, seg, seg + 2 * nkeys + 1, dest, status};
    KBBQ_CUDA(cudaMemsetAsync(a.cursor, 0, sizeof(unsigned int) * nkeys, st));
    const int per_thread = 8;
    const long long per_block = (long long)SEG_THREADS * per_thread;
    const unsigned int blocks = (unsigned int)((N + per_block - 1) / per_block);
    const size_t smem = nkeys <= SEG_SMEM_KEYS ? sizeof(unsigned int) * nkeys : 0;
    if (blocks) {
        seg_bucket_kernel<0><<<blocks, SEG_THREADS, smem, st>>>(a, per_thread);
        KBBQ_LAUNCHED();
    }
    seg_scan_kernel<<<1, 1024, 0, st>>>(a);
    KBBQ_LAUNCHED();
    if (blocks) {
        seg_bucket_kernel<1><<<blocks, SEG_THREADS, smem, st>>>(a, per_thread);
        KBBQ_LAUNCHED();
    }
    return KBBQ_OK;
}

static int move_rows(const uint8_t *src, const uint32_t *dest, int64_t N, int L, uint8_t *dst, int64_t src_rows, bool scatter,
                     cudaStream_t st) {
    if (N < 0 || L < 1 || src_rows < 0) return KBBQ_E_ARG;
    if (N == 0) return KBBQ_OK;
    if (!src || !dest || !dst) return KBBQ_E_ARG;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    const long long warps_per_block = SEG_THREADS / 32;
    const unsigned int blocks = (unsigned int)std::min<long long>((N + warps_per_block - 1) / warps_per_block, (long long)sms * 32);
    if (scatter) seg_move_rows_kernel<true><<<blocks, SEG_THREADS, 0, st>>>(src, dst, dest, N, L, src_rows);
    else seg_move_rows_kernel<false><<<blocks, SEG_THREADS, 0, st>>>(src, dst, dest, N, L, src_rows);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_segment_rows(const uint8_t *src, const uint32_t *dest, int64_t N, int L, uint8_t *dst_segmented, void *stream) {
    return move_rows(src, dest, N, L, dst_segmented, N, true, (cudaStream_t)stream);
}

int kbbq_unsegment_rows(const uint8_t *src_segmented, const uint32_t *dest, int64_t N, int L, int64_t rows_bound,
                        uint8_t *dst, void *stream) {
    return move_rows(src_segmented, dest, N, L, dst, rows_bound, false, (cudaStream_t)stream);
}

int kbbq_segment_pad(const uint32_t *seg, int R, int L, uint8_t *seq, uint8_t *qual, uint8_t *corr, void *stream) {
    if (!seg || R < 1 || R > 65535 || L < 1) return KBBQ_E_ARG;
    seg_pad_kernel<<<2 * R, 128, 0, (cudaStream_t)stream>>>(seg, 2 * R, L, seq, qual, corr);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_synth_reads(uint64_t seed, int64_t first_read, int64_t n, int L, int R, uint8_t *seq, uint8_t *qual,
                     uint8_t *corr, uint16_t *rg, uint8_t *second, void *stream) {
    if (n < 0 || L < 1 || R < 1 || R > 65535 || first_read < 0) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    if (!seq || !qual || !corr) return KBBQ_E_ARG;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    synth_kernel<<<sms * 16, 256, 0, (cudaStream_t)stream>>>(seed, first_read, n, L, R, seq, qual, corr, rg, second);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

// ------------------------------------------------------------------------------------------------
// Host-buffer entry points
// ------------------------------------------------------------------------------------------------

}  // extern "C"

namespace {

struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t n) { KBBQ_CUDA(cudaMalloc(&p, n ? n : 1)); return KBBQ_OK; }
    template <class T> T *as() { return (T *)p; }
};

// corr[i] = seq[i] ^ bit i of the mismatch map: a byte array that differs from seq exactly where the
// corrected read did (host_pack.cpp), which is all the build kernel looks at.  16 bases per thread.
__global__ void expand_corr_kernel(const uint8_t *seq, const uint32_t *bits, uint8_t *corr, long long n) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long i = t * 16;
    if (i >= n) return;
    const uint32_t m = (bits[t >> 1] >> ((t & 1) * 16)) & 0xFFFFu;
    if (i + 16 <= n) {
        uint4 v = *reinterpret_cast<const uint4 *>(seq + i);
        // bits 0..3 of a nibble -> bit 0 of bytes 0..3
        v.x ^= ((m & 0xFu) * 0x00204081u) & 0x01010101u;
        v.y ^= (((m >> 4) & 0xFu) * 0x00204081u) & 0x01010101u;
        v.z ^= (((m >> 8) & 0xFu) * 0x00204081u) & 0x01010101u;
        v.w ^= (((m >> 12) & 0xFu) * 0x00204081u) & 0x01010101u;
        *reinterpret_cast<uint4 *>(corr + i) = v;
    } else {
        for (int j = 0; i + j < n; ++j) corr[i + j] = seq[i + j] ^ (uint8_t)((m >> j) & 1u);
    }
}

// The 4-bit form of (seq, corrected) (host_pack.cpp: kbbq_host_pack_nibbles) back into two byte arrays: seq from
// the 3-bit base code through a byte-permute table, corr = seq ^ 1 where bit 3 of the nibble says the corrected
// read differed.  32 bases per thread: one 16-byte load, two 16-byte stores per array.
__device__ __forceinline__ void expand_nibbles4(uint32_t p16, uint32_t &sw, uint32_t &cw) {
    // four nibbles = the four selector nibbles of a byte permute over {A C T G | . . . N}
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(sw) : "r"(0x47544341u), "r"(0x4E000000u), "r"(p16 & 0x7777u));
    // bit 3 of nibbles 1, 3 are the sign bits of bytes 0, 1 of p16; those of nibbles 0, 2 after a shift by 4
    const uint32_t w = (p16 & 0xFFFFu) | (p16 << 20);
    uint32_t m;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(m) : "r"(w), "r"(0u), "r"(0x9B8Au));
    cw = sw ^ (m & 0x01010101u);
}

__global__ void expand_nibbles_kernel(const uint8_t *packed, uint8_t *seq, uint8_t *corr, long long n) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long i = t * 32;
    if (i >= n) return;
    if (i + 32 <= n) {
        const uint4 v = *reinterpret_cast<const uint4 *>(packed + i / 2);
        const uint32_t in[4] = {v.x, v.y, v.z, v.w};
        uint32_t s[8], c[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            expand_nibbles4(in[k] & 0xFFFFu, s[2 * k], c[2 * k]);
            expand_nibbles4(in[k] >> 16, s[2 * k + 1], c[2 * k + 1]);
        }
        *reinterpret_cast<uint4 *>(seq + i) = make_uint4(s[0], s[1], s[2], s[3]);
        *reinterpret_cast<uint4 *>(seq + i + 16) = make_uint4(s[4], s[5], s[6], s[7]);
        *reinterpret_cast<uint4 *>(corr + i) = make_uint4(c[0], c[1], c[2], c[3]);
        *reinterpret_cast<uint4 *>(corr + i + 16) = make_uint4(c[4], c[5], c[6], c[7]);
    } else {
        for (long long j = i; j < n; ++j) {
            const uint32_t nib = (packed[j >> 1] >> ((j & 1) * 4)) & 0xFu;
            const uint32_t code = nib & 7u;
            const uint8_t b = code == 7u ? 'N' : code == 0u ? 'A' : code == 1u ? 'C' : code == 2u ? 'T' : code == 3u ? 'G' : 0;
            seq[j] = b;
            corr[j] = b ^ (uint8_t)(nib >> 3);
        }
    }
}

// bump allocator over one device allocation (first pass with base == nullptr measures)
struct Carver {
    char *base;
    size_t off = 0;
    explicit Carver(void *b) : base((char *)b) {}
    template <class T> T *take(size_t n_elems) {
        T *p = base ? (T *)(base + off) : nullptr;
        off = (off + n_elems * sizeof(T) + 255) / 256 * 256;
        return p;
    }
};

#define KBBQ_TRY(x) do { int rc_ = (x); if (rc_) return rc_; } while (0)

}  // namespace

extern "C" {

int kbbq_expand_mismatch_bits(const uint8_t *seq, const uint32_t *bits, int64_t n, uint8_t *corr, void *stream) {
    if (n < 0 || (n > 0 && (!seq || !bits || !corr))) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    if (((uintptr_t)seq | (uintptr_t)corr) & 15u) return KBBQ_E_ARG;
    expand_corr_kernel<<<(unsigned)((n + 16 * 256 - 1) / (16 * 256)), 256, 0, (cudaStream_t)stream>>>(seq, bits, corr, n);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_expand_nibbles(const uint8_t *packed, int64_t n, uint8_t *seq, uint8_t *corr, void *stream) {
    if (n < 0 || (n > 0 && (!packed || !seq || !corr))) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    if (((uintptr_t)packed | (uintptr_t)seq | (uintptr_t)corr) & 15u) return KBBQ_E_ARG;
    expand_nibbles_kernel<<<(unsigned)((n + 32 * 256 - 1) / (32 * 256)), 256, 0, (cudaStream_t)stream>>>(packed, seq, corr, n);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_build_host(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
                    const uint8_t *second, int64_t N, int L, int R, int minscore, int64_t *pos_errs,
                    int64_t *pos_total, int64_t *din_errs, int64_t *din_total, int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535) return KBBQ_E_ARG;
    if (!pos_errs || !pos_total || !din_errs || !din_total) return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(device));
    const size_t npos = (size_t)R * NQ * 2 * L, ndin = (size_t)R * NQ * 16, nb = (size_t)N * L;
    DevBuf d_seq, d_qual, d_corr, d_rg, d_sec, d_tab, d_ws, d_status;
    KBBQ_TRY(d_seq.alloc(nb)); KBBQ_TRY(d_qual.alloc(nb)); KBBQ_TRY(d_corr.alloc(nb));
    KBBQ_TRY(d_tab.alloc((2 * npos + 2 * ndin) * 8));
    KBBQ_TRY(d_status.alloc(sizeof(int)));
    size_t ws_bytes = 0;
    KBBQ_TRY(kbbq_workspace_bytes(N, L, R, &ws_bytes));
    KBBQ_TRY(d_ws.alloc(ws_bytes));
    KBBQ_CUDA(cudaMemcpy(d_seq.p, seq, nb, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(d_qual.p, qual, nb, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(d_corr.p, corr, nb, cudaMemcpyHostToDevice));
    if (rg) { KBBQ_TRY(d_rg.alloc((size_t)N * 2)); KBBQ_CUDA(cudaMemcpy(d_rg.p, rg, (size_t)N * 2, cudaMemcpyHostToDevice)); }
    if (second) { KBBQ_TRY(d_sec.alloc((size_t)N)); KBBQ_CUDA(cudaMemcpy(d_sec.p, second, (size_t)N, cudaMemcpyHostToDevice)); }
    KBBQ_CUDA(cudaMemset(d_tab.p, 0, (2 * npos + 2 * ndin) * 8));
    KBBQ_CUDA(cudaMemset(d_status.p, 0, sizeof(int)));
    int64_t *pe = d_tab.as<int64_t>(), *pt = pe + npos, *de = pt + npos, *dt = de + ndin;
    KBBQ_TRY(kbbq_build(d_seq.as<uint8_t>(), d_qual.as<uint8_t>(), d_corr.as<uint8_t>(), rg ? d_rg.as<uint16_t>() : nullptr,
                        second ? d_sec.as<uint8_t>() : nullptr, N, L, R, minscore, pe, pt, de, dt, d_ws.p, ws_bytes,
                        d_status.as<int>(), 0, nullptr));
    KBBQ_CUDA(cudaMemcpy(pos_errs, pe, npos * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(pos_total, pt, npos * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(din_errs, de, ndin * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(din_total, dt, ndin * 8, cudaMemcpyDeviceToHost));
    int st_host = 0;
    KBBQ_CUDA(cudaMemcpy(&st_host, d_status.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (status_out) *status_out = st_host;
    return st_host ? KBBQ_E_DATA : KBBQ_OK;
}

int kbbq_apply_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second, int64_t N,
                    int L, int R, int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                    const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual,
                    int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || nq < 1 || nq > NQ || ndin1 < 16 || ndin1 > 64) return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(device));
    const size_t nb = (size_t)N * L;
    const size_t n_q = (size_t)R * nq, n_pos = n_q * 2 * L, n_din = n_q * ndin1;
    DevBuf d_seq, d_qual, d_out, d_rg, d_sec, d_dq, d_ws, d_status;
    KBBQ_TRY(d_seq.alloc(nb)); KBBQ_TRY(d_qual.alloc(nb)); KBBQ_TRY(d_out.alloc(nb));
    KBBQ_TRY(d_dq.alloc((2 * (size_t)R + n_q + n_pos + n_din) * 8));
    KBBQ_TRY(d_status.alloc(sizeof(int)));
    size_t ws_bytes = 0;
    KBBQ_TRY(kbbq_workspace_bytes(N, L, R, &ws_bytes));
    KBBQ_TRY(d_ws.alloc(ws_bytes));
    int64_t *d_meanq = d_dq.as<int64_t>(), *d_rgdq = d_meanq + R, *d_qdq = d_rgdq + R, *d_posdq = d_qdq + n_q,
            *d_dindq = d_posdq + n_pos;
    KBBQ_CUDA(cudaMemcpy(d_seq.p, seq, nb, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(d_qual.p, qual, nb, cudaMemcpyHostToDevice));
    if (rg) { KBBQ_TRY(d_rg.alloc((size_t)N * 2)); KBBQ_CUDA(cudaMemcpy(d_rg.p, rg, (size_t)N * 2, cudaMemcpyHostToDevice)); }
    if (second) { KBBQ_TRY(d_sec.alloc((size_t)N)); KBBQ_CUDA(cudaMemcpy(d_sec.p, second, (size_t)N, cudaMemcpyHostToDevice)); }
    KBBQ_CUDA(cudaMemcpy(d_meanq, meanq, (size_t)R * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(d_rgdq, rgdq, (size_t)R * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(d_qdq, qdq, n_q * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(d_posdq, posdq, n_pos * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(d_dindq, dindq, n_din * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemset(d_status.p, 0, sizeof(int)));
    KBBQ_TRY(kbbq_apply(d_seq.as<uint8_t>(), d_qual.as<uint8_t>(), rg ? d_rg.as<uint16_t>() : nullptr,
                        second ? d_sec.as<uint8_t>() : nullptr, N, L, R, minscore, d_meanq, d_rgdq, d_qdq, d_posdq,
                        d_dindq, nq, ndin1, d_out.as<uint8_t>(), d_ws.p, ws_bytes, d_status.as<int>(), 0, nullptr));
    KBBQ_CUDA(cudaMemcpy(out_qual, d_out.p, nb, cudaMemcpyDeviceToHost));
    int st_host = 0;
    KBBQ_CUDA(cudaMemcpy(&st_host, d_status.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (status_out) *status_out = st_host;
    return st_host ? KBBQ_E_DATA : KBBQ_OK;
}

int kbbq_get_delta_qs_host(const int64_t *meanq, const int64_t *rg_errs, const int64_t *rg_total,
                           const int64_t *q_errs, const int64_t *q_total, const int64_t *pos_errs,
                           const int64_t *pos_total, const int64_t *din_errs, const int64_t *din_total, int R,
                           int nq, int ncyc, int ndin, int64_t *rgdq, int64_t *qdq, int64_t *posdq,
                           int64_t *dindq, int device) {
    if (R < 1 || nq < 1 || ncyc < 0 || ndin < 0) return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(device));
    const size_t n_q = (size_t)R * nq, n_pos = n_q * ncyc, n_din = n_q * ndin, n_din1 = n_q * (ndin + 1);
    const size_t in_elems = 3 * (size_t)R + 2 * n_q + 2 * n_pos + 2 * n_din;
    const size_t out_elems = (size_t)R + n_q + n_pos + n_din1;
    DevBuf d;
    KBBQ_TRY(d.alloc((in_elems + out_elems) * 8));
    int64_t *p = d.as<int64_t>();
    int64_t *d_meanq = p; p += R;
    int64_t *d_rge = p; p += R;
    int64_t *d_rgt = p; p += R;
    int64_t *d_qe = p; p += n_q;
    int64_t *d_qt = p; p += n_q;
    int64_t *d_pe = p; p += n_pos;
    int64_t *d_pt = p; p += n_pos;
    int64_t *d_de = p; p += n_din;
    int64_t *d_dt = p; p += n_din;
    int64_t *o_rg = p; p += R;
    int64_t *o_q = p; p += n_q;
    int64_t *o_pos = p; p += n_pos;
    int64_t *o_din = p;
    const struct { int64_t *dst; const int64_t *src; size_t n; } ups[] = {
        {d_meanq, meanq, (size_t)R}, {d_rge, rg_errs, (size_t)R}, {d_rgt, rg_total, (size_t)R}, {d_qe, q_errs, n_q},
        {d_qt, q_total, n_q}, {d_pe, pos_errs, n_pos}, {d_pt, pos_total, n_pos}, {d_de, din_errs, n_din},
        {d_dt, din_total, n_din}};
    for (auto &u : ups)
        if (u.n) KBBQ_CUDA(cudaMemcpy(u.dst, u.src, u.n * 8, cudaMemcpyHostToDevice));
    KBBQ_TRY(kbbq_get_delta_qs(d_meanq, d_rge, d_rgt, d_qe, d_qt, d_pe, d_pt, d_de, d_dt, R, nq, ncyc, ndin, o_rg, o_q,
                               o_pos, o_din, nullptr));
    KBBQ_CUDA(cudaMemcpy(rgdq, o_rg, (size_t)R * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(qdq, o_q, n_q * 8, cudaMemcpyDeviceToHost));
    if (n_pos) KBBQ_CUDA(cudaMemcpy(posdq, o_pos, n_pos * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(dindq, o_din, n_din1 * 8, cudaMemcpyDeviceToHost));
    return KBBQ_OK;
}

int kbbq_delta_q_host(const int64_t *prior_q, const int64_t *numerrs, const int64_t *numtotal, int64_t n,
                      int64_t *delta, int device) {
    if (n < 0) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    KBBQ_CUDA(cudaSetDevice(device));
    DevBuf d;
    KBBQ_TRY(d.alloc((size_t)n * 4 * 8));
    int64_t *p = d.as<int64_t>();
    KBBQ_CUDA(cudaMemcpy(p, prior_q, (size_t)n * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(p + n, numerrs, (size_t)n * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(p + 2 * n, numtotal, (size_t)n * 8, cudaMemcpyHostToDevice));
    KBBQ_TRY(kbbq_delta_q(p, p + n, p + 2 * n, n, p + 3 * n, nullptr));
    KBBQ_CUDA(cudaMemcpy(delta, p + 3 * n, (size_t)n * 8, cudaMemcpyDeviceToHost));
    return KBBQ_OK;
}

int kbbq_posterior_q_real_host(const double *prior_q, const int64_t *numerrs, const int64_t *numtotal, int64_t n,
                               int64_t *posterior, int device) {
    if (n < 0) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    KBBQ_CUDA(cudaSetDevice(device));
    DevBuf d;
    KBBQ_TRY(d.alloc((size_t)n * 4 * 8));
    int64_t *p = d.as<int64_t>();
    KBBQ_CUDA(cudaMemcpy(p, prior_q, (size_t)n * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(p + n, numerrs, (size_t)n * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(p + 2 * n, numtotal, (size_t)n * 8, cudaMemcpyHostToDevice));
    KBBQ_TRY(kbbq_posterior_q_real(reinterpret_cast<const double *>(p), p + n, p + 2 * n, n, p + 3 * n, nullptr));
    KBBQ_CUDA(cudaMemcpy(posterior, p + 3 * n, (size_t)n * 8, cudaMemcpyDeviceToHost));
    return KBBQ_OK;
}

// Host-buffer forms of the BAM-side entry points: copy, run, copy back (a BAM batch is small next to
// what the host spends parsing it).
int kbbq_build_bam_host(const uint8_t *seq, const uint8_t *qual, const uint8_t *err, const uint8_t *skip,
                        const uint16_t *rg, const uint8_t *flags, const uint16_t *aln_start, const uint16_t *aln_end,
                        int64_t N, int L, int R, int minscore, int64_t *pos_errs, int64_t *pos_total,
                        int64_t *din_errs, int64_t *din_total, int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535) return KBBQ_E_ARG;
    if (!pos_errs || !pos_total || !din_errs || !din_total) return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(device));
    const size_t npos = (size_t)R * NQ * 2 * L, ndin = (size_t)R * NQ * 16, nb = (size_t)N * L;
    Carver c(nullptr);
    auto carve = [&](Carver &cv, uint8_t **ds, uint8_t **dq, uint8_t **de, uint8_t **dk, uint16_t **dr, uint8_t **df,
                     uint16_t **d0, uint16_t **d1, int64_t **dt, int **dst) {
        *ds = cv.take<uint8_t>(nb); *dq = cv.take<uint8_t>(nb); *de = cv.take<uint8_t>(nb); *dk = cv.take<uint8_t>(nb);
        *dr = cv.take<uint16_t>((size_t)N); *df = cv.take<uint8_t>((size_t)N);
        *d0 = cv.take<uint16_t>((size_t)N); *d1 = cv.take<uint16_t>((size_t)N);
        *dt = cv.take<int64_t>(2 * npos + 2 * ndin); *dst = cv.take<int>(64);
    };
    uint8_t *ds, *dq, *de, *dk, *df; uint16_t *dr, *d0, *d1; int64_t *dt; int *dst;
    carve(c, &ds, &dq, &de, &dk, &dr, &df, &d0, &d1, &dt, &dst);
    DevBuf buf;
    KBBQ_TRY(buf.alloc(c.off));
    Carver c2(buf.p);
    carve(c2, &ds, &dq, &de, &dk, &dr, &df, &d0, &d1, &dt, &dst);
    auto up = [&](void *d, const void *h, size_t n) { return h && n ? cudaMemcpy(d, h, n, cudaMemcpyHostToDevice) : cudaSuccess; };
    KBBQ_CUDA(up(ds, seq, nb)); KBBQ_CUDA(up(dq, qual, nb)); KBBQ_CUDA(up(de, err, nb)); KBBQ_CUDA(up(dk, skip, nb));
    KBBQ_CUDA(up(dr, rg, (size_t)N * 2)); KBBQ_CUDA(up(df, flags, (size_t)N));
    KBBQ_CUDA(up(d0, aln_start, (size_t)N * 2)); KBBQ_CUDA(up(d1, aln_end, (size_t)N * 2));
    KBBQ_CUDA(cudaMemcpy(dt, pos_errs, npos * 8, cudaMemcpyHostToDevice));   // the tables accumulate
    KBBQ_CUDA(cudaMemcpy(dt + npos, pos_total, npos * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(dt + 2 * npos, din_errs, ndin * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(dt + 2 * npos + ndin, din_total, ndin * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemset(dst, 0, sizeof(int)));
    size_t ws_bytes = 0;
    KBBQ_TRY(kbbq_bam_workspace_bytes(N, L, R, &ws_bytes));
    DevBuf ws;
    KBBQ_TRY(ws.alloc(ws_bytes));
    KBBQ_TRY(kbbq_build_bam(ds, dq, de, skip ? dk : nullptr, rg ? dr : nullptr, flags ? df : nullptr,
                            aln_start ? d0 : nullptr, aln_end ? d1 : nullptr, N, L, R, minscore, dt, dt + npos,
                            dt + 2 * npos, dt + 2 * npos + ndin, ws.p, ws_bytes, dst, nullptr));
    KBBQ_CUDA(cudaMemcpy(pos_errs, dt, npos * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(pos_total, dt + npos, npos * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(din_errs, dt + 2 * npos, ndin * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(din_total, dt + 2 * npos + ndin, ndin * 8, cudaMemcpyDeviceToHost));
    int st = 0;
    KBBQ_CUDA(cudaMemcpy(&st, dst, sizeof(int), cudaMemcpyDeviceToHost));
    if (status_out) *status_out = st;
    return st ? KBBQ_E_DATA : KBBQ_OK;
}

int kbbq_apply_bam_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *flags, int64_t N,
                        int L, int R, int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                        const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual,
                        int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || nq < 1 || ndin1 != 17) return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(device));
    const size_t nb = (size_t)N * L, n_q = (size_t)R * nq;
    uint8_t *ds, *dq, *dout, *df; uint16_t *dr; int64_t *dm; int *dst;
    DevBuf buf;
    for (int pass = 0; pass < 2; ++pass) {
        Carver cv(pass ? buf.p : nullptr);
        ds = cv.take<uint8_t>(nb); dq = cv.take<uint8_t>(nb); dout = cv.take<uint8_t>(nb);
        dr = cv.take<uint16_t>((size_t)N); df = cv.take<uint8_t>((size_t)N);
        dm = cv.take<int64_t>(2 * (size_t)R + n_q * (1 + 2 * (size_t)L + ndin1)); dst = cv.take<int>(64);
        if (!pass) KBBQ_TRY(buf.alloc(cv.off));
    }
    int64_t *d_meanq = dm, *d_rgdq = dm + R, *d_qdq = d_rgdq + R, *d_posdq = d_qdq + n_q, *d_dindq = d_posdq + n_q * 2 * L;
    auto up = [&](void *d, const void *h, size_t n) { return h && n ? cudaMemcpy(d, h, n, cudaMemcpyHostToDevice) : cudaSuccess; };
    KBBQ_CUDA(up(ds, seq, nb)); KBBQ_CUDA(up(dq, qual, nb));
    KBBQ_CUDA(up(dr, rg, (size_t)N * 2)); KBBQ_CUDA(up(df, flags, (size_t)N));
    KBBQ_CUDA(up(d_meanq, meanq, (size_t)R * 8)); KBBQ_CUDA(up(d_rgdq, rgdq, (size_t)R * 8));
    KBBQ_CUDA(up(d_qdq, qdq, n_q * 8)); KBBQ_CUDA(up(d_posdq, posdq, n_q * 2 * L * 8));
    KBBQ_CUDA(up(d_dindq, dindq, n_q * ndin1 * 8));
    KBBQ_CUDA(cudaMemset(dst, 0, sizeof(int)));
    size_t ws_bytes = 0;
    KBBQ_TRY(kbbq_bam_workspace_bytes(N, L, R, &ws_bytes));
    DevBuf ws;
    KBBQ_TRY(ws.alloc(ws_bytes));
    KBBQ_TRY(kbbq_apply_bam(ds, dq, rg ? dr : nullptr, flags ? df : nullptr, N, L, R, minscore, d_meanq, d_rgdq, d_qdq,
                            d_posdq, d_dindq, nq, ndin1, dout, ws.p, ws_bytes, dst, nullptr));
    if (nb) KBBQ_CUDA(cudaMemcpy(out_qual, dout, nb, cudaMemcpyDeviceToHost));
    int st = 0;
    KBBQ_CUDA(cudaMemcpy(&st, dst, sizeof(int), cudaMemcpyDeviceToHost));
    if (status_out) *status_out = st;
    return st ? KBBQ_E_DATA : KBBQ_OK;
}

int kbbq_calibration_counts_host(const uint8_t *qual, const uint8_t *err, const uint8_t *seq, const uint8_t *corr,
                                 const uint8_t *skip, int64_t n, int64_t *total, int64_t *errs, int device) {
    if (n < 0 || !total || !errs) return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(device));
    const size_t nb = ((size_t)n + 15) / 16 * 16;
    const int narr = 1 + (err ? 1 : 2) + (skip ? 1 : 0);
    DevBuf d;
    KBBQ_TRY(d.alloc(nb * narr + 2 * 256 * 8));
    uint8_t *p = d.as<uint8_t>();
    int64_t *cnt = reinterpret_cast<int64_t *>(p + nb * narr);
    KBBQ_CUDA(cudaMemset(cnt, 0, 2 * 256 * 8));
    uint8_t *dq = p, *de = nullptr, *ds = nullptr, *dc = nullptr, *dk = nullptr;
    size_t o = nb;
    KBBQ_CUDA(cudaMemcpy(dq, qual, (size_t)n, cudaMemcpyHostToDevice));
    if (err) { de = p + o; o += nb; KBBQ_CUDA(cudaMemcpy(de, err, (size_t)n, cudaMemcpyHostToDevice)); }
    else {
        if (!seq || !corr) return KBBQ_E_ARG;
        ds = p + o; o += nb; dc = p + o; o += nb;
        KBBQ_CUDA(cudaMemcpy(ds, seq, (size_t)n, cudaMemcpyHostToDevice));
        KBBQ_CUDA(cudaMemcpy(dc, corr, (size_t)n, cudaMemcpyHostToDevice));
    }
    if (skip) { dk = p + o; KBBQ_CUDA(cudaMemcpy(dk, skip, (size_t)n, cudaMemcpyHostToDevice)); }
    KBBQ_TRY(kbbq_calibration_counts(dq, de, ds, dc, dk, n, cnt, cnt + 256, nullptr));
    KBBQ_CUDA(cudaMemcpy(total, cnt, 256 * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(errs, cnt + 256, 256 * 8, cudaMemcpyDeviceToHost));
    return KBBQ_OK;
}

int kbbq_marginals_host(const int64_t *pos_errs, const int64_t *pos_total, int L, int R, int64_t *q_errs,
                        int64_t *q_total, int64_t *rg_errs, int64_t *rg_total, int64_t *meanq, int device) {
    if (L < 1 || R < 1) return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(device));
    const size_t npos = (size_t)R * NQ * 2 * L, n_q = (size_t)R * NQ;
    DevBuf d;
    KBBQ_TRY(d.alloc((2 * npos + 2 * n_q + 3 * (size_t)R) * 8));
    int64_t *pe = d.as<int64_t>(), *pt = pe + npos, *qe = pt + npos, *qt = qe + n_q, *ge = qt + n_q, *gt = ge + R,
            *mq = gt + R;
    KBBQ_CUDA(cudaMemcpy(pe, pos_errs, npos * 8, cudaMemcpyHostToDevice));
    KBBQ_CUDA(cudaMemcpy(pt, pos_total, npos * 8, cudaMemcpyHostToDevice));
    KBBQ_TRY(kbbq_marginals(pe, pt, L, R, qe, qt, ge, gt, mq, nullptr));
    KBBQ_CUDA(cudaMemcpy(q_errs, qe, n_q * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(q_total, qt, n_q * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(rg_errs, ge, (size_t)R * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(rg_total, gt, (size_t)R * 8, cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(meanq, mq, (size_t)R * 8, cudaMemcpyDeviceToHost));
    return KBBQ_OK;
}

}  // extern "C"
