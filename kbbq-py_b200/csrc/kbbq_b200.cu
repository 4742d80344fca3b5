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
#include "expand.cuh"
#include "kmer.cuh"
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

static int upload_constants() {
    int device;
    KBBQ_CUDA(cudaGetDevice(&device));
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

// The shared-memory kernels by groups per thread-group and stage (plan_smem: 1..8); apply also by whether it checks
// the bases
static void (*const build_smem_kernels[8])(BuildArgs) = {
    build_smem_kernel<1, true>, build_smem_kernel<2, true>, build_smem_kernel<3, true>, build_smem_kernel<4, true>,
    build_smem_kernel<5, true>, build_smem_kernel<6, true>, build_smem_kernel<7, true>, build_smem_kernel<8, true>};
static void (*const apply_smem_kernels[2][8])(ApplyArgs) = {
    {apply_smem_kernel<1, false>, apply_smem_kernel<2, false>, apply_smem_kernel<3, false>, apply_smem_kernel<4, false>,
     apply_smem_kernel<5, false>, apply_smem_kernel<6, false>, apply_smem_kernel<7, false>, apply_smem_kernel<8, false>},
    {apply_smem_kernel<1, true>, apply_smem_kernel<2, true>, apply_smem_kernel<3, true>, apply_smem_kernel<4, true>,
     apply_smem_kernel<5, true>, apply_smem_kernel<6, true>, apply_smem_kernel<7, true>, apply_smem_kernel<8, true>}};

template <class Args>
static int launch_smem(void (*kern)(Args), const Args &a, int grid, cudaStream_t st) {
    KBBQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, a.sl.total));
    kern<<<grid, a.g.threads + 32 * a.g.nprod, a.sl.total, st>>>(a);  // + the producer warp(s)
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

// What kbbq_build (narr 3) and kbbq_apply (narr 2) share once their arguments are checked: the shared-memory plan,
// or, when there is none, the generic kernel over the whole batch; then the prepare pass of the shared-memory kernel.
// generic(r0, n, grid) enqueues the generic kernel over reads [r0, r0 + n).  seg_rows != NULL: a segmented batch of
// at most N rows (segment.cuh).  On return p->smem says whether the shared-memory kernel is to take reads [0, p->N).
struct SmemPlan {
    Geom g;
    TableCfg tc;
    StageLayout sl;
    Workspace w;
    int sms;
    int64_t N;
    bool smem;
};

template <class Generic>
static int plan_and_prepare(int narr, bool aligned, int64_t N, int L, int R, int minscore, const uint16_t *rg,
                            const uint8_t *second, void *workspace, size_t workspace_bytes, int *status, int path,
                            const unsigned int *seg_rows, cudaStream_t st, const Generic &generic, SmemPlan *p) {
    const bool segmode = seg_rows != nullptr;
    int device, max_smem;
    int rc = current_device_info(&device, &p->sms, &max_smem);
    if (rc) return rc;
    p->smem = path != 2 && aligned && plan_kernel(L, R, minscore, narr, max_smem, &p->g, &p->tc, &p->sl, segmode) &&
              (uint64_t)((N + p->g.G - 1) / p->g.G) < 0xFFFFFFFFull;
    if (!p->smem) {
        if (path == 1 || segmode) return KBBQ_E_ARG;
        return generic(0, N, p->sms * 8);
    }
    p->w = carve_workspace(workspace, N, L, R);
    if (!workspace || workspace_bytes < p->w.bytes) return KBBQ_E_WORKSPACE;
    p->N = N;
    if (segmode) {
        seg_prepare_kernel<<<1, 256, 0, st>>>(seg_rows, 2 * R, p->g.G, (unsigned long long)N, p->w.seg, p->w.uni, status);
        KBBQ_LAUNCHED();
        return KBBQ_OK;
    }
    // One read group: a partial last group would be the only one with untallied rows and cost the
    // whole batch its header-free fast path; its few reads go through the generic kernel instead.
    const int64_t tail = (R == 1 && N > p->g.G) ? N % p->g.G : 0;
    if (tail) {
        p->N = N - tail;
        rc = generic(p->N, tail, 1);
        if (rc) return rc;
    }
    return run_prepare(rg, second, p->N, p->g.G, R, p->w, status, p->sms, p->sl.ngs, p->g.gbytes, p->sl.slot, st);
}

// bam_canon_kernel / bam_uncanon_kernel: one thread per output word; 32-bit thread indices, so very large batches take
// several launches.  launch(grid, r0, wmax) enqueues the reads from r0 on.
template <class Launch>
static int launch_bam_chunks(long long N, int L, const Launch &launch) {
    const unsigned int wmax = (unsigned int)((3 + L + 3) >> 2);
    const long long per = std::max<long long>(1, (long long)(0x7FFFFFFFu / wmax) / 256 * 256);  // reads per launch
    for (long long r0 = 0; r0 < N; r0 += per) {
        const long long n = std::min<long long>(per, N - r0);
        launch((unsigned)((n * wmax + BAM_WARPS * 32 - 1) / (BAM_WARPS * 32)), r0, wmax);
        KBBQ_LAUNCHED();
    }
    return KBBQ_OK;
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

// kbbq_build / kbbq_build_segmented
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
    auto generic = [&](int64_t r0, int64_t n, int grid) {
        BuildGenericArgs a = {seq + r0 * L, qual + r0 * L, corr + r0 * L, rg ? rg + r0 : nullptr,
                              second ? second + r0 : nullptr, n, L, R, minscore,
                              (unsigned long long *)pos_errs, (unsigned long long *)pos_total,
                              (unsigned long long *)din_errs, (unsigned long long *)din_total, status};
        build_generic_kernel<<<grid, 256, 0, st>>>(a);
        KBBQ_LAUNCHED();
        return KBBQ_OK;
    };
    const bool aligned = !misaligned(seq, 16) && !misaligned(qual, 16) && !misaligned(corr, 16);
    SmemPlan p;
    int rc = plan_and_prepare(3, aligned, N, L, R, minscore, rg, second, workspace, workspace_bytes, status, path,
                              seg_rows, st, generic, &p);
    if (rc || !p.smem) return rc;

    BuildArgs a;
    a.seq = seq; a.qual = qual; a.corr = corr; a.total_bytes = p.N * L; a.g = p.g; a.t = p.tc; a.R = R;
    a.nsub = segmode ? 2 * R : R; a.segmode = segmode ? 1 : 0;
    a.sl = p.sl;
    a.entries = p.w.entries; a.seg = p.w.seg; a.uni = p.w.uni;
    a.pos_errs = (unsigned long long *)pos_errs; a.pos_total = (unsigned long long *)pos_total;
    a.din_errs = (unsigned long long *)din_errs; a.din_total = (unsigned long long *)din_total;
    a.status = status;
    return launch_smem(build_smem_kernels[a.sl.kps - 1], a, p.sms, st);
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
    int rc = upload_constants();
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
    int rc = upload_constants();
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
    int rc = upload_constants();
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
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const long long blocks = std::min<long long>(((long long)N * L + 255) / 256, (long long)sms * 16);
    if (workspace && minscore >= 1) {  // canonical form + the shared-memory build kernel
        BamWorkspace w = carve_bam_workspace(workspace, N, L, R);
        if (workspace_bytes < w.bytes) return KBBQ_E_WORKSPACE;
        BamCanonArgs c = {seq, qual, err, skip, rg, flags, aln_start, aln_end, N, L, R, minscore, NQ, true,
                          w.cseq, w.cqual, w.cthird, w.csecond,
                          (unsigned long long *)pos_errs, (unsigned long long *)pos_total,
                          (unsigned long long *)din_errs, (unsigned long long *)din_total, status};
        rc = launch_bam_chunks(N, L, [&](unsigned grid, long long r0, unsigned wmax) {
            bam_canon_kernel<<<grid, BAM_WARPS * 32, 0, st>>>(c, r0, wmax);
        });
        if (rc) return rc;
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
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const long long blocks = std::min<long long>(((long long)N * L + 255) / 256, (long long)sms * 16);
    if (workspace && minscore >= 1 && nq <= NQ) {  // canonical form + the shared-memory apply kernel + flip back
        BamWorkspace w = carve_bam_workspace(workspace, N, L, R);
        if (workspace_bytes < w.bytes) return KBBQ_E_WORKSPACE;
        BamCanonArgs c = {seq, qual, nullptr, nullptr, rg, flags, nullptr, nullptr, N, L, R, minscore, nq, false,
                          w.cseq, w.cqual, nullptr, w.csecond, nullptr, nullptr, nullptr, nullptr, status};
        rc = launch_bam_chunks(N, L, [&](unsigned grid, long long r0, unsigned wmax) {
            bam_canon_kernel<<<grid, BAM_WARPS * 32, 0, st>>>(c, r0, wmax);
        });
        if (rc) return rc;
        // the canonical reads hold A, C, G, T, N only: bam_canon_kernel has already applied the reference's rule
        rc = kbbq_apply(w.cseq, w.cqual, rg, w.csecond, N, L, R, minscore, meanq, rgdq, qdq, posdq, dindq, nq, ndin1,
                        w.cthird, w.inner, w.inner_bytes, status, KBBQ_APPLY_BASES_CHECKED, stream);
        if (rc) return rc;
        return launch_bam_chunks(N, L, [&](unsigned grid, long long r0, unsigned wmax) {
            bam_uncanon_kernel<<<grid, BAM_WARPS * 32, 0, st>>>(w.cthird, flags, N, L, out_qual, r0, wmax);
        });
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
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
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
    int rc = upload_constants();
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
    Workspace w = carve_workspace(workspace, N, L, R);
    if (!workspace || workspace_bytes < w.bytes) return KBBQ_E_WORKSPACE;

    const long long fold_cells = (long long)R * NQ * (2 * L + 16);
    fold_kernel<<<(unsigned)((fold_cells + 255) / 256), 256, 0, st>>>(
        (const long long *)meanq, (const long long *)rgdq, (const long long *)qdq, (const long long *)posdq,
        (const long long *)dindq, R, nq, 2 * L, ndin1, w.fold_cyc, w.fold_din);
    KBBQ_LAUNCHED();

    auto generic = [&](int64_t r0, int64_t n, int grid) {
        ApplyGenericArgs a = {seq + r0 * L, qual + r0 * L, rg ? rg + r0 : nullptr, second ? second + r0 : nullptr,
                              out_qual + r0 * L, n, L, R, minscore, nq, w.fold_cyc, w.fold_din, status, validate};
        apply_generic_kernel<<<grid, 256, 0, st>>>(a);
        KBBQ_LAUNCHED();
        return KBBQ_OK;
    };
    const bool aligned = !misaligned(seq, 16) && !misaligned(qual, 16) && !misaligned(out_qual, 4);
    SmemPlan p;
    int rc = plan_and_prepare(2, aligned, N, L, R, minscore, rg, second, workspace, workspace_bytes, status, path,
                              seg_rows, st, generic, &p);
    if (rc || !p.smem) return rc;

    ApplyArgs a;
    a.nsub = segmode ? 2 * R : R; a.segmode = segmode ? 1 : 0;
    a.seq = seq; a.qual = qual; a.out = out_qual; a.total_bytes = p.N * L; a.g = p.g; a.t = p.tc; a.R = R; a.nq = nq;
    a.sl = p.sl;
    a.entries = w.entries; a.seg = w.seg; a.uni = w.uni; a.fold_cyc = w.fold_cyc; a.fold_din = w.fold_din; a.status = status;
    return launch_smem(apply_smem_kernels[validate][a.sl.kps - 1], a, p.sms, st);
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

// ---- k-mer errors (kmer.cuh) ----

static bool kmer_table_ok(const void *table, uint64_t capacity) {
    return table && !misaligned(table, 16) && capacity >= 1 && (capacity & (capacity - 1)) == 0;
}

// the default capacity: the smallest power of two >= 1.5 x windows; 0 when that is past 2^59
static uint64_t kmer_exact_capacity(uint64_t windows) {
    const uint64_t need = windows + (windows + 1) / 2;   // ceil(1.5 x windows)
    if (need > (1ull << 59)) return 0;
    uint64_t cap = 1;
    while (cap < need) cap <<= 1;
    return cap;
}

int kbbq_kmer_table_bytes(int64_t N, int L, int k, uint64_t *capacity, size_t *bytes) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || !capacity) return KBBQ_E_ARG;
    const uint64_t cap = kmer_exact_capacity((uint64_t)N * (uint64_t)std::max(0, L - k + 1));
    if (!cap) return KBBQ_E_ARG;
    *capacity = cap;
    if (bytes) *bytes = (size_t)(cap * 16);
    return KBBQ_OK;
}

int kbbq_kmer_clear(void *table, uint64_t capacity, void *stream) {
    if (!kmer_table_ok(table, capacity)) return KBBQ_E_ARG;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    const uint64_t blocks = std::min<uint64_t>((capacity + 255) / 256, (uint64_t)sms * 16);
    kmer_clear_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((ulonglong2 *)table, capacity);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_kmer_count(const uint8_t *seq, int64_t N, int L, int k, void *table, uint64_t capacity, int *status,
                    void *stream) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || !status || !kmer_table_ok(table, capacity)) return KBBQ_E_ARG;
    if (N == 0 || L < k) return KBBQ_OK;
    if (!seq) return KBBQ_E_ARG;
    kmer_count_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        seq, N, L, k, (unsigned long long *)table, capacity - 1, status);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_kmer_histogram(const void *table, uint64_t capacity, uint64_t *hist, void *stream) {
    if (!kmer_table_ok(table, capacity) || !hist) return KBBQ_E_ARG;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    KBBQ_CUDA(cudaMemsetAsync(hist, 0, 256 * sizeof(uint64_t), (cudaStream_t)stream));
    const uint64_t blocks = std::min<uint64_t>((capacity + 255) / 256, (uint64_t)sms * 8);
    kmer_hist_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const ulonglong2 *)table, capacity,
                                                                         (unsigned long long *)hist);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_kmer_flag(const uint8_t *seq, int64_t N, int L, int k, const void *table, uint64_t capacity, int min_count,
                   uint32_t *bits, int *status, void *stream) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || min_count < 1 || !status || !kmer_table_ok(table, capacity))
        return KBBQ_E_ARG;
    if (N == 0) return KBBQ_OK;
    if (!seq || !bits) return KBBQ_E_ARG;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    // a warp assembles the L words of its 32 reads in shared memory: 4 warps a block while that stays under 48 KB
    const int warps = std::max(1, std::min(4, 49152 / (4 * L)));
    const size_t smem = (size_t)warps * L * 4;
    if (smem > (size_t)max_smem) return KBBQ_E_ARG;
    if (smem > 49152) KBBQ_CUDA(cudaFuncSetAttribute(kmer_flag_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t blocks = (N + 32 * warps - 1) / (32 * warps);
    kmer_flag_kernel<false><<<(unsigned)blocks, 32 * warps, smem, (cudaStream_t)stream>>>(
        seq, N, L, k, (const ulonglong2 *)table, capacity - 1, (unsigned long long)min_count, bits, status);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_kmer_min_count(const uint64_t *hist) {
    if (!hist) return KBBQ_E_ARG;
    for (int c = 2; c <= 254; ++c)
        if (hist[c] <= hist[c + 1]) return c;
    return 255;
}

// ---- the sieved table (kmer.cuh, DESIGN.md §10 "Streaming") ----

static bool pow2(uint64_t x) { return x >= 1 && (x & (x - 1)) == 0; }

int kbbq_kmer_stream_plan(uint64_t windows, uint64_t budget_bytes, uint64_t *filter_words, uint64_t *capacity) {
    if (!filter_words || !capacity) return KBBQ_E_ARG;
    const uint64_t exact = kmer_exact_capacity(windows);
    if (!exact) return KBBQ_E_ARG;
    // filter: the largest power of two with 8 F <= min(W, budget / 4) bytes (one byte per window), at least one word
    const uint64_t fbytes = std::min(windows, budget_bytes / 4);
    uint64_t F = 1;
    while (F <= (1ull << 40) && 16 * F <= fbytes) F <<= 1;
    // table: the exact rule's capacity, or the largest power of two that fits what the filter leaves
    const uint64_t min_cap = std::min<uint64_t>(exact, KBBQ_KMER_MIN_SLOTS);
    if (budget_bytes < 8 * F || (budget_bytes - 8 * F) / 16 < min_cap) return KBBQ_E_UNSUPPORTED;
    const uint64_t slots = (budget_bytes - 8 * F) / 16;
    uint64_t cap = min_cap;
    while (cap < exact && 2 * cap <= slots) cap <<= 1;
    *filter_words = F;
    *capacity = cap;
    return KBBQ_OK;
}

int kbbq_kmer_sieve(const uint8_t *seq, int64_t N, int L, int k, void *filter, uint64_t filter_words, void *table,
                    uint64_t capacity, int *status, void *stream) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || !status || !kmer_table_ok(table, capacity) || !filter ||
        misaligned(filter, 8) || !pow2(filter_words))
        return KBBQ_E_ARG;
    if (N == 0 || L < k) return KBBQ_OK;
    if (!seq) return KBBQ_E_ARG;
    kmer_sieve_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        seq, N, L, k, (unsigned long long *)filter, filter_words - 1, (unsigned long long *)table, capacity - 1, status);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_kmer_count_present(const uint8_t *seq, int64_t N, int L, int k, void *table, uint64_t capacity,
                            uint64_t *windows, int *status, void *stream) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || !status || !windows || misaligned(windows, 8) ||
        !kmer_table_ok(table, capacity))
        return KBBQ_E_ARG;
    if (N == 0 || L < k) return KBBQ_OK;
    if (!seq) return KBBQ_E_ARG;
    kmer_count_present_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        seq, N, L, k, (unsigned long long *)table, capacity - 1, (unsigned long long *)windows, status);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_kmer_histogram_sieved(const void *table, uint64_t capacity, const uint64_t *windows, uint64_t *hist,
                               void *stream) {
    if (!kmer_table_ok(table, capacity) || !hist || !windows || misaligned(windows, 8)) return KBBQ_E_ARG;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    KBBQ_CUDA(cudaMemsetAsync(hist, 0, 256 * sizeof(uint64_t), st));
    const uint64_t blocks = std::min<uint64_t>((capacity + 255) / 256, (uint64_t)sms * 8);
    kmer_hist_sieved_kernel<<<(unsigned)blocks, 256, 0, st>>>((const ulonglong2 *)table, capacity,
                                                              (unsigned long long *)hist);
    KBBQ_LAUNCHED();
    kmer_hist_tail_kernel<<<1, 1, 0, st>>>((const unsigned long long *)windows, (unsigned long long *)hist);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

int kbbq_kmer_flag_sieved(const uint8_t *seq, int64_t N, int L, int k, const void *table, uint64_t capacity,
                          int min_count, uint32_t *bits, int *status, void *stream) {
    if (min_count != 1) return kbbq_kmer_flag(seq, N, L, k, table, capacity, min_count, bits, status, stream);
    if (N < 0 || L < 1 || k < 1 || k > 31 || !status || !kmer_table_ok(table, capacity)) return KBBQ_E_ARG;
    if (N == 0) return KBBQ_OK;
    if (!seq || !bits) return KBBQ_E_ARG;
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    const int warps = std::max(1, std::min(4, 49152 / (4 * L)));   // as kbbq_kmer_flag
    const size_t smem = (size_t)warps * L * 4;
    if (smem > (size_t)max_smem) return KBBQ_E_ARG;
    if (smem > 49152) KBBQ_CUDA(cudaFuncSetAttribute(kmer_flag_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t blocks = (N + 32 * warps - 1) / (32 * warps);
    kmer_flag_kernel<true><<<(unsigned)blocks, 32 * warps, smem, (cudaStream_t)stream>>>(
        seq, N, L, k, (const ulonglong2 *)table, capacity - 1, 1ull, bits, status);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

// ---- the correcting walk (kmer.cuh, DESIGN.md §10 "The correcting walk") ----

int kbbq_kmer_correct(const uint8_t *seq, int64_t N, int L, int k, const void *table, uint64_t capacity, int min_count,
                      uint32_t *bits, int *status, void *stream) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || min_count < 1 || !status || !kmer_table_ok(table, capacity))
        return KBBQ_E_ARG;
    if (N == 0) return KBBQ_OK;
    if (!seq || !bits) return KBBQ_E_ARG;
    if (min_count == 1) {   // every valid window is solid: nothing is flagged
        KBBQ_CUDA(cudaMemsetAsync(bits, 0, ((size_t)N * L + 31) / 32 * 4, (cudaStream_t)stream));
        return KBBQ_OK;
    }
    int device, sms, max_smem;
    int rc = current_device_info(&device, &sms, &max_smem);
    if (rc) return rc;
    // a warp's map words and its reads' solid bits: 4 warps a block while that stays under 48 KB
    const int words = kmer_correct_warp_words(L, k);
    const int warps = std::max(1, std::min(4, 49152 / (4 * words)));
    const size_t smem = (size_t)warps * words * 4;
    if (smem > (size_t)max_smem) return KBBQ_E_ARG;
    if (smem > 49152) KBBQ_CUDA(cudaFuncSetAttribute(kmer_correct_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t blocks = (N + 32 * warps - 1) / (32 * warps);
    kmer_correct_kernel<<<(unsigned)blocks, 32 * warps, smem, (cudaStream_t)stream>>>(
        seq, N, L, k, (const ulonglong2 *)table, capacity - 1, (unsigned long long)min_count, bits, status);
    KBBQ_LAUNCHED();
    return KBBQ_OK;
}

}  // extern "C"
