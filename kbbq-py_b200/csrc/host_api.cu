// host_api.cu -- host-buffer side of the C ABI: sessions, the whole-path entry points, several GPUs.
//
// What recalibrate.recalibrate_fastq (kbbq/recalibrate.py:123-156) does between parsing and printing is two
// passes over the reads around one small model step.  A SESSION is that path on one device, fed chunk by
// chunk from host memory:
//
//     kbbq_session_build_chunk  x n     H2D (seq, qual, 1-bit mismatch map) -> [segment rows] -> build   pass 1
//     (tables may be summed with other sessions / ranks here: they are additive integers)
//     kbbq_session_model                marginals + delta tables
//     kbbq_session_apply_*      x n     [H2D] -> apply -> [unsegment] -> D2H                              pass 2
//
// Three streams (upload, compute, download) and two staging slots per direction keep the copy engines and the
// SMs busy together; chunks can stay resident in HBM between the passes (segmented when there are several read
// groups, segment.cuh) or be sent again (files larger than the device).  kbbq_recalibrate_host is one session
// over one buffer, kbbq_recalibrate_host_multi one session per device on its own host thread with the partial
// tables summed over NVLink peer memory (one kernel per device reads every peer's table and writes the sum),
// through pinned host memory when the devices cannot reach each other.  Every kernel launched here goes through
// the device-pointer entry points of kbbq_b200.cu.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <sched.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <fcntl.h>
#include <thread>
#include <unistd.h>
#include <vector>

#include "common.cuh"

using namespace kbbq;

namespace {

#define KBBQ_TRY(x) do { int rc_ = (x); if (rc_) return rc_; } while (0)

constexpr int MAX_DEVICES = 16;

struct Carver {  // bump allocator over one allocation (first pass with base == nullptr measures)
    char *base;
    size_t off = 0;
    explicit Carver(void *b) : base((char *)b) {}
    template <class T> T *take(size_t n_elems) {
        T *p = base ? (T *)(base + off) : nullptr;
        off = (off + n_elems * sizeof(T) + 255) / 256 * 256;
        return p;
    }
};

// [q_errs R*43 | q_total R*43 | rg_errs R | rg_total R | meanq R | rgdq R | qdq R*43 | posdq R*43*2L | dindq R*43*17]
struct ModelPtrs {
    int64_t *q_errs, *q_total, *rg_errs, *rg_total, *meanq, *rgdq, *qdq, *posdq, *dindq;
    size_t elems;
};
ModelPtrs carve_model(int64_t *base, int L, int R) {
    ModelPtrs m;
    size_t o = 0;
    m.q_errs = base + o; o += (size_t)R * NQ;
    m.q_total = base + o; o += (size_t)R * NQ;
    m.rg_errs = base + o; o += R;
    m.rg_total = base + o; o += R;
    m.meanq = base + o; o += R;
    m.rgdq = base + o; o += R;
    m.qdq = base + o; o += (size_t)R * NQ;
    m.posdq = base + o; o += (size_t)R * NQ * 2 * L;
    m.dindq = base + o; o += (size_t)R * NQ * 17;
    m.elems = o;
    return m;
}

struct PeerTables {
    const long long *src[MAX_DEVICES];
};

// out[i] = sum over the n tables; src[k] may live on a peer device (NVLink loads)
__global__ void sum_tables_kernel(PeerTables p, int n, long long *out, size_t elems) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < elems; i += (size_t)gridDim.x * blockDim.x) {
        long long v = 0;
        for (int k = 0; k < n; ++k) v += p.src[k][i];
        out[i] = v;
    }
}

enum { PACK_NONE = 0, PACK_BITS = 1, PACK_NIBBLES = 2 };

struct UpSlot {   // one upload in flight: the chunk as the host has it (read order)
    uint8_t *seq = nullptr, *qual = nullptr, *corr = nullptr, *sec = nullptr;
    uint16_t *rg = nullptr;
    uint32_t *bits = nullptr;     // PACK_BITS: 1 bit per base; PACK_NIBBLES: 4 bits per base
    // streaming sessions with several read groups: the segmented copy of the chunk
    uint8_t *sseq = nullptr, *squal = nullptr, *scorr = nullptr;
    uint32_t *seg = nullptr, *dest = nullptr;
    uint32_t *h_bits = nullptr;   // pinned
    cudaEvent_t uploaded = nullptr, consumed = nullptr;
};

struct Resident {  // a chunk kept in HBM between the passes
    uint8_t *seq = nullptr, *qual = nullptr, *sec = nullptr;
    uint16_t *rg = nullptr;
    uint32_t *seg = nullptr, *dest = nullptr;
    int64_t n = 0;
};

struct OutSlot {
    uint8_t *out = nullptr, *out_seg = nullptr;
    cudaEvent_t applied = nullptr, drained = nullptr;
};

}  // namespace

struct kbbq_session {
    int device = 0, L = 0, R = 1, minscore = 6;
    int64_t C = 0;          // reads per chunk (capacity)
    int64_t M = 0;          // reads that can stay resident (0: streaming session)
    int64_t rowsC = 0;      // rows of a chunk in the segmented layout
    bool segmode = false;
    int pack = PACK_NIBBLES;   // how the reads and the corrected reads cross PCIe (PACK_*)
    int host_status = 0;       // KBBQ_FLAG_* found by the host-side packer
    int host_threads = 0;
    void *base = nullptr;
    size_t cap = 0;
    void *pinned = nullptr;
    cudaStream_t s_up = nullptr, s_comp = nullptr, s_down = nullptr;
    int64_t *d_tab = nullptr, *d_sum = nullptr, *d_model = nullptr;
    int *d_status = nullptr;
    void *d_ws = nullptr;
    size_t ws_bytes = 0, ntab = 0;
    ModelPtrs mp;
    UpSlot up[2];
    OutSlot down[2];
    std::vector<Resident> res;
    int64_t built = 0, applied = 0;
    bool summed = false;    // the model reads d_sum (tables of several sessions added up) instead of d_tab
    int64_t h2d_bytes = 0, d2h_bytes = 0;
    std::mutex mu;

    ~kbbq_session() {
        cudaSetDevice(device);
        for (auto s : {s_up, s_comp, s_down}) if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
        for (auto &u : up) { if (u.uploaded) cudaEventDestroy(u.uploaded); if (u.consumed) cudaEventDestroy(u.consumed); }
        for (auto &o : down) { if (o.applied) cudaEventDestroy(o.applied); if (o.drained) cudaEventDestroy(o.drained); }
        if (base) cudaFree(base);
        if (pinned) cudaFreeHost(pinned);
    }
};

namespace {

int64_t default_chunk_reads(int L) {
    int64_t chunk = std::max<int64_t>(1, ((int64_t)256 << 20) / L);   // ~256 MiB per array per chunk
    if (const char *e = getenv("KBBQ_HOST_CHUNK_READS")) chunk = std::max<int64_t>(16, atoll(e));  // test hook
    return (chunk + 15) / 16 * 16;                                    // chunk starts stay 16-byte aligned
}

bool env_flag_off(const char *name) {   // unset or "0"
    const char *e = getenv(name);
    return !e || atoi(e) == 0;
}

int usable_cpus() {
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof(set), &set) == 0) return std::max(1, CPU_COUNT(&set));
    return std::max(1, (int)std::thread::hardware_concurrency());
}

// What crosses PCIe in pass 1, per base (the reference only ever compares the corrected reads with the reads,
// find_corrected_sites, kbbq/recalibrate.py:13-20):
//   PACK_NIBBLES  qual as it is + 4 bits (base code | mismatch) made by the host cores while the copy engine moves
//                 the qualities (host_pack.cpp): 1.5 B instead of 3;
//   PACK_BITS     seq + qual as they are + a 1-bit mismatch map: 2.125 B;
//   PACK_NONE     seq + qual + corrected reads: 3 B, no host work.
// Packing reads 2 B per base of host memory, so it only pays when this session has the cores for it: with fewer
// than 8 threads (an 8-GPU box shares 32 cores, and its host memory, between 8 sessions) it takes longer than the
// bytes it saves (B200 x 8: 389 ms per step with the bit map, 343 ms with the corrected reads as they are; 4 GPUs,
// 8 threads each: map).  KBBQ_HOST_NO_BITMAP=1 forces PACK_NONE, KBBQ_HOST_BITMAP=1 packing whatever the core
// count, KBBQ_HOST_NO_NIBBLES=1 the bit map instead of the nibbles.
int pack_mode(int host_threads) {
    if (!env_flag_off("KBBQ_HOST_NO_BITMAP")) return PACK_NONE;
    const int packed = env_flag_off("KBBQ_HOST_NO_NIBBLES") ? PACK_NIBBLES : PACK_BITS;
    if (!env_flag_off("KBBQ_HOST_BITMAP")) return packed;
    return (host_threads > 0 ? host_threads : usable_cpus()) >= 8 ? packed : PACK_NONE;
}

// several read groups: chunks are rewritten into the segmented layout on the device (segment.cuh) unless the
// shape has no shared-memory plan or the padding (32 R rows per chunk) would rival the chunk itself
bool want_segmode(int L, int R, int minscore, int64_t C) {
    return R > 1 && kbbq_segmented_supported(L, R, minscore) && (int64_t)32 * R * 8 <= C && env_flag_off("KBBQ_HOST_NO_SEGMENT");
}

// pack < 0: the transport follows from the host threads this session has (pack_mode)
int session_create(int device, int L, int R, int minscore, int64_t C, int64_t M, int host_threads, int pack, kbbq_session **out) {
    if (device < 0 || L < 1 || R < 1 || R > 65535 || minscore < 0 || minscore >= NQ || C < 1 || M < 0 || !out)
        return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(device));
    std::unique_ptr<kbbq_session> S(new kbbq_session);
    S->device = device; S->L = L; S->R = R; S->minscore = minscore;
    S->C = (C + 15) / 16 * 16;
    S->M = M;
    S->host_threads = host_threads;
    S->pack = pack < 0 ? pack_mode(host_threads) : pack;
    S->segmode = want_segmode(L, R, minscore, S->C);
    S->rowsC = S->segmode ? kbbq_segment_rows_bound(S->C, R) : S->C;
    KBBQ_CUDA(cudaStreamCreateWithFlags(&S->s_up, cudaStreamNonBlocking));
    KBBQ_CUDA(cudaStreamCreateWithFlags(&S->s_comp, cudaStreamNonBlocking));
    KBBQ_CUDA(cudaStreamCreateWithFlags(&S->s_down, cudaStreamNonBlocking));
    for (auto &u : S->up) {
        KBBQ_CUDA(cudaEventCreateWithFlags(&u.uploaded, cudaEventDisableTiming));
        KBBQ_CUDA(cudaEventCreateWithFlags(&u.consumed, cudaEventDisableTiming));
    }
    for (auto &o : S->down) {
        KBBQ_CUDA(cudaEventCreateWithFlags(&o.applied, cudaEventDisableTiming));
        KBBQ_CUDA(cudaEventCreateWithFlags(&o.drained, cudaEventDisableTiming));
    }
    const size_t npos = (size_t)R * NQ * 2 * L, ndin = (size_t)R * NQ * 16;
    S->ntab = 2 * npos + 2 * ndin;
    const size_t nmodel = carve_model(nullptr, L, R).elems;
    KBBQ_TRY(kbbq_workspace_bytes(S->rowsC, L, R, &S->ws_bytes));
    const size_t cb = (size_t)S->C * L + 16, rb = (size_t)S->rowsC * L + 16;
    // words of the packed form of a chunk: 1 bit or 4 bits per base
    const size_t bits_words = S->pack == PACK_NIBBLES ? ((size_t)S->C * L + 7) / 8 + 4 : ((size_t)S->C * L + 31) / 32 + 4;
    const size_t seg_elems = (size_t)kbbq_segment_table_elems(R);
    const int64_t nres = M ? (M + S->C - 1) / S->C : 0;
    const bool seg = S->segmode, stream_seg = seg && nres == 0;
    S->res.resize((size_t)nres);
    for (int pass = 0; pass < 2; ++pass) {
        Carver c(pass ? S->base : nullptr);
        S->d_tab = c.take<int64_t>(S->ntab);
        S->d_sum = c.take<int64_t>(S->ntab);
        S->d_model = c.take<int64_t>(nmodel);
        S->d_status = c.take<int>(64);
        S->d_ws = c.take<uint8_t>(S->ws_bytes);
        for (auto &u : S->up) {
            // resident chunks of a plain batch are uploaded straight into their place: no staging copy of seq / qual
            const bool staged = seg || nres == 0;
            u.seq = staged ? c.take<uint8_t>(cb) : nullptr;
            u.qual = staged ? c.take<uint8_t>(cb) : nullptr;
            u.rg = staged ? c.take<uint16_t>((size_t)S->C + 8) : nullptr;
            u.sec = staged ? c.take<uint8_t>((size_t)S->C + 16) : nullptr;
            u.corr = c.take<uint8_t>(cb);
            u.bits = S->pack ? c.take<uint32_t>(bits_words) : nullptr;
            u.scorr = seg ? c.take<uint8_t>(rb) : nullptr;
            u.sseq = stream_seg ? c.take<uint8_t>(rb) : nullptr;
            u.squal = stream_seg ? c.take<uint8_t>(rb) : nullptr;
            u.seg = stream_seg ? c.take<uint32_t>(seg_elems) : nullptr;
            u.dest = stream_seg ? c.take<uint32_t>((size_t)S->C) : nullptr;
        }
        for (auto &o : S->down) {
            o.out = c.take<uint8_t>(cb);
            o.out_seg = seg ? c.take<uint8_t>(rb) : nullptr;
        }
        for (auto &r : S->res) {
            r.seq = c.take<uint8_t>(seg ? rb : cb);
            r.qual = c.take<uint8_t>(seg ? rb : cb);
            r.rg = seg ? nullptr : c.take<uint16_t>((size_t)S->C + 8);
            r.sec = seg ? nullptr : c.take<uint8_t>((size_t)S->C + 16);
            r.seg = seg ? c.take<uint32_t>(seg_elems) : nullptr;
            r.dest = seg ? c.take<uint32_t>((size_t)S->C) : nullptr;
        }
        if (!pass) {
            S->cap = c.off;
            KBBQ_CUDA(cudaMalloc(&S->base, S->cap));
        }
    }
    S->mp = carve_model(S->d_model, L, R);
    if (S->pack) {
        KBBQ_CUDA(cudaHostAlloc(&S->pinned, 2 * bits_words * 4, cudaHostAllocDefault));
        S->up[0].h_bits = (uint32_t *)S->pinned;
        S->up[1].h_bits = (uint32_t *)S->pinned + bits_words;
    }
    KBBQ_CUDA(cudaMemsetAsync(S->d_tab, 0, S->ntab * 8, S->s_comp));
    KBBQ_CUDA(cudaMemsetAsync(S->d_status, 0, 64 * sizeof(int), S->s_comp));
    *out = S.release();
    return KBBQ_OK;
}

// Forget the tables and chunks of the previous run (the device memory stays).
int session_reset(kbbq_session *S) {
    KBBQ_CUDA(cudaSetDevice(S->device));
    KBBQ_CUDA(cudaStreamSynchronize(S->s_up));
    KBBQ_CUDA(cudaStreamSynchronize(S->s_down));
    KBBQ_CUDA(cudaMemsetAsync(S->d_tab, 0, S->ntab * 8, S->s_comp));
    KBBQ_CUDA(cudaMemsetAsync(S->d_status, 0, sizeof(int), S->s_comp));
    S->built = S->applied = 0;
    S->host_status = 0;
    S->summed = false;
    S->h2d_bytes = S->d2h_bytes = 0;
    for (auto &r : S->res) r.n = 0;
    return KBBQ_OK;
}

int upload_reads(kbbq_session *S, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second,
                 int64_t n, uint8_t *d_seq, uint8_t *d_qual, uint16_t *d_rg, uint8_t *d_sec) {
    const size_t nb = (size_t)n * S->L;
    if (seq) { KBBQ_CUDA(cudaMemcpyAsync(d_seq, seq, nb, cudaMemcpyHostToDevice, S->s_up)); S->h2d_bytes += (int64_t)nb; }
    KBBQ_CUDA(cudaMemcpyAsync(d_qual, qual, nb, cudaMemcpyHostToDevice, S->s_up));
    S->h2d_bytes += (int64_t)nb;
    if (rg) { KBBQ_CUDA(cudaMemcpyAsync(d_rg, rg, (size_t)n * 2, cudaMemcpyHostToDevice, S->s_up)); S->h2d_bytes += 2 * n; }
    if (second) { KBBQ_CUDA(cudaMemcpyAsync(d_sec, second, (size_t)n, cudaMemcpyHostToDevice, S->s_up)); S->h2d_bytes += n; }
    return KBBQ_OK;
}

// Where chunk k of pass 1 lives on the device.  keep: it stays in HBM for kbbq_session_apply_resident; a plain
// (one read group) resident chunk is uploaded / expanded straight into its place, no staging copy.
struct ChunkPlace {
    UpSlot *u;
    Resident *r;
    uint8_t *d_seq, *d_qual, *d_sec;
    uint16_t *d_rg;
};
ChunkPlace chunk_place(kbbq_session *S, int64_t k, bool keep, bool has_rg, bool has_second) {
    ChunkPlace p;
    p.u = &S->up[k & 1];
    p.r = keep ? &S->res[(size_t)k] : nullptr;
    const bool direct = keep && !S->segmode;
    p.d_seq = direct ? p.r->seq : p.u->seq;
    p.d_qual = direct ? p.r->qual : p.u->qual;
    p.d_rg = has_rg ? (direct ? p.r->rg : p.u->rg) : nullptr;
    p.d_sec = has_second ? (direct ? p.r->sec : p.u->sec) : nullptr;
    return p;
}

bool chunk_args_ok(const kbbq_session *S, int64_t k, int64_t n, bool keep) {
    return n > 0 && n <= S->C && (!keep || k < (int64_t)S->res.size());
}

// Pass 1 of chunk k, first half: enqueue the copies that come straight from the caller's memory (the qualities,
// read groups and mate flags; the reads too unless they travel as nibbles).  Nothing waits for the device.
int build_chunk_upload(kbbq_session *S, int64_t k, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg,
                       const uint8_t *second, int64_t n, bool keep) {
    if (!chunk_args_ok(S, k, n, keep) || !seq || !qual) return KBBQ_E_ARG;
    const ChunkPlace p = chunk_place(S, k, keep, rg != nullptr, second != nullptr);
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_up, p.u->consumed, 0));   // the slot's previous chunk has been built
    return upload_reads(S, S->pack == PACK_NIBBLES ? nullptr : seq, qual, rg, second, n, p.d_seq, p.d_qual, p.d_rg, p.d_sec);
}

// Second half: the host cores pack (seq, corrected) of the chunk while the copy engine is busy with what
// build_chunk_upload queued (of this chunk and, in run_build_pass, of the next one too), the packed form follows,
// and the compute stream expands it, segments the rows when there are several read groups, and builds.  The only
// wait is for the pinned packing slot (two chunks back).
int build_chunk_finish(kbbq_session *S, int64_t k, const uint8_t *seq, const uint8_t *corr, bool has_rg, bool has_second,
                       int64_t n, bool keep) {
    if (!chunk_args_ok(S, k, n, keep) || !seq || !corr) return KBBQ_E_ARG;
    const ChunkPlace p = chunk_place(S, k, keep, has_rg, has_second);
    UpSlot &u = *p.u;
    Resident *r = p.r;
    const int L = S->L, R = S->R;
    const size_t nb = (size_t)n * L;
    if (r) r->n = n;
    if (S->pack) {
        KBBQ_CUDA(cudaEventSynchronize(u.uploaded));           // the slot's packed chunk of two chunks back is on the device
        size_t bb;
        if (S->pack == PACK_NIBBLES) {
            int bad = 0;
            KBBQ_TRY(kbbq_host_pack_nibbles(seq, corr, (int64_t)nb, (uint8_t *)u.h_bits, S->host_threads, &bad));
            if (bad) S->host_status |= KBBQ_FLAG_BAD_BASE;
            bb = (nb + 1) / 2;
        } else {
            KBBQ_TRY(kbbq_host_mismatch_bits(seq, corr, (int64_t)nb, u.h_bits, S->host_threads));
            bb = ((nb + 31) / 32) * 4;
        }
        KBBQ_CUDA(cudaMemcpyAsync(u.bits, u.h_bits, bb, cudaMemcpyHostToDevice, S->s_up));
        S->h2d_bytes += (int64_t)bb;
    } else {
        KBBQ_CUDA(cudaMemcpyAsync(u.corr, corr, nb, cudaMemcpyHostToDevice, S->s_up));
        S->h2d_bytes += (int64_t)nb;
    }
    KBBQ_CUDA(cudaEventRecord(u.uploaded, S->s_up));
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_comp, u.uploaded, 0));
    if (S->pack == PACK_NIBBLES) KBBQ_TRY(kbbq_expand_nibbles((const uint8_t *)u.bits, (int64_t)nb, p.d_seq, u.corr, S->s_comp));
    else if (S->pack == PACK_BITS) KBBQ_TRY(kbbq_expand_mismatch_bits(p.d_seq, u.bits, (int64_t)nb, u.corr, S->s_comp));
    const size_t npos = (size_t)R * NQ * 2 * L, ndin = (size_t)R * NQ * 16;
    int64_t *pe = S->d_tab, *pt = pe + npos, *de = pt + npos, *dt = de + ndin;
    if (S->segmode) {
        uint32_t *seg = keep ? r->seg : u.seg, *dest = keep ? r->dest : u.dest;
        uint8_t *sseq = keep ? r->seq : u.sseq, *squal = keep ? r->qual : u.squal;
        KBBQ_TRY(kbbq_segment_plan(p.d_rg, p.d_sec, n, R, seg, dest, S->d_status, S->s_comp));
        KBBQ_TRY(kbbq_segment_rows(p.d_seq, dest, n, L, sseq, S->s_comp));
        KBBQ_TRY(kbbq_segment_rows(p.d_qual, dest, n, L, squal, S->s_comp));
        KBBQ_TRY(kbbq_segment_rows(u.corr, dest, n, L, u.scorr, S->s_comp));
        KBBQ_TRY(kbbq_segment_pad(seg, R, L, sseq, squal, u.scorr, S->s_comp));
        KBBQ_TRY(kbbq_build_segmented(sseq, squal, u.scorr, seg, S->rowsC, L, R, S->minscore, pe, pt, de, dt, S->d_ws,
                                      S->ws_bytes, S->d_status, S->s_comp));
    } else {
        KBBQ_TRY(kbbq_build(p.d_seq, p.d_qual, u.corr, p.d_rg, p.d_sec, n, L, R, S->minscore, pe, pt, de, dt, S->d_ws, S->ws_bytes,
                            S->d_status, 0, S->s_comp));
    }
    KBBQ_CUDA(cudaEventRecord(u.consumed, S->s_comp));
    return KBBQ_OK;
}

// Pass 1 of one chunk in one go.
int build_chunk_async(kbbq_session *S, const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
                      const uint8_t *second, int64_t n, bool keep) {
    if (n < 0 || n > S->C) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    if (!seq || !qual || !corr) return KBBQ_E_ARG;
    const int64_t k = S->built;
    if (keep && k >= (int64_t)S->res.size()) return KBBQ_E_ARG;
    S->built++;
    KBBQ_TRY(build_chunk_upload(S, k, seq, qual, rg, second, n, keep));
    return build_chunk_finish(S, k, seq, corr, rg != nullptr, second != nullptr, n, keep);
}

int model_async(kbbq_session *S) {
    const int L = S->L, R = S->R;
    const size_t npos = (size_t)R * NQ * 2 * L, ndin = (size_t)R * NQ * 16;
    int64_t *pe = S->summed ? S->d_sum : S->d_tab, *pt = pe + npos, *de = pt + npos, *dt = de + ndin;
    const ModelPtrs &mp = S->mp;
    KBBQ_TRY(kbbq_marginals(pe, pt, L, R, mp.q_errs, mp.q_total, mp.rg_errs, mp.rg_total, mp.meanq, S->s_comp));
    KBBQ_TRY(kbbq_get_delta_qs(mp.meanq, mp.rg_errs, mp.rg_total, mp.q_errs, mp.q_total, pe, pt, de, dt, R, NQ, 2 * L, 16,
                               mp.rgdq, mp.qdq, mp.posdq, mp.dindq, S->s_comp));
    return KBBQ_OK;
}

// apply + (unsegment) + D2H of one chunk that is on the device; the compute stream is positioned behind whatever
// put it there
int apply_and_download(kbbq_session *S, const uint8_t *d_seq, const uint8_t *d_qual, const uint16_t *d_rg,
                       const uint8_t *d_sec, const uint32_t *seg, const uint32_t *dest, int64_t n, uint8_t *out_host) {
    const int L = S->L, R = S->R;
    OutSlot &o = S->down[S->applied++ & 1];
    const ModelPtrs &mp = S->mp;
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_comp, o.drained, 0));   // the slot's previous chunk is in host memory
    if (S->segmode) {
        KBBQ_TRY(kbbq_apply_segmented(d_seq, d_qual, seg, S->rowsC, L, R, S->minscore, mp.meanq, mp.rgdq, mp.qdq, mp.posdq,
                                      mp.dindq, NQ, 17, o.out_seg, S->d_ws, S->ws_bytes, S->d_status, S->s_comp));
        KBBQ_TRY(kbbq_unsegment_rows(o.out_seg, dest, n, L, S->rowsC, o.out, S->s_comp));
    } else {
        KBBQ_TRY(kbbq_apply(d_seq, d_qual, d_rg, d_sec, n, L, R, S->minscore, mp.meanq, mp.rgdq, mp.qdq, mp.posdq, mp.dindq,
                            NQ, 17, o.out, S->d_ws, S->ws_bytes, S->d_status, 0, S->s_comp));
    }
    KBBQ_CUDA(cudaEventRecord(o.applied, S->s_comp));
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_down, o.applied, 0));
    KBBQ_CUDA(cudaMemcpyAsync(out_host, o.out, (size_t)n * L, cudaMemcpyDeviceToHost, S->s_down));
    S->d2h_bytes += n * L;
    KBBQ_CUDA(cudaEventRecord(o.drained, S->s_down));
    return KBBQ_OK;
}

int apply_resident_async(kbbq_session *S, int64_t k, uint8_t *out_host) {
    if (k < 0 || k >= (int64_t)S->res.size() || !out_host) return KBBQ_E_ARG;
    const Resident &r = S->res[(size_t)k];
    if (r.n == 0) return KBBQ_OK;
    return apply_and_download(S, r.seq, r.qual, r.rg, r.sec, r.seg, r.dest, r.n, out_host);
}

// pass 2 of a chunk that is not resident: the reads are sent again
int apply_chunk_async(kbbq_session *S, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second,
                      int64_t n, uint8_t *out_host) {
    if (n < 0 || n > S->C || !S->up[0].seq) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    if (!seq || !qual || !out_host) return KBBQ_E_ARG;
    UpSlot &u = S->up[S->applied & 1];
    const int L = S->L, R = S->R;
    uint16_t *d_rg = rg ? u.rg : nullptr;
    uint8_t *d_sec = second ? u.sec : nullptr;
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_up, u.consumed, 0));
    KBBQ_TRY(upload_reads(S, seq, qual, rg, second, n, u.seq, u.qual, d_rg, d_sec));
    KBBQ_CUDA(cudaEventRecord(u.uploaded, S->s_up));
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_comp, u.uploaded, 0));
    const uint8_t *a_seq = u.seq, *a_qual = u.qual;
    if (S->segmode) {
        uint8_t *sseq = u.sseq ? u.sseq : nullptr, *squal = u.squal;
        if (!sseq) return KBBQ_E_ARG;   // a resident session has no streaming buffers
        KBBQ_TRY(kbbq_segment_plan(d_rg, d_sec, n, R, u.seg, u.dest, S->d_status, S->s_comp));
        KBBQ_TRY(kbbq_segment_rows(u.seq, u.dest, n, L, sseq, S->s_comp));
        KBBQ_TRY(kbbq_segment_rows(u.qual, u.dest, n, L, squal, S->s_comp));
        KBBQ_TRY(kbbq_segment_pad(u.seg, R, L, sseq, squal, nullptr, S->s_comp));
        a_seq = sseq; a_qual = squal;
    }
    KBBQ_TRY(apply_and_download(S, a_seq, a_qual, d_rg, d_sec, u.seg, u.dest, n, out_host));
    KBBQ_CUDA(cudaEventRecord(u.consumed, S->s_comp));
    return KBBQ_OK;
}

int session_sync(kbbq_session *S, int *status_out) {
    int st = 0;
    KBBQ_CUDA(cudaStreamSynchronize(S->s_up));
    KBBQ_CUDA(cudaStreamSynchronize(S->s_comp));
    KBBQ_CUDA(cudaStreamSynchronize(S->s_down));
    KBBQ_CUDA(cudaMemcpy(&st, S->d_status, sizeof(int), cudaMemcpyDeviceToHost));
    st |= S->host_status;
    if (status_out) *status_out = st;
    return st ? KBBQ_E_DATA : KBBQ_OK;
}

// ---- sessions kept between calls of the whole-path entry points (allocating several GB per call costs tens of
// milliseconds to a second of driver page scrubbing, far more than the kernels) ----
struct CacheSlot {
    std::mutex mu;
    std::unique_ptr<kbbq_session> s;
};
CacheSlot g_cache[MAX_DEVICES];

int cached_session(int slot, int device, int L, int R, int minscore, int64_t C, int64_t M, int host_threads, int pack,
                   kbbq_session **out) {
    CacheSlot &c = g_cache[slot];
    kbbq_session *s = c.s.get();
    const int64_t C16 = (C + 15) / 16 * 16;
    const int64_t nres = M ? (M + C16 - 1) / C16 : 0;
    if (s && s->device == device && s->L == L && s->R == R && s->minscore == minscore && s->C == C16 &&
        (int64_t)s->res.size() >= nres && (nres > 0) == (s->M > 0) && s->pack == (pack < 0 ? pack_mode(host_threads) : pack) &&
        s->segmode == want_segmode(L, R, minscore, C16)) {
        s->host_threads = host_threads;
        KBBQ_TRY(session_reset(s));
        *out = s;
        return KBBQ_OK;
    }
    c.s.reset();
    kbbq_session *fresh = nullptr;
    KBBQ_TRY(session_create(device, L, R, minscore, C, M, host_threads, pack, &fresh));
    c.s.reset(fresh);
    *out = fresh;
    return KBBQ_OK;
}

// how many reads of a batch of N can stay resident on `device` (0: stream them twice)
int64_t resident_reads(int device, int64_t N, int L, int R, int64_t C, size_t already_ours) {
    size_t free_b = 0, total_b = 0;
    if (cudaSetDevice(device) != cudaSuccess || cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return 0;
    free_b += already_ours;
    const double per_read = 2.0 * L + 8.0;   // seq + qual + (dest or rg / second)
    const double staging = 12.0 * (double)(C + 32 * R) * L;
    bool resident = (double)N * per_read * 1.02 + staging < 0.85 * (double)free_b;
    if (const char *e = getenv("KBBQ_HOST_FORCE_STREAMING")) resident = resident && atoi(e) == 0;   // test hook
    return resident ? N : 0;
}

// one device's share of the two passes
int run_build_pass(kbbq_session *S, const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
                   const uint8_t *second, int64_t N) {
    const int L = S->L;
    const int64_t C = S->C, nchunks = N ? (N + C - 1) / C : 0;
    const bool keep = S->M > 0;
    const int64_t k0 = S->built;   // chunks already in the session (a range may follow single chunks or another range)
    if (keep && k0 + nchunks > (int64_t)S->res.size()) return KBBQ_E_ARG;
    auto upload = [&](int64_t k) {
        const int64_t r0 = k * C, n = std::min(C, N - r0);
        return build_chunk_upload(S, k0 + k, seq + (size_t)r0 * L, qual + (size_t)r0 * L, rg ? rg + r0 : nullptr,
                                  second ? second + r0 : nullptr, n, keep);
    };
    // the direct copies of chunk k + 1 are queued before chunk k is packed: the copy engine never waits for the cores
    if (nchunks) KBBQ_TRY(upload(0));
    for (int64_t k = 0; k < nchunks; ++k) {
        const int64_t r0 = k * C, n = std::min(C, N - r0);
        if (k + 1 < nchunks) KBBQ_TRY(upload(k + 1));
        KBBQ_TRY(build_chunk_finish(S, k0 + k, seq + (size_t)r0 * L, corr + (size_t)r0 * L, rg != nullptr, second != nullptr, n, keep));
    }
    S->built = k0 + nchunks;
    return KBBQ_OK;
}

int run_apply_pass(kbbq_session *S, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second,
                   int64_t N, uint8_t *out_qual) {
    const int L = S->L;
    const int64_t C = S->C, nchunks = N ? (N + C - 1) / C : 0;
    KBBQ_TRY(model_async(S));
    for (int64_t k = 0; k < nchunks; ++k) {
        const int64_t r0 = k * C, n = std::min(C, N - r0);
        if (S->M > 0) KBBQ_TRY(apply_resident_async(S, k, out_qual + (size_t)r0 * L));
        else KBBQ_TRY(apply_chunk_async(S, seq + (size_t)r0 * L, qual + (size_t)r0 * L, rg ? rg + r0 : nullptr,
                                        second ? second + r0 : nullptr, n, out_qual + (size_t)r0 * L));
    }
    return KBBQ_OK;
}

int fetch_results(kbbq_session *S, int64_t *tables_host, int64_t *deltas_host) {
    const int L = S->L, R = S->R;
    if (tables_host)
        KBBQ_CUDA(cudaMemcpyAsync(tables_host, S->summed ? S->d_sum : S->d_tab, S->ntab * 8, cudaMemcpyDeviceToHost, S->s_comp));
    if (deltas_host)
        KBBQ_CUDA(cudaMemcpyAsync(deltas_host, S->mp.meanq, ((size_t)2 * R + (size_t)R * NQ * (1 + 2 * L + 17)) * 8,
                                  cudaMemcpyDeviceToHost, S->s_comp));
    return KBBQ_OK;
}

struct Barrier {   // std::barrier is C++20
    std::mutex mu;
    std::condition_variable cv;
    int n, waiting = 0, generation = 0;
    explicit Barrier(int n_) : n(n_) {}
    void wait() {
        std::unique_lock<std::mutex> lk(mu);
        const int gen = generation;
        if (++waiting == n) { waiting = 0; ++generation; cv.notify_all(); }
        else cv.wait(lk, [&] { return gen != generation; });
    }
};

}  // namespace

extern "C" {

int kbbq_session_create(int device, int L, int R, int minscore, int64_t chunk_reads, int64_t resident_reads_cap,
                        int host_threads, kbbq_session **out) {
    if (chunk_reads <= 0) chunk_reads = default_chunk_reads(L > 0 ? L : 1);
    return session_create(device, L, R, minscore, chunk_reads, resident_reads_cap, host_threads, -1, out);
}

void kbbq_session_destroy(kbbq_session *s) { delete s; }

int64_t kbbq_session_chunk_reads(const kbbq_session *s) { return s ? s->C : -1; }

int kbbq_session_reset(kbbq_session *s) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    return session_reset(s);
}

int kbbq_session_build_chunk(kbbq_session *s, const uint8_t *seq, const uint8_t *qual, const uint8_t *corr,
                             const uint16_t *rg, const uint8_t *second, int64_t n, int keep_resident) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    const int64_t k = s->built;
    KBBQ_TRY(build_chunk_async(s, seq, qual, corr, rg, second, n, keep_resident != 0));
    if (n > 0) KBBQ_CUDA(cudaEventSynchronize(s->up[k & 1].uploaded));   // the caller may reuse its buffers
    return KBBQ_OK;
}

int kbbq_session_build_range(kbbq_session *s, const uint8_t *seq, const uint8_t *qual, const uint8_t *corr,
                             const uint16_t *rg, const uint8_t *second, int64_t n) {
    if (!s || n < 0 || (n > 0 && (!seq || !qual || !corr))) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    KBBQ_TRY(run_build_pass(s, seq, qual, corr, rg, second, n));
    KBBQ_CUDA(cudaStreamSynchronize(s->s_up));   // the caller may reuse its buffers
    return KBBQ_OK;
}

int kbbq_session_tables(kbbq_session *s, int64_t *tables_host) {
    if (!s || !tables_host) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    KBBQ_CUDA(cudaMemcpyAsync(tables_host, s->summed ? s->d_sum : s->d_tab, s->ntab * 8, cudaMemcpyDeviceToHost, s->s_comp));
    KBBQ_CUDA(cudaStreamSynchronize(s->s_comp));
    return KBBQ_OK;
}

int kbbq_session_set_tables(kbbq_session *s, const int64_t *tables_host) {
    if (!s || !tables_host) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    KBBQ_CUDA(cudaMemcpyAsync(s->d_tab, tables_host, s->ntab * 8, cudaMemcpyHostToDevice, s->s_comp));
    KBBQ_CUDA(cudaStreamSynchronize(s->s_comp));
    s->summed = false;
    return KBBQ_OK;
}

int kbbq_session_tables_dev(kbbq_session *s, int64_t **tables_dev, int64_t *elems, void **stream) {
    if (!s || !tables_dev) return KBBQ_E_ARG;
    *tables_dev = s->d_tab;
    if (elems) *elems = (int64_t)s->ntab;
    if (stream) *stream = (void *)s->s_comp;
    return KBBQ_OK;
}

int kbbq_session_model(kbbq_session *s, int64_t *deltas_host) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    KBBQ_TRY(model_async(s));
    if (deltas_host) {
        KBBQ_TRY(fetch_results(s, nullptr, deltas_host));
        KBBQ_CUDA(cudaStreamSynchronize(s->s_comp));
    }
    return KBBQ_OK;
}

int kbbq_session_apply_resident(kbbq_session *s, int64_t chunk, uint8_t *out_qual) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    return apply_resident_async(s, chunk, out_qual);
}

int kbbq_session_apply_chunk(kbbq_session *s, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg,
                             const uint8_t *second, int64_t n, uint8_t *out_qual) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    const int64_t k = s->applied;
    KBBQ_TRY(apply_chunk_async(s, seq, qual, rg, second, n, out_qual));
    if (n > 0) KBBQ_CUDA(cudaEventSynchronize(s->up[k & 1].uploaded));   // the caller may reuse its input buffers
    return KBBQ_OK;
}

int kbbq_session_flush(kbbq_session *s) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    KBBQ_CUDA(cudaStreamSynchronize(s->s_up));
    KBBQ_CUDA(cudaStreamSynchronize(s->s_comp));
    return KBBQ_OK;
}

int kbbq_session_sync(kbbq_session *s, int *status_out) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    return session_sync(s, status_out);
}

int kbbq_session_traffic(const kbbq_session *s, int64_t *h2d_bytes, int64_t *d2h_bytes) {
    if (!s) return KBBQ_E_ARG;
    if (h2d_bytes) *h2d_bytes = s->h2d_bytes;
    if (d2h_bytes) *d2h_bytes = s->d2h_bytes;
    return KBBQ_OK;
}

int kbbq_host_pack_mode(int host_threads) { return pack_mode(host_threads); }

int kbbq_host_last_traffic(int device, int64_t *h2d_bytes, int64_t *d2h_bytes) {
    if (device < 0) return KBBQ_E_ARG;
    int64_t up = 0, down = 0;
    for (auto &c : g_cache) {
        std::lock_guard<std::mutex> lock(c.mu);
        if (c.s && c.s->device == device) { up += c.s->h2d_bytes; down += c.s->d2h_bytes; }
    }
    if (h2d_bytes) *h2d_bytes = up;
    if (d2h_bytes) *d2h_bytes = down;
    return KBBQ_OK;
}

int kbbq_host_release(int device) {
    if (device < 0) return KBBQ_E_ARG;
    for (auto &c : g_cache) {
        std::lock_guard<std::mutex> lock(c.mu);
        if (c.s && c.s->device == device) c.s.reset();
    }
    return KBBQ_OK;
}

// ---- FASTQ files in, recalibrated FASTQ out: the whole of recalibrate.recalibrate_fastq (kbbq/recalibrate.py:123-156) ----
namespace {

struct PinnedCache {   // staging slots of the FASTQ pipeline, kept between calls (page-locking costs ~0.1 ms per MB)
    std::mutex mu;
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return KBBQ_OK;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        KBBQ_CUDA(cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
        cap = bytes;
        return KBBQ_OK;
    }
};
PinnedCache g_pinned;

struct FastqPair {
    kbbq_fastq *reads = nullptr, *corr = nullptr;
    // unmapping two large files and freeing their indices takes milliseconds nobody has to wait for
    ~FastqPair() {
        kbbq_fastq *a = reads, *b = corr;
        if (!a && !b) return;
        try { std::thread([a, b] { kbbq_fastq_close(a); kbbq_fastq_close(b); }).detach(); }
        catch (...) { kbbq_fastq_close(a); kbbq_fastq_close(b); }
    }
};

struct OutputMap {   // the output file mapped read-write (fastq_io.cpp: kbbq_fastq_write), or a buffer + write()
    int fd = -1, rw = -1;
    off_t pos0 = 0, base = 0, size0 = 0;
    char *map = nullptr;
    size_t span = 0;
    int64_t total = 0;
    bool finished = false;
    std::vector<char> buf;
    std::thread ahead;
    std::atomic<bool> stop{false};
    int open_for(int out_fd, int64_t bytes) {
        fd = out_fd;
        total = bytes;
        pos0 = lseek(fd, 0, SEEK_CUR);
        const int fl = fcntl(fd, F_GETFL);
        struct stat st;
        if (pos0 >= 0 && fl >= 0 && !(fl & O_APPEND) && bytes > 0 && fstat(fd, &st) == 0 && S_ISREG(st.st_mode) &&
            !getenv("KBBQ_FASTQ_NO_MMAP")) {
            char link[64];
            snprintf(link, sizeof(link), "/proc/self/fd/%d", fd);
            rw = open(link, O_RDWR);
            if (rw >= 0) {
                const long page = sysconf(_SC_PAGESIZE);
                size0 = st.st_size;
                base = pos0 / page * page;
                span = (size_t)(pos0 - base) + (size_t)bytes;
                void *m = MAP_FAILED;
                if (ftruncate(rw, pos0 + (off_t)bytes) == 0) m = mmap(nullptr, span, PROT_READ | PROT_WRITE, MAP_SHARED, rw, base);
                if (m != MAP_FAILED) map = (char *)m;
                else { if (ftruncate(rw, size0)) {} close(rw); rw = -1; }
            }
        }
        // A new file's pages are instantiated one fault at a time, and adding a page to the file is serialised per
        // file (~8 GB/s into a tmpfs however many threads write).  One background thread allocates the blocks ahead
        // of the formatting threads with fallocate -- no zeroing, no mapping -- while the reads are still being
        // tokenised and built; the faults behind it only zero and map.  (Pre-faulting with MADV_POPULATE_WRITE,
        // which zeroes and maps as well, was measured slower than plain faults.)  KBBQ_FASTQ_NO_FALLOCATE=1: off.
        if (map && !getenv("KBBQ_FASTQ_NO_FALLOCATE")) {
            ahead = std::thread([this] {
                const off_t slice = (off_t)32 << 20;
                for (off_t o = 0; o < (off_t)total && !stop.load(std::memory_order_relaxed); o += slice) {
                    const off_t n = std::min<off_t>(slice, (off_t)total - o);
                    if (fallocate(rw, 0, pos0 + o, n) != 0) break;   // not supported here: plain faults do the work
                }
            });
        }
        return KBBQ_OK;
    }
    char *at(int64_t off, int64_t bytes) {   // where `bytes` of output starting at `off` are formatted
        if (map) return map + (pos0 - base) + off;
        buf.resize((size_t)bytes);
        return buf.data();
    }
    int commit(int64_t bytes) {   // unmapped output: write the chunk just formatted
        if (map) return KBBQ_OK;
        const char *p = buf.data();
        size_t left = (size_t)bytes;
        while (left) {
            const ssize_t k = write(fd, p, left);
            if (k < 0) return KBBQ_E_IO;
            p += k;
            left -= (size_t)k;
        }
        return KBBQ_OK;
    }
    void join_ahead() {
        stop.store(true);
        if (ahead.joinable()) ahead.join();
    }
    int finish() {
        join_ahead();
        finished = true;
        if (map) {
            // the text is in the page cache whether or not this process still maps it: tearing the mapping down
            // (one page-table entry per 4 KB) is left to a thread nobody waits for
            char *m = map;
            const size_t len = span;
            map = nullptr;
            try { std::thread([m, len] { munmap(m, len); }).detach(); }
            catch (...) { munmap(m, len); }
            if (lseek(fd, pos0 + (off_t)total, SEEK_SET) < 0) return KBBQ_E_IO;
        }
        return KBBQ_OK;
    }
    ~OutputMap() {
        join_ahead();
        if (map) munmap(map, span);
        // an error before the end: nothing has been printed as far as the caller is concerned (the reference raises
        // in its first pass, before any output), so the file gets its size back
        if (rw >= 0 && !finished && ftruncate(rw, size0)) {}
        if (rw >= 0) close(rw);
    }
};

}  // namespace

int kbbq_recalibrate_fastq(const char *reads_path, const char *corrected_path, int infer_rg, int minscore, int out_fd,
                           int device, int threads, int64_t *n_reads_out, int *n_rg_out, int *status_out) {
    if (!reads_path || !corrected_path || out_fd < 0 || device < 0) return KBBQ_E_ARG;
    const bool trace = !env_flag_off("KBBQ_HOST_TRACE");
    const auto t_start = std::chrono::steady_clock::now();
    auto stamp = [&](const char *what) {
        if (trace)
            fprintf(stderr, "[kbbq fastq] %-30s %8.2f ms\n", what,
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count());
    };
    const int T = threads > 0 ? threads : usable_cpus();
    const int half = std::max(1, T / 2);
    FastqPair fq;
    int rc_a = KBBQ_OK, rc_b = KBBQ_OK;
    {   // both files are indexed at the same time
        std::thread tb([&] { rc_b = kbbq_fastq_open(corrected_path, T - half > 0 ? T - half : 1, &fq.corr); });
        rc_a = kbbq_fastq_open(reads_path, half, &fq.reads);
        tb.join();
    }
    if (rc_a) return rc_a;
    if (rc_b) return rc_b;
    stamp("files indexed");
    const int64_t n = kbbq_fastq_num_reads(fq.reads);
    if (n_reads_out) *n_reads_out = n;
    if (n_rg_out) *n_rg_out = 1;
    if (status_out) *status_out = 0;
    if (kbbq_fastq_num_reads(fq.corr) != n) return KBBQ_E_UNSUPPORTED;   // zip() semantics: the chunked Python driver
    if (n == 0) return KBBQ_OK;
    const int L = kbbq_fastq_read_len(fq.reads);
    if (L < 0 || kbbq_fastq_read_len(fq.corr) != L) return KBBQ_E_RAGGED;
    if (L < 1) return KBBQ_E_FORMAT;

    int64_t C = 262144;
    if (const char *e = getenv("KBBQ_FASTQ_CHUNK_READS")) C = std::max<int64_t>(16, atoll(e));
    C = std::min<int64_t>((C + 15) / 16 * 16, (n + 15) / 16 * 16);
    const int64_t nchunks = (n + C - 1) / C;
    // where every chunk's text goes.  The output is sized, mapped and its blocks allocated (by a background thread)
    // before anything else: the later that starts, the more of it is left for pass 2 to wait for.  Every error
    // return below gives the file its size back (~OutputMap).
    std::vector<int64_t> off((size_t)nchunks + 1, 0);
    for (int64_t k = 0; k < nchunks; ++k) {
        int64_t b = 0;
        KBBQ_TRY(kbbq_fastq_format_size(fq.reads, k * C, std::min(C, n - k * C), T, &b));
        off[(size_t)k + 1] = off[(size_t)k] + b;
    }
    OutputMap out;
    KBBQ_TRY(out.open_for(out_fd, off[(size_t)nchunks]));
    stamp("output sized and mapped");

    std::vector<uint16_t> rg((size_t)n);
    std::vector<uint8_t> second((size_t)n);
    int R = 1;
    {   // name check (find_corrected_sites) and read-group / mate inference side by side
        int64_t bad = -1;
        std::thread tb([&] { rc_b = kbbq_fastq_check_names(fq.reads, fq.corr, n, T - half > 0 ? T - half : 1, &bad); });
        rc_a = kbbq_fastq_infer(fq.reads, infer_rg, rg.data(), second.data(), &R, half);
        tb.join();
    }
    if (rc_b) return rc_b;
    if (rc_a) return rc_a;
    if (R < 1) R = 1;
    if (n_rg_out) *n_rg_out = R;
    stamp("names checked, groups inferred");

    KBBQ_CUDA(cudaSetDevice(device));
    std::unique_lock<std::mutex> cache_lock(g_cache[0].mu);
    size_t ours = g_cache[0].s && g_cache[0].s->device == device ? g_cache[0].s->cap : 0;
    if (resident_reads(device, n, L, R, C, ours) == 0) return KBBQ_E_UNSUPPORTED;   // larger than the device: chunked driver
    kbbq_session *S = nullptr;
    // every core is busy tokenising and the copy engine has time to spare (3 B per base at 55 GB/s against 10 GB/s
    // of FASTQ text): the chunks cross PCIe as they are, no packing pass (KBBQ_FASTQ_PACK=1: as the host-buffer path)
    KBBQ_TRY(cached_session(0, device, L, R, minscore, C, n, T, env_flag_off("KBBQ_FASTQ_PACK") ? PACK_NONE : -1, &S));
    const size_t cb = (size_t)C * L;
    std::lock_guard<std::mutex> pin_lock(g_pinned.mu);
    KBBQ_TRY(g_pinned.ensure(8 * cb));
    uint8_t *pin = (uint8_t *)g_pinned.p;
    uint8_t *h_seq[2] = {pin, pin + cb}, *h_qual[2] = {pin + 2 * cb, pin + 3 * cb}, *h_corr[2] = {pin + 4 * cb, pin + 5 * cb},
            *h_out[2] = {pin + 6 * cb, pin + 7 * cb};
    stamp("session and staging ready");

    // pass 1: tokenise a chunk into a pinned slot while the previous one is on its way to the device
    for (int64_t k = 0; k < nchunks; ++k) {
        const int b = (int)(k & 1);
        const int64_t r0 = k * C, m = std::min(C, n - r0);
        KBBQ_CUDA(cudaEventSynchronize(S->up[b].uploaded));   // the slot's previous chunk has left host memory
        KBBQ_TRY(kbbq_fastq_pack(fq.reads, r0, m, h_seq[b], h_qual[b], T));
        KBBQ_TRY(kbbq_fastq_pack(fq.corr, r0, m, h_corr[b], nullptr, T));
        KBBQ_TRY(build_chunk_async(S, h_seq[b], h_qual[b], h_corr[b], R > 1 ? rg.data() + r0 : nullptr, second.data() + r0, m, true));
    }
    stamp("pass 1 enqueued");
    KBBQ_TRY(model_async(S));
    // pass 2: chunk k is applied and copied back while chunk k - 1 is formatted into the output file
    auto emit = [&](int64_t k) -> int {
        const int b = (int)(k & 1);
        const int64_t r0 = k * C, m = std::min(C, n - r0);
        KBBQ_CUDA(cudaEventSynchronize(S->down[b].drained));
        if (k == 0) {   // bad input raises before anything is printed, as the reference's first pass does
            int st = 0;
            KBBQ_CUDA(cudaMemcpy(&st, S->d_status, sizeof(int), cudaMemcpyDeviceToHost));
            st |= S->host_status;
            if (st) { if (status_out) *status_out = st; return KBBQ_E_DATA; }
        }
        const int64_t bytes = off[(size_t)k + 1] - off[(size_t)k];
        KBBQ_TRY(kbbq_fastq_format(fq.reads, r0, m, h_out[b], out.at(off[(size_t)k], bytes), bytes, T));
        return out.commit(bytes);
    };
    for (int64_t k = 0; k < nchunks; ++k) {
        KBBQ_TRY(apply_resident_async(S, k, h_out[k & 1]));
        if (k >= 1) KBBQ_TRY(emit(k - 1));
    }
    KBBQ_TRY(emit(nchunks - 1));
    stamp("pass 2 done");
    int st = 0;
    const int rc = session_sync(S, &st);
    if (status_out) *status_out = st;
    KBBQ_TRY(out.finish());
    stamp("all done");
    return rc;
}

int kbbq_recalibrate_host(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
                          const uint8_t *second, int64_t N, int L, int R, int minscore, uint8_t *out_qual,
                          int64_t *tables_host, int64_t *deltas_host, int *status_out, int device) {
    const int devices[1] = {device};
    return kbbq_recalibrate_host_multi(seq, qual, corr, rg, second, N, L, R, minscore, out_qual, tables_host, deltas_host,
                                       status_out, devices, 1);
}

int kbbq_recalibrate_host_multi(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
                                const uint8_t *second, int64_t N, int L, int R, int minscore, uint8_t *out_qual,
                                int64_t *tables_host, int64_t *deltas_host, int *status_out, const int *devices,
                                int n_dev) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || !devices || n_dev < 1 || n_dev > MAX_DEVICES) return KBBQ_E_ARG;
    if (N > 0 && (!seq || !qual || !corr || !out_qual)) return KBBQ_E_ARG;
    int ndev_visible = 0;
    KBBQ_CUDA(cudaGetDeviceCount(&ndev_visible));
    for (int i = 0; i < n_dev; ++i)
        if (devices[i] < 0 || devices[i] >= ndev_visible) return KBBQ_E_ARG;

    // can every device read every other device's tables?  (the same device listed twice trivially can)
    bool p2p = n_dev > 1;
    if (const char *e = getenv("KBBQ_MULTI_NO_P2P")) p2p = p2p && atoi(e) == 0;   // test hook: sum through the host
    for (int i = 0; i < n_dev && p2p; ++i)
        for (int j = 0; j < n_dev && p2p; ++j) {
            if (devices[i] == devices[j]) continue;
            int ok = 0;
            if (cudaDeviceCanAccessPeer(&ok, devices[i], devices[j]) != cudaSuccess || !ok) p2p = false;
        }
    if (p2p)
        for (int i = 0; i < n_dev; ++i) {
            KBBQ_CUDA(cudaSetDevice(devices[i]));
            for (int j = 0; j < n_dev; ++j) {
                if (devices[i] == devices[j]) continue;
                const cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
                if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                else if (e != cudaSuccess) { cudaGetLastError(); p2p = false; }
            }
        }

    std::vector<std::unique_lock<std::mutex>> locks;
    for (int i = 0; i < n_dev; ++i) locks.emplace_back(g_cache[i].mu);
    const int host_threads = std::max(1, usable_cpus() / n_dev);
    const int64_t units = (N + 15) / 16;
    std::vector<kbbq_session *> S((size_t)n_dev, nullptr);
    std::vector<int64_t> lo((size_t)n_dev), hi((size_t)n_dev);
    for (int i = 0; i < n_dev; ++i) {   // kbbq/parallel.py: shard_range -- contiguous, boundaries at multiples of 16 reads
        lo[i] = std::min(N, units * i / n_dev * 16);
        hi[i] = std::min(N, units * (i + 1) / n_dev * 16);
    }
    for (int i = 0; i < n_dev; ++i) {
        const int64_t n = hi[i] - lo[i];
        const int64_t C = std::min<int64_t>(default_chunk_reads(L), std::max<int64_t>(16, (n + 15) / 16 * 16));
        size_t ours = 0;
        for (int j = 0; j < n_dev; ++j)
            if (g_cache[j].s && g_cache[j].s->device == devices[i]) ours += j == i ? g_cache[j].s->cap : 0;
        KBBQ_TRY(cached_session(i, devices[i], L, R, minscore, C, resident_reads(devices[i], n, L, R, C, ours), host_threads, -1, &S[i]));
    }

    std::vector<int> rcs((size_t)n_dev, KBBQ_OK), sts((size_t)n_dev, 0);
    Barrier bar(n_dev);
    std::vector<int64_t> h_sum;              // the sum through the host when the devices cannot reach each other
    std::vector<std::vector<int64_t>> h_part;
    if (n_dev > 1 && !p2p) { h_sum.assign(S[0]->ntab, 0); h_part.resize((size_t)n_dev); }
    std::atomic<int> failed{0};

    // Sum of the partial tables, called by every worker between its passes.  Each worker passes the same barriers
    // whatever happened to it, so that a failure on one device cannot leave the others waiting.
    auto sum_tables = [&](int i, int rc) -> int {
        kbbq_session *self = S[i];
        if (n_dev == 1) return rc;
        // every session's tables complete ...
        if (rc == KBBQ_OK && cudaStreamSynchronize(self->s_comp) != cudaSuccess) rc = KBBQ_E_CUDA;
        if (rc == KBBQ_OK && !p2p) {
            h_part[i].resize(self->ntab);
            if (cudaMemcpy(h_part[i].data(), self->d_tab, self->ntab * 8, cudaMemcpyDeviceToHost) != cudaSuccess) rc = KBBQ_E_CUDA;
        }
        if (rc) failed.store(1);
        bar.wait();
        const bool go = !failed.load();
        // ... then each device adds them all up for itself: identical integers everywhere, no broadcast
        if (go && p2p) {
            PeerTables p;
            for (int j = 0; j < n_dev; ++j) p.src[j] = (const long long *)S[j]->d_tab;
            int sms = KBBQ_SM_COUNT_FALLBACK;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, self->device);
            sum_tables_kernel<<<sms * 2, 256, 0, self->s_comp>>>(p, n_dev, (long long *)self->d_sum, self->ntab);
            ++g_launches;
            // a peer must not start its next run (which clears its tables) before this kernel has read them
            if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(self->s_comp) != cudaSuccess) rc = KBBQ_E_CUDA;
        }
        if (!p2p) {
            if (go && i == 0)
                for (int j = 0; j < n_dev; ++j)
                    for (size_t e = 0; e < h_sum.size(); ++e) h_sum[e] += h_part[j][e];
            bar.wait();
            if (go && (cudaMemcpyAsync(self->d_sum, h_sum.data(), self->ntab * 8, cudaMemcpyHostToDevice, self->s_comp) != cudaSuccess ||
                       cudaStreamSynchronize(self->s_comp) != cudaSuccess)) rc = KBBQ_E_CUDA;
        }
        self->summed = true;
        if (rc) failed.store(1);
        bar.wait();
        if (rc == KBBQ_OK && failed.load()) rc = KBBQ_E_CUDA;   // another device failed: nothing to apply
        return rc;
    };
    const bool trace = !env_flag_off("KBBQ_HOST_TRACE");   // where a call spends its time (stderr, device 0's worker)
    const auto t_start = std::chrono::steady_clock::now();
    auto stamp = [&](int i, const char *what) {
        if (trace && i == 0)
            fprintf(stderr, "[kbbq host] %-28s %8.2f ms\n", what,
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count());
    };
    auto worker = [&](int i) {
        kbbq_session *s = S[i];
        const int64_t r0 = lo[i], n = hi[i] - lo[i];
        const uint16_t *rg_i = rg ? rg + r0 : nullptr;
        const uint8_t *sec_i = second ? second + r0 : nullptr;
        int rc = cudaSetDevice(s->device) == cudaSuccess ? KBBQ_OK : KBBQ_E_CUDA;
        stamp(i, "sessions ready");
        if (rc == KBBQ_OK) rc = run_build_pass(s, seq + (size_t)r0 * L, qual + (size_t)r0 * L, corr + (size_t)r0 * L, rg_i, sec_i, n);
        stamp(i, "build pass enqueued");
        if (trace) { cudaStreamSynchronize(s->s_comp); stamp(i, "build pass done"); }
        rc = sum_tables(i, rc);
        if (rc == KBBQ_OK) rc = run_apply_pass(s, seq + (size_t)r0 * L, qual + (size_t)r0 * L, rg_i, sec_i, n, out_qual + (size_t)r0 * L);
        stamp(i, "apply pass enqueued");
        if (rc == KBBQ_OK && i == 0) rc = fetch_results(s, tables_host, deltas_host);
        const int rc2 = session_sync(s, &sts[i]);
        stamp(i, "all done");
        rcs[i] = rc ? rc : rc2;
    };
    if (n_dev == 1) {
        worker(0);
    } else {
        std::vector<std::thread> th;
        for (int i = 0; i < n_dev; ++i) th.emplace_back(worker, i);
        for (auto &t : th) t.join();
    }
    int st = 0, rc = KBBQ_OK;
    for (int i = 0; i < n_dev; ++i) {
        st |= sts[i];
        if (rcs[i] && rcs[i] != KBBQ_E_DATA && rc == KBBQ_OK) rc = rcs[i];
    }
    if (status_out) *status_out = st;
    if (rc) return rc;
    return st ? KBBQ_E_DATA : KBBQ_OK;
}

}  // extern "C"
