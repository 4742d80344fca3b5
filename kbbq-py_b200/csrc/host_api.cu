// host_api.cu -- host-buffer side of the C ABI: sessions, the whole-path entry points, several GPUs, and the
// host-buffer forms of the device-pointer entry points (kbbq_build_host, ...).
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
//
// `kbbq recalibrate -r` streams through the same session: kbbq_session_kmer_sieve x n and kbbq_session_kmer_count x n
// fill a sieved k-mer table (kmer.cuh) in the same slots and streams, kbbq_session_kmer_threshold takes the exact
// histogram, and kbbq_session_build_chunk_kmer is pass 1 with the map flagged on the device in place of the corrected
// reads -- by the boundary rule, or by the correcting walk after kbbq_session_kmer_rule (`-r --correct`).  After
// kbbq_session_kmer_begin_parts the table is split by key across devices: every chunk is copied from the session's
// device to each other partition for its passes, and the map reads the other partitions' tables as peer memory.
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

// where a session is in `kbbq recalibrate -r` (kbbq_session_kmer_*): the calls must come in this order
enum { KMER_NONE = 0, KMER_SIEVE, KMER_COUNT, KMER_READY };

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

// Partition p >= 1 of a k-mer table split by key across devices (kbbq_session_kmer_begin_parts): on `device`, its
// copies of the two staging slots, filter, table, window count, histogram and status word.  Partition 0 is the
// session's own k-mer buffers.
struct KmerPartition {
    int device = 0;
    cudaStream_t up = nullptr, comp = nullptr;       // the peer copy of a chunk; the passes over it
    cudaEvent_t copied[2] = {}, consumed[2] = {};    // per chunk buffer
    uint8_t *chunk[2] = {};
    void *filter = nullptr, *base = nullptr;
    ulonglong2 *table = nullptr;
    uint64_t *windows = nullptr, *hist = nullptr;
    int *status = nullptr;

    void release() {   // waits for its streams; leaves `device` current
        cudaSetDevice(device);
        for (auto s : {up, comp}) if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
        for (auto e : {copied[0], copied[1], consumed[0], consumed[1]}) if (e) cudaEventDestroy(e);
        if (filter) cudaFree(filter);
        if (base) cudaFree(base);
        *this = KmerPartition();
    }
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
    // the sieved k-mer table of kbbq_session_kmer_*: the filter (released when pass B starts), and one allocation of
    // table, window count, histogram and the map of a chunk
    int kmer_stage = KMER_NONE, kmer_k = 0, kmer_t = 0;
    int64_t kmer_chunks = 0;
    uint64_t filter_words = 0, kmer_cap = 0;
    void *kmer_filter = nullptr, *kmer_base = nullptr, *kmer_table = nullptr;
    uint64_t *kmer_windows = nullptr, *kmer_hist = nullptr;
    uint32_t *kmer_bits = nullptr;
    // the rule build_chunk_kmer flags by (kbbq_session_kmer_rule), and whether it has flagged a chunk yet
    int kmer_rule = KBBQ_KMER_BOUNDARIES;
    bool kmer_built = false;
    // partitions 1.. of a table split across devices (kbbq_session_kmer_begin_parts); empty: one table
    std::vector<KmerPartition> kparts;
    std::mutex mu;

    ~kbbq_session() {
        for (auto &q : kparts) q.release();
        cudaSetDevice(device);
        for (auto s : {s_up, s_comp, s_down}) if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
        for (auto &u : up) { if (u.uploaded) cudaEventDestroy(u.uploaded); if (u.consumed) cudaEventDestroy(u.consumed); }
        for (auto &o : down) { if (o.applied) cudaEventDestroy(o.applied); if (o.drained) cudaEventDestroy(o.drained); }
        if (kmer_filter) cudaFree(kmer_filter);
        if (kmer_base) cudaFree(kmer_base);
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

// Free the k-mer buffers once the compute stream is done with them.
int kmer_release(kbbq_session *S) {
    for (auto &q : S->kparts) q.release();
    S->kparts.clear();
    KBBQ_CUDA(cudaSetDevice(S->device));
    if (S->kmer_filter || S->kmer_base) KBBQ_CUDA(cudaStreamSynchronize(S->s_comp));
    if (S->kmer_filter) KBBQ_CUDA(cudaFree(S->kmer_filter));
    if (S->kmer_base) KBBQ_CUDA(cudaFree(S->kmer_base));
    S->kmer_filter = S->kmer_base = S->kmer_table = nullptr;
    S->kmer_windows = S->kmer_hist = nullptr;
    S->kmer_bits = nullptr;
    S->filter_words = S->kmer_cap = 0;
    S->kmer_stage = KMER_NONE;
    S->kmer_chunks = 0;
    S->kmer_rule = KBBQ_KMER_BOUNDARIES;
    S->kmer_built = false;
    return KBBQ_OK;
}

// Forget the tables and chunks of the previous run (the device memory stays; the k-mer buffers go).
int session_reset(kbbq_session *S) {
    KBBQ_CUDA(cudaSetDevice(S->device));
    KBBQ_CUDA(cudaStreamSynchronize(S->s_up));
    KBBQ_CUDA(cudaStreamSynchronize(S->s_down));
    KBBQ_TRY(kmer_release(S));
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
// read groups and mate flags; the reads too unless they travel as nibbles -- and always on the k-mer path, whose map
// is made on the device from the reads).  Nothing waits for the device.
int build_chunk_upload(kbbq_session *S, int64_t k, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg,
                       const uint8_t *second, int64_t n, bool keep, bool kmer = false) {
    if (!chunk_args_ok(S, k, n, keep) || !seq || !qual) return KBBQ_E_ARG;
    const ChunkPlace p = chunk_place(S, k, keep, rg != nullptr, second != nullptr);
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_up, p.u->consumed, 0));   // the slot's previous chunk has been built
    return upload_reads(S, S->pack == PACK_NIBBLES && !kmer ? nullptr : seq, qual, rg, second, n, p.d_seq, p.d_qual,
                        p.d_rg, p.d_sec);
}

// Second half: the host cores pack (seq, corrected) of the chunk while the copy engine is busy with what
// build_chunk_upload queued (of this chunk and, in run_build_pass, of the next one too), the packed form follows,
// and the compute stream expands it, segments the rows when there are several read groups, and builds.  The only
// wait is for the pinned packing slot (two chunks back).  corr == NULL: the k-mer path -- nothing more goes up, the
// map is flagged from the session's k-mer table and expanded on the device.
int build_chunk_finish(kbbq_session *S, int64_t k, const uint8_t *seq, const uint8_t *corr, bool has_rg, bool has_second,
                       int64_t n, bool keep) {
    const bool kmer = corr == nullptr;
    if (!chunk_args_ok(S, k, n, keep) || !seq || (kmer && S->kmer_stage != KMER_READY)) return KBBQ_E_ARG;
    const ChunkPlace p = chunk_place(S, k, keep, has_rg, has_second);
    UpSlot &u = *p.u;
    Resident *r = p.r;
    const int L = S->L, R = S->R;
    const size_t nb = (size_t)n * L;
    if (r) r->n = n;
    if (kmer) {
    } else if (S->pack) {
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
    if (kmer) {   // every lookup in its owner's table; the tables of other devices are peer memory (NVLink)
        const void *tables[MAX_DEVICES];
        const int n_parts = 1 + (int)S->kparts.size();
        tables[0] = S->kmer_table;
        for (int q = 1; q < n_parts; ++q) tables[q] = S->kparts[(size_t)q - 1].table;
        if (S->kmer_rule == KBBQ_KMER_CORRECT)
            KBBQ_TRY(kbbq_kmer_correct_parts(p.d_seq, n, L, S->kmer_k, tables, n_parts, S->kmer_cap, S->kmer_t,
                                             S->kmer_bits, S->d_status, S->s_comp));
        else
            KBBQ_TRY(kbbq_kmer_flag_parts(p.d_seq, n, L, S->kmer_k, tables, n_parts, S->kmer_cap, S->kmer_t,
                                          S->kmer_bits, S->d_status, S->s_comp));
        KBBQ_TRY(kbbq_expand_mismatch_bits(p.d_seq, S->kmer_bits, (int64_t)nb, u.corr, S->s_comp));
    } else if (S->pack == PACK_NIBBLES) KBBQ_TRY(kbbq_expand_nibbles((const uint8_t *)u.bits, (int64_t)nb, p.d_seq, u.corr, S->s_comp));
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
// between kbbq_session_kmer_begin and kbbq_session_kmer_threshold only the k-mer passes may run on a session
bool kmer_counting(const kbbq_session *S) { return S->kmer_stage == KMER_SIEVE || S->kmer_stage == KMER_COUNT; }

int build_chunk_async(kbbq_session *S, const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
                      const uint8_t *second, int64_t n, bool keep) {
    if (n < 0 || n > S->C || kmer_counting(S)) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    if (!seq || !qual || !corr) return KBBQ_E_ARG;
    const int64_t k = S->built;
    if (keep && k >= (int64_t)S->res.size()) return KBBQ_E_ARG;
    S->built++;
    KBBQ_TRY(build_chunk_upload(S, k, seq, qual, rg, second, n, keep));
    return build_chunk_finish(S, k, seq, corr, rg != nullptr, second != nullptr, n, keep);
}

// ---- kbbq recalibrate -r through a streaming session (kbbq_session_kmer_*, DESIGN.md §10 "Streaming") ----

// Partition p of the table on devices[p] (devices[0] = the session's device; n = 1: one table, as before there were
// several).  Nothing is allocated unless every check passes.
int kmer_begin(kbbq_session *S, int k, int64_t windows, uint64_t F, uint64_t cap, const int *devices, int n) {
    auto pow2 = [](uint64_t x) { return x >= 1 && (x & (x - 1)) == 0; };
    if (k < 1 || k > 31 || windows < 0 || S->kmer_stage != KMER_NONE || S->M > 0) return KBBQ_E_ARG;   // streaming only
    if ((F == 0) != (cap == 0) || (F && (!pow2(F) || !pow2(cap)))) return KBBQ_E_ARG;
    if (!devices || n < 1 || n > MAX_DEVICES || devices[0] != S->device || (n > 1 && cap > (1ull << 32)))
        return KBBQ_E_ARG;
    int ndev = 0;
    KBBQ_CUDA(cudaGetDeviceCount(&ndev));
    for (int p = 0; p < n; ++p)
        if (devices[p] < 0 || devices[p] >= ndev) return KBBQ_E_ARG;
    // the session's device reads every partition's table when it flags (the same device listed twice trivially can)
    if (n > 1 && !env_flag_off("KBBQ_MULTI_NO_P2P")) return KBBQ_E_PEER;   // test hook: as if no peer were reachable
    for (int p = 1; p < n; ++p) {
        if (devices[p] == S->device) continue;
        int ok = 0;
        if (cudaDeviceCanAccessPeer(&ok, S->device, devices[p]) != cudaSuccess || !ok) return KBBQ_E_PEER;
    }
    for (int p = 1; p < n; ++p) {
        if (devices[p] == S->device) continue;
        const cudaError_t e = cudaDeviceEnablePeerAccess(devices[p], 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) { cudaGetLastError(); return KBBQ_E_PEER; }
    }
    const size_t chunk_bytes = (size_t)S->C * S->L + 16;
    if (!F) {
        // each partition's budget: 90 % of its device's free memory shared by the partitions there, less the two chunk
        // copies of a partition p >= 1; every partition gets the sizes of the smallest budget
        double budget = 0;
        for (int p = 0; p < n; ++p) {
            size_t free_b = 0, total_b = 0;
            KBBQ_CUDA(cudaSetDevice(devices[p]));
            KBBQ_CUDA(cudaMemGetInfo(&free_b, &total_b));
            const int hosts = (int)std::count(devices, devices + n, devices[p]);
            const double b = 0.9 * (double)free_b / hosts - (p ? 2.0 * (double)chunk_bytes : 0.0);
            budget = p ? std::min(budget, b) : b;
        }
        KBBQ_CUDA(cudaSetDevice(S->device));
        if (budget < 0) return KBBQ_E_UNSUPPORTED;
        KBBQ_TRY(kbbq_kmer_stream_plan(((uint64_t)windows + n - 1) / n, (uint64_t)budget, &F, &cap));
        if (n > 1) cap = std::min<uint64_t>(cap, 1ull << 32);
    }
    const size_t bits_words = ((size_t)S->C * S->L + 31) / 32 + 4;
    Carver c(nullptr);
    c.take<ulonglong2>(cap);
    c.take<uint64_t>(1);
    c.take<uint64_t>(256);
    c.take<uint32_t>(bits_words);
    // a request the device cannot hold is a size problem (KBBQ_E_UNSUPPORTED), not a CUDA failure
    auto alloc = [&](void **p, size_t bytes) -> int {
        const cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) return KBBQ_OK;
        cudaGetLastError();
        *p = nullptr;
        kmer_release(S);
        return e == cudaErrorMemoryAllocation ? KBBQ_E_UNSUPPORTED : KBBQ_E_CUDA;
    };
    KBBQ_TRY(alloc(&S->kmer_filter, F * 8));
    KBBQ_TRY(alloc(&S->kmer_base, c.off));
    Carver d(S->kmer_base);
    S->kmer_table = d.take<ulonglong2>(cap);
    S->kmer_windows = d.take<uint64_t>(1);
    S->kmer_hist = d.take<uint64_t>(256);
    S->kmer_bits = d.take<uint32_t>(bits_words);
    S->filter_words = F;
    S->kmer_cap = cap;
    S->kmer_k = k;
    S->kmer_chunks = 0;
    KBBQ_CUDA(cudaMemsetAsync(S->kmer_filter, 0, F * 8, S->s_comp));
    KBBQ_CUDA(cudaMemsetAsync(S->kmer_windows, 0, 8, S->s_comp));
    KBBQ_TRY(kbbq_kmer_clear(S->kmer_table, cap, S->s_comp));
    S->kmer_stage = KMER_SIEVE;   // from here on kmer_release (reset) frees whatever has been allocated
    for (int p = 1; p < n; ++p) {
        S->kparts.emplace_back();
        KmerPartition &q = S->kparts.back();
        q.device = devices[p];
        KBBQ_CUDA(cudaSetDevice(q.device));
        KBBQ_CUDA(cudaStreamCreateWithFlags(&q.up, cudaStreamNonBlocking));
        KBBQ_CUDA(cudaStreamCreateWithFlags(&q.comp, cudaStreamNonBlocking));
        for (auto e : {&q.copied[0], &q.copied[1], &q.consumed[0], &q.consumed[1]})
            KBBQ_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        Carver m(nullptr);
        m.take<uint8_t>(chunk_bytes);
        m.take<uint8_t>(chunk_bytes);
        m.take<ulonglong2>(cap);
        m.take<uint64_t>(1);
        m.take<uint64_t>(256);
        m.take<int>(64);
        KBBQ_TRY(alloc(&q.filter, F * 8));
        KBBQ_TRY(alloc(&q.base, m.off));
        Carver e(q.base);
        q.chunk[0] = e.take<uint8_t>(chunk_bytes);
        q.chunk[1] = e.take<uint8_t>(chunk_bytes);
        q.table = e.take<ulonglong2>(cap);
        q.windows = e.take<uint64_t>(1);
        q.hist = e.take<uint64_t>(256);
        q.status = e.take<int>(64);
        KBBQ_CUDA(cudaMemsetAsync(q.filter, 0, F * 8, q.comp));
        KBBQ_CUDA(cudaMemsetAsync(q.windows, 0, 8, q.comp));
        KBBQ_CUDA(cudaMemsetAsync(q.status, 0, sizeof(int), q.comp));
        KBBQ_TRY(kbbq_kmer_clear(q.table, cap, q.comp));
    }
    KBBQ_CUDA(cudaSetDevice(S->device));
    return KBBQ_OK;
}

// Whether partition p >= 1 found its table full (its status word; waits for its passes), and the host-side flag that
// makes kbbq_session_sync report it as the session's own status word reports partition 0.
int kmer_parts_full(kbbq_session *S, bool *full) {
    *full = false;
    for (auto &q : S->kparts) {
        int st = 0;
        KBBQ_CUDA(cudaSetDevice(q.device));
        KBBQ_CUDA(cudaMemcpyAsync(&st, q.status, sizeof(int), cudaMemcpyDeviceToHost, q.comp));
        KBBQ_CUDA(cudaStreamSynchronize(q.comp));
        if (st & KBBQ_FLAG_KMER_FULL) *full = true;
    }
    KBBQ_CUDA(cudaSetDevice(S->device));
    if (*full) S->host_status |= KBBQ_FLAG_KMER_FULL;
    return KBBQ_OK;
}

// Pass A (count = false) or B of one chunk: its bytes go up into a staging slot while the previous chunk's kernel runs.
// Partition 0 runs on the slot in place; every other partition copies the slot into its own chunk buffer first, and
// the slot is free again (consumed) once every copy is done.
int kmer_chunk(kbbq_session *S, const uint8_t *seq, int64_t n, bool count, UpSlot **slot) {
    *slot = nullptr;
    const bool in_order = S->kmer_stage == KMER_SIEVE || (count && S->kmer_stage == KMER_COUNT);
    if (!in_order) return KBBQ_E_ARG;
    if (n < 0 || n > S->C || (n > 0 && !seq)) return KBBQ_E_ARG;
    if (count && S->kmer_stage == KMER_SIEVE) {   // pass A is over: its filters are not needed any more
        int st = 0;
        bool parts_full = false;
        KBBQ_CUDA(cudaMemcpyAsync(&st, S->d_status, sizeof(int), cudaMemcpyDeviceToHost, S->s_comp));
        KBBQ_CUDA(cudaStreamSynchronize(S->s_comp));
        KBBQ_TRY(kmer_parts_full(S, &parts_full));
        KBBQ_CUDA(cudaFree(S->kmer_filter));
        S->kmer_filter = nullptr;
        for (auto &q : S->kparts) {
            KBBQ_CUDA(cudaSetDevice(q.device));
            KBBQ_CUDA(cudaFree(q.filter));
            q.filter = nullptr;
        }
        KBBQ_CUDA(cudaSetDevice(S->device));
        S->kmer_stage = KMER_COUNT;
        // a table that filled in pass A is reported here, before pass B; one that fills in pass B stops its kernels
        // (kmer.cuh) and is reported by kbbq_session_kmer_threshold
        if ((st & KBBQ_FLAG_KMER_FULL) || parts_full) return KBBQ_E_DATA;
    }
    if (n == 0) return KBBQ_OK;
    const int b = (int)(S->kmer_chunks++ & 1);
    UpSlot &u = S->up[b];
    const size_t nb = (size_t)n * S->L;
    const int L = S->L, k = S->kmer_k, n_parts = 1 + (int)S->kparts.size();
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_up, u.consumed, 0));
    KBBQ_CUDA(cudaMemcpyAsync(u.seq, seq, nb, cudaMemcpyHostToDevice, S->s_up));
    S->h2d_bytes += (int64_t)nb;
    KBBQ_CUDA(cudaEventRecord(u.uploaded, S->s_up));
    KBBQ_CUDA(cudaStreamWaitEvent(S->s_comp, u.uploaded, 0));
    if (count)
        KBBQ_TRY(kbbq_kmer_count_present_part(u.seq, n, L, k, 0, n_parts, S->kmer_table, S->kmer_cap, S->kmer_windows,
                                              S->d_status, S->s_comp));
    else
        KBBQ_TRY(kbbq_kmer_sieve_part(u.seq, n, L, k, 0, n_parts, S->kmer_filter, S->filter_words, S->kmer_table,
                                      S->kmer_cap, S->d_status, S->s_comp));
    for (int p = 1; p < n_parts; ++p) {   // a copy even on the session's own device: one GPU runs this path too
        KmerPartition &q = S->kparts[(size_t)p - 1];
        KBBQ_CUDA(cudaSetDevice(q.device));
        KBBQ_CUDA(cudaStreamWaitEvent(q.up, u.uploaded, 0));
        KBBQ_CUDA(cudaStreamWaitEvent(q.up, q.consumed[b], 0));   // the partition's pass over its previous copy
        KBBQ_CUDA(cudaMemcpyPeerAsync(q.chunk[b], q.device, u.seq, S->device, nb, q.up));
        KBBQ_CUDA(cudaEventRecord(q.copied[b], q.up));
        KBBQ_CUDA(cudaStreamWaitEvent(q.comp, q.copied[b], 0));
        if (count)
            KBBQ_TRY(kbbq_kmer_count_present_part(q.chunk[b], n, L, k, p, n_parts, q.table, S->kmer_cap, q.windows,
                                                  q.status, q.comp));
        else
            KBBQ_TRY(kbbq_kmer_sieve_part(q.chunk[b], n, L, k, p, n_parts, q.filter, S->filter_words, q.table,
                                          S->kmer_cap, q.status, q.comp));
        KBBQ_CUDA(cudaEventRecord(q.consumed[b], q.comp));
        KBBQ_CUDA(cudaSetDevice(S->device));
        KBBQ_CUDA(cudaStreamWaitEvent(S->s_comp, q.copied[b], 0));
    }
    KBBQ_CUDA(cudaEventRecord(u.consumed, S->s_comp));
    *slot = &u;
    return KBBQ_OK;
}

// One sieved histogram per partition, summed on the host: the exact histogram of the input.
int kmer_threshold(kbbq_session *S, int min_count, uint64_t *hist_out, int *t_used) {
    if (S->kmer_stage != KMER_COUNT || min_count < 0) return KBBQ_E_ARG;
    std::vector<uint64_t> h(256 * (1 + S->kparts.size()));
    int st = 0;
    for (size_t p = 1; p <= S->kparts.size(); ++p) {
        KmerPartition &q = S->kparts[p - 1];
        KBBQ_CUDA(cudaSetDevice(q.device));
        KBBQ_TRY(kbbq_kmer_histogram_sieved(q.table, S->kmer_cap, q.windows, q.hist, q.comp));
        KBBQ_CUDA(cudaMemcpyAsync(&h[256 * p], q.hist, 256 * sizeof(uint64_t), cudaMemcpyDeviceToHost, q.comp));
    }
    KBBQ_CUDA(cudaSetDevice(S->device));
    KBBQ_TRY(kbbq_kmer_histogram_sieved(S->kmer_table, S->kmer_cap, S->kmer_windows, S->kmer_hist, S->s_comp));
    KBBQ_CUDA(cudaMemcpyAsync(h.data(), S->kmer_hist, 256 * sizeof(uint64_t), cudaMemcpyDeviceToHost, S->s_comp));
    KBBQ_CUDA(cudaMemcpyAsync(&st, S->d_status, sizeof(int), cudaMemcpyDeviceToHost, S->s_comp));
    KBBQ_CUDA(cudaStreamSynchronize(S->s_comp));
    bool parts_full = false;
    KBBQ_TRY(kmer_parts_full(S, &parts_full));
    if ((st & KBBQ_FLAG_KMER_FULL) || parts_full) return KBBQ_E_DATA;
    uint64_t hist[256];
    for (int c = 0; c < 256; ++c) {
        hist[c] = 0;
        for (size_t p = 0; p < h.size() / 256; ++p) hist[c] += h[256 * p + c];
    }
    S->kmer_t = min_count > 0 ? min_count : kbbq_kmer_min_count(hist);
    S->kmer_stage = KMER_READY;
    if (hist_out) memcpy(hist_out, hist, sizeof(hist));
    if (t_used) *t_used = S->kmer_t;
    return KBBQ_OK;
}

// the rule may change from kmer_begin until a chunk has been flagged: every chunk of a run is flagged by one rule
int kmer_rule(kbbq_session *S, int rule) {
    if ((rule != KBBQ_KMER_BOUNDARIES && rule != KBBQ_KMER_CORRECT) || S->kmer_stage == KMER_NONE || S->kmer_built)
        return KBBQ_E_ARG;
    S->kmer_rule = rule;
    return KBBQ_OK;
}

int build_chunk_kmer_async(kbbq_session *S, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg,
                           const uint8_t *second, int64_t n) {
    if (S->kmer_stage != KMER_READY || n < 0 || n > S->C) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    if (!seq || !qual) return KBBQ_E_ARG;
    S->kmer_built = true;
    const int64_t k = S->built++;
    KBBQ_TRY(build_chunk_upload(S, k, seq, qual, rg, second, n, false, true));
    return build_chunk_finish(S, k, seq, nullptr, rg != nullptr, second != nullptr, n, false);
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
    if (n < 0 || n > S->C || !S->up[0].seq || kmer_counting(S)) return KBBQ_E_ARG;
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
    if (kmer_counting(s)) return KBBQ_E_ARG;
    KBBQ_CUDA(cudaSetDevice(s->device));
    KBBQ_TRY(run_build_pass(s, seq, qual, corr, rg, second, n));
    KBBQ_CUDA(cudaStreamSynchronize(s->s_up));   // the caller may reuse its buffers
    return KBBQ_OK;
}

int kbbq_session_kmer_begin(kbbq_session *s, int k, int64_t windows, uint64_t filter_words, uint64_t capacity) {
    if (!s) return KBBQ_E_ARG;
    return kbbq_session_kmer_begin_parts(s, k, windows, filter_words, capacity, &s->device, 1);
}

int kbbq_session_kmer_begin_parts(kbbq_session *s, int k, int64_t windows, uint64_t filter_words, uint64_t capacity,
                                  const int *devices, int n_parts) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    return kmer_begin(s, k, windows, filter_words, capacity, devices, n_parts);
}

static int session_kmer_chunk(kbbq_session *s, const uint8_t *seq, int64_t n, bool count) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    UpSlot *u = nullptr;
    KBBQ_TRY(kmer_chunk(s, seq, n, count, &u));
    if (u) KBBQ_CUDA(cudaEventSynchronize(u->uploaded));   // the caller may reuse its buffer
    return KBBQ_OK;
}

int kbbq_session_kmer_sieve(kbbq_session *s, const uint8_t *seq, int64_t n) { return session_kmer_chunk(s, seq, n, false); }

int kbbq_session_kmer_count(kbbq_session *s, const uint8_t *seq, int64_t n) { return session_kmer_chunk(s, seq, n, true); }

int kbbq_session_kmer_threshold(kbbq_session *s, int min_count, uint64_t *hist_out, int *t_used) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    return kmer_threshold(s, min_count, hist_out, t_used);
}

int kbbq_session_kmer_rule(kbbq_session *s, int rule) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    return kmer_rule(s, rule);
}

int kbbq_session_build_chunk_kmer(kbbq_session *s, const uint8_t *seq, const uint8_t *qual, const uint16_t *rg,
                                  const uint8_t *second, int64_t n) {
    if (!s) return KBBQ_E_ARG;
    std::lock_guard<std::mutex> lock(s->mu);
    KBBQ_CUDA(cudaSetDevice(s->device));
    const int64_t k = s->built;
    KBBQ_TRY(build_chunk_kmer_async(s, seq, qual, rg, second, n));
    if (n > 0) KBBQ_CUDA(cudaEventSynchronize(s->up[k & 1].uploaded));   // the caller may reuse its buffers
    return KBBQ_OK;
}

int kbbq_session_kmer_sizes(const kbbq_session *s, uint64_t *filter_words, uint64_t *capacity) {
    if (!s) return KBBQ_E_ARG;
    if (filter_words) *filter_words = s->filter_words;
    if (capacity) *capacity = s->kmer_cap;
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
                // the file only grows: bytes already behind the text stay, as write() leaves them
                void *m = MAP_FAILED;
                if (!grew() || ftruncate(rw, pos0 + (off_t)bytes) == 0) m = mmap(nullptr, span, PROT_READ | PROT_WRITE, MAP_SHARED, rw, base);
                if (m != MAP_FAILED) map = (char *)m;
                else { if (grew() && ftruncate(rw, size0)) {} close(rw); rw = -1; }
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
    bool grew() const { return pos0 + (off_t)total > size0; }   // the text reaches past the file's old end
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
        // in its first pass, before any output), so the file gets its size back: what the call added goes, the bytes
        // that were there stay
        if (rw >= 0 && !finished && grew() && ftruncate(rw, size0)) {}
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

// ---- host-buffer forms of the device-pointer entry points: copy in, run, copy back, synchronously ----

namespace {

enum SpanDir { IN, OUT, INOUT, SCRATCH };

// One synchronous call of a device-pointer entry point on host buffers.  The wrapper lists its spans (a host pointer,
// a byte count, a direction); begin() carves them from one allocation, uploads the IN / INOUT spans and zeroes the OUT
// spans and the status word; finish() downloads the OUT / INOUT spans and maps a non-zero status to KBBQ_E_DATA.
// Every span starts 256-byte aligned and is readable up to its 16-byte end, as the TMA ring and the vector
// calibration kernel need to take their fast paths.  A NULL host pointer gives a NULL device pointer.
struct HostCall {
    struct Span {
        SpanDir dir;
        void *host;
        size_t bytes;
        char *d;
    };
    template <class T> struct Dev {  // device pointer of a span, valid once begin() has run
        const std::vector<Span> *spans;
        int i;
        operator T *() const { return i < 0 ? nullptr : (T *)(*spans)[i].d; }
    };

    int device;
    bool with_status;
    std::vector<Span> spans;
    void *base = nullptr;
    int *status = nullptr;  // the device status word, with_status only

    HostCall(int device_, bool with_status_) : device(device_), with_status(with_status_) {}
    HostCall(const HostCall &) = delete;
    HostCall &operator=(const HostCall &) = delete;
    ~HostCall() {
        if (base) cudaFree(base);
    }

    template <class T> Dev<T> span(SpanDir dir, T *host, size_t bytes) {
        if (!host && dir != SCRATCH) return {&spans, -1};
        spans.push_back({dir, (void *)host, bytes, nullptr});
        return {&spans, (int)spans.size() - 1};
    }
    Dev<void> scratch(size_t bytes) { return span<void>(SCRATCH, nullptr, bytes); }

    size_t bytes() const {
        Carver size(nullptr);
        for (const Span &s : spans) size.take<char>(s.bytes);
        if (with_status) size.take<int>(1);
        return size.off;
    }

    // *ok = the spans fit the device's free memory now
    int fits(bool *ok) {
        KBBQ_CUDA(cudaSetDevice(device));
        size_t free_b = 0, total_b = 0;
        KBBQ_CUDA(cudaMemGetInfo(&free_b, &total_b));
        *ok = bytes() <= free_b;
        return KBBQ_OK;
    }

    int begin() {
        KBBQ_CUDA(cudaSetDevice(device));
        KBBQ_CUDA(cudaMalloc(&base, bytes()));
        Carver c(base);
        for (Span &s : spans) {
            s.d = c.take<char>(s.bytes);
            if (!s.bytes) continue;
            if (s.dir == IN || s.dir == INOUT) KBBQ_CUDA(cudaMemcpy(s.d, s.host, s.bytes, cudaMemcpyHostToDevice));
            if (s.dir == OUT) KBBQ_CUDA(cudaMemset(s.d, 0, s.bytes));
        }
        if (with_status) {
            status = c.take<int>(1);
            KBBQ_CUDA(cudaMemset(status, 0, sizeof(int)));
        }
        return KBBQ_OK;
    }

    int finish(int *status_out = nullptr) {
        for (const Span &s : spans)
            if (s.bytes && (s.dir == OUT || s.dir == INOUT))
                KBBQ_CUDA(cudaMemcpy(s.host, s.d, s.bytes, cudaMemcpyDeviceToHost));
        if (!with_status) return KBBQ_OK;
        int st = 0;
        KBBQ_CUDA(cudaMemcpy(&st, status, sizeof(int), cudaMemcpyDeviceToHost));
        if (status_out) *status_out = st;
        return st ? KBBQ_E_DATA : KBBQ_OK;
    }
};

}  // namespace

extern "C" {

int kbbq_build_host(const uint8_t *seq, const uint8_t *qual, const uint8_t *corr, const uint16_t *rg,
                    const uint8_t *second, int64_t N, int L, int R, int minscore, int64_t *pos_errs,
                    int64_t *pos_total, int64_t *din_errs, int64_t *din_total, int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535) return KBBQ_E_ARG;
    if (!pos_errs || !pos_total || !din_errs || !din_total || (N > 0 && (!seq || !qual || !corr))) return KBBQ_E_ARG;
    const size_t nb = (size_t)N * L, npos = (size_t)R * NQ * 2 * L * 8, ndin = (size_t)R * NQ * 16 * 8;
    size_t ws_bytes = 0;
    KBBQ_TRY(kbbq_workspace_bytes(N, L, R, &ws_bytes));
    HostCall c(device, true);
    const auto d_seq = c.span(IN, seq, nb);
    const auto d_qual = c.span(IN, qual, nb);
    const auto d_corr = c.span(IN, corr, nb);
    const auto d_rg = c.span(IN, rg, (size_t)N * 2);
    const auto d_sec = c.span(IN, second, (size_t)N);
    const auto pe = c.span(OUT, pos_errs, npos);  // fresh tables
    const auto pt = c.span(OUT, pos_total, npos);
    const auto de = c.span(OUT, din_errs, ndin);
    const auto dt = c.span(OUT, din_total, ndin);
    const auto ws = c.scratch(ws_bytes);
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_build(d_seq, d_qual, d_corr, d_rg, d_sec, N, L, R, minscore, pe, pt, de, dt, ws, ws_bytes, c.status, 0,
                        nullptr));
    return c.finish(status_out);
}

int kbbq_apply_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second, int64_t N,
                    int L, int R, int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                    const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual,
                    int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || nq < 1 || nq > NQ || ndin1 < 16 || ndin1 > 64) return KBBQ_E_ARG;
    if (!meanq || !rgdq || !qdq || !posdq || !dindq || (N > 0 && (!seq || !qual || !out_qual))) return KBBQ_E_ARG;
    const size_t nb = (size_t)N * L, n_q = (size_t)R * nq * 8;
    size_t ws_bytes = 0;
    KBBQ_TRY(kbbq_workspace_bytes(N, L, R, &ws_bytes));
    HostCall c(device, true);
    const auto d_seq = c.span(IN, seq, nb);
    const auto d_qual = c.span(IN, qual, nb);
    const auto d_rg = c.span(IN, rg, (size_t)N * 2);
    const auto d_sec = c.span(IN, second, (size_t)N);
    const auto d_meanq = c.span(IN, meanq, (size_t)R * 8);
    const auto d_rgdq = c.span(IN, rgdq, (size_t)R * 8);
    const auto d_qdq = c.span(IN, qdq, n_q);
    const auto d_posdq = c.span(IN, posdq, n_q * 2 * L);
    const auto d_dindq = c.span(IN, dindq, n_q * ndin1);
    const auto d_out = c.span(OUT, out_qual, nb);
    const auto ws = c.scratch(ws_bytes);
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_apply(d_seq, d_qual, d_rg, d_sec, N, L, R, minscore, d_meanq, d_rgdq, d_qdq, d_posdq, d_dindq, nq,
                        ndin1, d_out, ws, ws_bytes, c.status, 0, nullptr));
    return c.finish(status_out);
}

int kbbq_get_delta_qs_host(const int64_t *meanq, const int64_t *rg_errs, const int64_t *rg_total,
                           const int64_t *q_errs, const int64_t *q_total, const int64_t *pos_errs,
                           const int64_t *pos_total, const int64_t *din_errs, const int64_t *din_total, int R,
                           int nq, int ncyc, int ndin, int64_t *rgdq, int64_t *qdq, int64_t *posdq,
                           int64_t *dindq, int device) {
    if (R < 1 || nq < 1 || ncyc < 0 || ndin < 0) return KBBQ_E_ARG;
    if (!meanq || !rg_errs || !rg_total || !q_errs || !q_total || !rgdq || !qdq) return KBBQ_E_ARG;
    if ((ncyc && (!pos_errs || !pos_total || !posdq)) || !dindq || (ndin && (!din_errs || !din_total)))
        return KBBQ_E_ARG;
    const size_t nr = (size_t)R * 8, n_q = (size_t)R * nq * 8, n_pos = n_q * ncyc, n_din = n_q * ndin;
    HostCall c(device, false);
    const auto d_meanq = c.span(IN, meanq, nr);
    const auto d_rge = c.span(IN, rg_errs, nr);
    const auto d_rgt = c.span(IN, rg_total, nr);
    const auto d_qe = c.span(IN, q_errs, n_q);
    const auto d_qt = c.span(IN, q_total, n_q);
    const auto d_pe = c.span(IN, pos_errs, n_pos);
    const auto d_pt = c.span(IN, pos_total, n_pos);
    const auto d_de = c.span(IN, din_errs, n_din);
    const auto d_dt = c.span(IN, din_total, n_din);
    const auto o_rg = c.span(OUT, rgdq, nr);
    const auto o_q = c.span(OUT, qdq, n_q);
    const auto o_pos = c.span(OUT, posdq, n_pos);
    const auto o_din = c.span(OUT, dindq, n_q * (ndin + 1));
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_get_delta_qs(d_meanq, d_rge, d_rgt, d_qe, d_qt, d_pe, d_pt, d_de, d_dt, R, nq, ncyc, ndin, o_rg, o_q,
                               o_pos, o_din, nullptr));
    return c.finish();
}

int kbbq_delta_q_host(const int64_t *prior_q, const int64_t *numerrs, const int64_t *numtotal, int64_t n,
                      int64_t *delta, int device) {
    if (n < 0 || (n > 0 && (!prior_q || !numerrs || !numtotal || !delta))) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    HostCall c(device, false);
    const auto d_prior = c.span(IN, prior_q, (size_t)n * 8);
    const auto d_errs = c.span(IN, numerrs, (size_t)n * 8);
    const auto d_total = c.span(IN, numtotal, (size_t)n * 8);
    const auto d_delta = c.span(OUT, delta, (size_t)n * 8);
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_delta_q(d_prior, d_errs, d_total, n, d_delta, nullptr));
    return c.finish();
}

int kbbq_posterior_q_real_host(const double *prior_q, const int64_t *numerrs, const int64_t *numtotal, int64_t n,
                               int64_t *posterior, int device) {
    if (n < 0 || (n > 0 && (!prior_q || !numerrs || !numtotal || !posterior))) return KBBQ_E_ARG;
    if (n == 0) return KBBQ_OK;
    HostCall c(device, false);
    const auto d_prior = c.span(IN, prior_q, (size_t)n * 8);
    const auto d_errs = c.span(IN, numerrs, (size_t)n * 8);
    const auto d_total = c.span(IN, numtotal, (size_t)n * 8);
    const auto d_post = c.span(OUT, posterior, (size_t)n * 8);
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_posterior_q_real(d_prior, d_errs, d_total, n, d_post, nullptr));
    return c.finish();
}

// Host-buffer forms of the BAM-side entry points: copy, run, copy back (a BAM batch is small next to
// what the host spends parsing it).
int kbbq_build_bam_host(const uint8_t *seq, const uint8_t *qual, const uint8_t *err, const uint8_t *skip,
                        const uint16_t *rg, const uint8_t *flags, const uint16_t *aln_start, const uint16_t *aln_end,
                        int64_t N, int L, int R, int minscore, int64_t *pos_errs, int64_t *pos_total,
                        int64_t *din_errs, int64_t *din_total, int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535) return KBBQ_E_ARG;
    if (!pos_errs || !pos_total || !din_errs || !din_total || (N > 0 && (!seq || !qual || !err))) return KBBQ_E_ARG;
    const size_t nb = (size_t)N * L, npos = (size_t)R * NQ * 2 * L * 8, ndin = (size_t)R * NQ * 16 * 8;
    size_t ws_bytes = 0;
    KBBQ_TRY(kbbq_bam_workspace_bytes(N, L, R, &ws_bytes));
    HostCall c(device, true);
    const auto d_seq = c.span(IN, seq, nb);
    const auto d_qual = c.span(IN, qual, nb);
    const auto d_err = c.span(IN, err, nb);
    const auto d_skip = c.span(IN, skip, nb);
    const auto d_rg = c.span(IN, rg, (size_t)N * 2);
    const auto d_flags = c.span(IN, flags, (size_t)N);
    const auto d_start = c.span(IN, aln_start, (size_t)N * 2);
    const auto d_end = c.span(IN, aln_end, (size_t)N * 2);
    const auto pe = c.span(INOUT, pos_errs, npos);  // the tables accumulate
    const auto pt = c.span(INOUT, pos_total, npos);
    const auto de = c.span(INOUT, din_errs, ndin);
    const auto dt = c.span(INOUT, din_total, ndin);
    const auto ws = c.scratch(ws_bytes);
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_build_bam(d_seq, d_qual, d_err, d_skip, d_rg, d_flags, d_start, d_end, N, L, R, minscore, pe, pt, de,
                            dt, ws, ws_bytes, c.status, nullptr));
    return c.finish(status_out);
}

int kbbq_apply_bam_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *flags, int64_t N,
                        int L, int R, int minscore, const int64_t *meanq, const int64_t *rgdq, const int64_t *qdq,
                        const int64_t *posdq, const int64_t *dindq, int nq, int ndin1, uint8_t *out_qual,
                        int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || nq < 1 || ndin1 != 17) return KBBQ_E_ARG;
    if (!meanq || !rgdq || !qdq || !posdq || !dindq || (N > 0 && (!seq || !qual || !out_qual))) return KBBQ_E_ARG;
    const size_t nb = (size_t)N * L, n_q = (size_t)R * nq * 8;
    size_t ws_bytes = 0;
    KBBQ_TRY(kbbq_bam_workspace_bytes(N, L, R, &ws_bytes));
    HostCall c(device, true);
    const auto d_seq = c.span(IN, seq, nb);
    const auto d_qual = c.span(IN, qual, nb);
    const auto d_rg = c.span(IN, rg, (size_t)N * 2);
    const auto d_flags = c.span(IN, flags, (size_t)N);
    const auto d_meanq = c.span(IN, meanq, (size_t)R * 8);
    const auto d_rgdq = c.span(IN, rgdq, (size_t)R * 8);
    const auto d_qdq = c.span(IN, qdq, n_q);
    const auto d_posdq = c.span(IN, posdq, n_q * 2 * L);
    const auto d_dindq = c.span(IN, dindq, n_q * ndin1);
    const auto d_out = c.span(OUT, out_qual, nb);
    const auto ws = c.scratch(ws_bytes);
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_apply_bam(d_seq, d_qual, d_rg, d_flags, N, L, R, minscore, d_meanq, d_rgdq, d_qdq, d_posdq, d_dindq,
                            nq, ndin1, d_out, ws, ws_bytes, c.status, nullptr));
    return c.finish(status_out);
}

int kbbq_calibration_counts_host(const uint8_t *qual, const uint8_t *err, const uint8_t *seq, const uint8_t *corr,
                                 const uint8_t *skip, int64_t n, int64_t *total, int64_t *errs, int device) {
    if (n < 0 || !total || !errs || (!err && (!seq || !corr)) || (n > 0 && !qual)) return KBBQ_E_ARG;
    HostCall c(device, false);
    const auto d_qual = c.span(IN, qual, (size_t)n);
    const auto d_err = c.span(IN, err, (size_t)n);
    const auto d_seq = c.span(IN, err ? nullptr : seq, (size_t)n);  // with an error mask, seq and corr are not read
    const auto d_corr = c.span(IN, err ? nullptr : corr, (size_t)n);
    const auto d_skip = c.span(IN, skip, (size_t)n);
    const auto d_total = c.span(OUT, total, 256 * 8);
    const auto d_errs = c.span(OUT, errs, 256 * 8);
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_calibration_counts(d_qual, d_err, d_seq, d_corr, d_skip, n, d_total, d_errs, nullptr));
    return c.finish();
}

int kbbq_marginals_host(const int64_t *pos_errs, const int64_t *pos_total, int L, int R, int64_t *q_errs,
                        int64_t *q_total, int64_t *rg_errs, int64_t *rg_total, int64_t *meanq, int device) {
    if (L < 1 || R < 1 || R > 65535) return KBBQ_E_ARG;
    if (!pos_errs || !pos_total || !q_errs || !q_total || !rg_errs || !rg_total || !meanq) return KBBQ_E_ARG;
    const size_t npos = (size_t)R * NQ * 2 * L * 8, n_q = (size_t)R * NQ * 8, nr = (size_t)R * 8;
    HostCall c(device, false);
    const auto pe = c.span(IN, pos_errs, npos);
    const auto pt = c.span(IN, pos_total, npos);
    const auto qe = c.span(OUT, q_errs, n_q);
    const auto qt = c.span(OUT, q_total, n_q);
    const auto ge = c.span(OUT, rg_errs, nr);
    const auto gt = c.span(OUT, rg_total, nr);
    const auto mq = c.span(OUT, meanq, nr);
    KBBQ_TRY(c.begin());
    KBBQ_TRY(kbbq_marginals(pe, pt, L, R, qe, qt, ge, gt, mq, nullptr));
    return c.finish();
}

}  // extern "C"

// ---- errors from k-mer counts on host buffers (kmer.cuh) ----

namespace {

// clear + count + histogram, the threshold on the host, then the flags by `rule`.  A full table stops before the
// flags: *status = KBBQ_FLAG_KMER_FULL and KBBQ_E_DATA.
int kmer_errors_dev(const uint8_t *seq, int64_t N, int L, int k, int min_count, int rule, void *table, uint64_t cap,
                    uint64_t *d_hist, uint32_t *bits, int *d_status, uint64_t *hist, int *t, int *status) {
    KBBQ_TRY(kbbq_kmer_clear(table, cap, nullptr));
    KBBQ_TRY(kbbq_kmer_count(seq, N, L, k, table, cap, d_status, nullptr));
    KBBQ_TRY(kbbq_kmer_histogram(table, cap, d_hist, nullptr));
    KBBQ_CUDA(cudaMemcpy(hist, d_hist, 256 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    KBBQ_CUDA(cudaMemcpy(status, d_status, sizeof(int), cudaMemcpyDeviceToHost));
    if (*status) return KBBQ_E_DATA;
    *t = min_count > 0 ? min_count : kbbq_kmer_min_count(hist);
    if (rule == KBBQ_KMER_CORRECT) return kbbq_kmer_correct(seq, N, L, k, table, cap, *t, bits, d_status, nullptr);
    return kbbq_kmer_flag(seq, N, L, k, table, cap, *t, bits, d_status, nullptr);
}

bool kmer_rule_ok(int rule) { return rule == KBBQ_KMER_BOUNDARIES || rule == KBBQ_KMER_CORRECT; }

}  // namespace

extern "C" {

int kbbq_kmer_errors_host(const uint8_t *seq, int64_t N, int L, int k, int min_count, uint32_t *bits_out,
                          uint64_t *hist_out, int *min_count_used, int device) {
    return kbbq_kmer_errors_rule_host(seq, N, L, k, min_count, KBBQ_KMER_BOUNDARIES, bits_out, hist_out, min_count_used,
                                      device);
}

int kbbq_kmer_errors_rule_host(const uint8_t *seq, int64_t N, int L, int k, int min_count, int rule, uint32_t *bits_out,
                               uint64_t *hist_out, int *min_count_used, int device) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || min_count < 0 || !kmer_rule_ok(rule) || (N > 0 && (!seq || !bits_out)))
        return KBBQ_E_ARG;
    uint64_t cap = 0;
    size_t table_bytes = 0;
    KBBQ_TRY(kbbq_kmer_table_bytes(N, L, k, &cap, &table_bytes));
    const size_t nb = (size_t)N * L;
    HostCall c(device, true);
    const auto d_seq = c.span(IN, seq, nb);
    const auto d_bits = c.span(OUT, bits_out, (nb + 31) / 32 * 4);
    const auto d_hist = c.scratch(256 * sizeof(uint64_t));
    const auto table = c.scratch(table_bytes);
    bool ok = false;
    KBBQ_TRY(c.fits(&ok));
    if (!ok) return KBBQ_E_UNSUPPORTED;
    KBBQ_TRY(c.begin());
    uint64_t hist[256];
    int t = 0, st = 0;
    KBBQ_TRY(kmer_errors_dev(d_seq, N, L, k, min_count, rule, table, cap, (uint64_t *)(void *)d_hist, d_bits, c.status,
                             hist, &t, &st));
    if (hist_out) memcpy(hist_out, hist, sizeof(hist));
    if (min_count_used) *min_count_used = t;
    return c.finish();
}

int kbbq_recalibrate_kmer_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second,
                               int64_t N, int L, int R, int minscore, int k, int min_count, uint8_t *out_qual,
                               int64_t *tables_host, int64_t *deltas_host, int *min_count_used, int *status_out,
                               int device) {
    return kbbq_recalibrate_kmer_rule_host(seq, qual, rg, second, N, L, R, minscore, k, min_count, KBBQ_KMER_BOUNDARIES,
                                           out_qual, tables_host, deltas_host, min_count_used, status_out, device);
}

int kbbq_recalibrate_kmer_rule_host(const uint8_t *seq, const uint8_t *qual, const uint16_t *rg, const uint8_t *second,
                                    int64_t N, int L, int R, int minscore, int k, int min_count, int rule,
                                    uint8_t *out_qual, int64_t *tables_host, int64_t *deltas_host, int *min_count_used,
                                    int *status_out, int device) {
    if (N < 0 || L < 1 || R < 1 || R > 65535 || minscore < 0 || minscore >= NQ || k < 1 || k > 31 || min_count < 0 ||
        !kmer_rule_ok(rule))
        return KBBQ_E_ARG;
    if (N > 0 && (!seq || !qual || !out_qual)) return KBBQ_E_ARG;
    uint64_t cap = 0;
    size_t table_bytes = 0, ws_bytes = 0;
    KBBQ_TRY(kbbq_kmer_table_bytes(N, L, k, &cap, &table_bytes));
    KBBQ_TRY(kbbq_workspace_bytes(N, L, R, &ws_bytes));
    const size_t nb = (size_t)N * L, npos = (size_t)R * NQ * 2 * L, ndin = (size_t)R * NQ * 16;
    const size_t ntab = 2 * npos + 2 * ndin, nmodel = carve_model(nullptr, L, R).elems;
    HostCall c(device, true);
    const auto d_seq = c.span(IN, seq, nb);
    const auto d_qual = c.span(IN, qual, nb);
    const auto d_rg = c.span(IN, rg, (size_t)N * 2);
    const auto d_sec = c.span(IN, second, (size_t)N);
    const auto d_out = c.span(OUT, out_qual, nb);
    const auto d_bits = c.scratch((nb + 31) / 32 * 4);
    const auto d_corr = c.scratch(nb);
    const auto d_hist = c.scratch(256 * sizeof(uint64_t));
    const auto d_tab = c.scratch(ntab * 8);
    const auto d_model = c.scratch(nmodel * 8);
    const auto ws = c.scratch(ws_bytes);
    const auto table = c.scratch(table_bytes);
    bool ok = false;
    KBBQ_TRY(c.fits(&ok));
    if (!ok) return KBBQ_E_UNSUPPORTED;
    KBBQ_TRY(c.begin());
    uint64_t hist[256];
    int t = 0, st = 0;
    const int rc = kmer_errors_dev(d_seq, N, L, k, min_count, rule, table, cap, (uint64_t *)(void *)d_hist,
                                   (uint32_t *)(void *)d_bits, c.status, hist, &t, &st);
    if (rc == KBBQ_E_DATA && status_out) *status_out = st;
    KBBQ_TRY(rc);
    if (min_count_used) *min_count_used = t;
    // from here on kbbq_recalibrate_host's steps on one batch, with the map in place of the corrected reads
    int64_t *pe = (int64_t *)(void *)d_tab, *pt = pe + npos, *de = pt + npos, *dt = de + ndin;
    const ModelPtrs mp = carve_model((int64_t *)(void *)d_model, L, R);
    uint8_t *corr = (uint8_t *)(void *)d_corr;
    KBBQ_CUDA(cudaMemset(pe, 0, ntab * 8));
    KBBQ_TRY(kbbq_expand_mismatch_bits(d_seq, (uint32_t *)(void *)d_bits, (int64_t)nb, corr, nullptr));
    KBBQ_TRY(kbbq_build(d_seq, d_qual, corr, d_rg, d_sec, N, L, R, minscore, pe, pt, de, dt, ws, ws_bytes, c.status, 0,
                        nullptr));
    KBBQ_TRY(kbbq_marginals(pe, pt, L, R, mp.q_errs, mp.q_total, mp.rg_errs, mp.rg_total, mp.meanq, nullptr));
    KBBQ_TRY(kbbq_get_delta_qs(mp.meanq, mp.rg_errs, mp.rg_total, mp.q_errs, mp.q_total, pe, pt, de, dt, R, NQ, 2 * L,
                               16, mp.rgdq, mp.qdq, mp.posdq, mp.dindq, nullptr));
    // the build has checked these very bases into the same status word
    KBBQ_TRY(kbbq_apply(d_seq, d_qual, d_rg, d_sec, N, L, R, minscore, mp.meanq, mp.rgdq, mp.qdq, mp.posdq, mp.dindq, NQ,
                        17, d_out, ws, ws_bytes, c.status, KBBQ_APPLY_BASES_CHECKED, nullptr));
    if (tables_host) KBBQ_CUDA(cudaMemcpy(tables_host, pe, ntab * 8, cudaMemcpyDeviceToHost));
    if (deltas_host)
        KBBQ_CUDA(cudaMemcpy(deltas_host, mp.meanq, ((size_t)2 * R + (size_t)R * NQ * (1 + 2 * L + 17)) * 8,
                             cudaMemcpyDeviceToHost));
    return c.finish(status_out);
}

}  // extern "C"
