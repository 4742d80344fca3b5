// fastq_io.cpp -- host FASTQ ingest / egress of libkbbq_b200.so (SURVEY.md section 8 row f1).
//
// Replaces what the reference does read by read in Python around the hot path:
//   pysam.FastxFile iteration + get_quality_array            (kbbq/recalibrate.py:56-57,92,141-142)
//   fastq_infer_rg / fastq_infer_secondinpair on every name  (kbbq/compare_reads.py:304-318, kbbq/recalibrate.py:59-64)
//   the name check of find_corrected_sites                   (kbbq/recalibrate.py:17)
//   the per-read print of the recalibrated FASTQ             (kbbq/recalibrate.py:152-156)
// with a multithreaded tokenizer that packs straight into the structure-of-arrays buffers the CUDA
// entry points take, and a multithreaded formatter.  Plain host C++ (no CUDA): line index by parallel
// newline counting, records packed in parallel, read-group numbering in first-seen FILE order
// (thread-local first-seen lists merged in thread order).
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/kbbq_b200.h"

struct kbbq_fastq {
    const char *data = nullptr;   // whole file (mmap, inflated copy, or caller's buffer)
    size_t len = 0;
    void *map = nullptr;          // non-null: munmap on close
    size_t map_len = 0;
    std::vector<char> owned;      // inflated .gz
    std::vector<int64_t> rec;     // rec[i] = offset of record i's '@'; rec[N] = end of data
    int64_t n = 0;
    int L = -1;                   // uniform read length, -1 = reads differ, 0 = no reads
    std::vector<std::string> rg_keys;
};

namespace {

int n_threads(int want, int64_t work_items) {
    int t = want > 0 ? want : (int)std::thread::hardware_concurrency();
    if (t < 1) t = 1;
    if (t > 64) t = 64;
    if ((int64_t)t > work_items) t = (int)std::max<int64_t>(1, work_items);
    return t;
}

// Worker threads kept between calls: the FASTQ pipeline runs some forty short parallel loops per file pair, and
// creating and joining sixteen threads for each costs more than some of the loops themselves.  Any number of callers
// may run loops at the same time (both files are indexed at once): the pool grows to the demand of all running
// loops, so a task never waits for a worker that is blocked in somebody else's loop.  The pool is never destroyed
// (its threads end with the process) and is rebuilt in a forked child.
class WorkerPool {
public:
    static WorkerPool &get() {
        static WorkerPool *p = new WorkerPool;   // leaked on purpose
        return *p;
    }
    // run f(1) .. f(n_tasks) on workers; the caller runs f(0) itself and then waits
    template <class F> void run(int n_tasks, F &f) {
        struct Join { std::mutex m; std::condition_variable c; int left; } j;
        j.left = n_tasks;
        {
            std::lock_guard<std::mutex> lk(mu_);
            if (owner_ != getpid()) {   // forked: the parent's threads do not exist here
                for (auto &w : workers_) w.release();
                workers_.clear();
                queue_.clear();
                idle_ = 0;
                owner_ = getpid();
            }
            for (int t = 1; t <= n_tasks; ++t)
                queue_.emplace_back([&f, &j, t] {
                    f(t);
                    std::lock_guard<std::mutex> g(j.m);
                    if (--j.left == 0) j.c.notify_one();
                });
            // every queued task gets a worker: idle ones first, new ones for the rest
            const int need = (int)queue_.size() - idle_;
            for (int i = 0; i < need && (int)workers_.size() < kMaxWorkers; ++i)
                workers_.emplace_back(new std::thread([this] { loop(); }));
        }
        cv_.notify_all();
        f(0);
        // help with whatever is still queued (ours or not) instead of sleeping, then wait for our tasks in flight
        for (;;) {
            std::function<void()> task;
            {
                std::lock_guard<std::mutex> lk(mu_);
                if (queue_.empty()) break;
                task = std::move(queue_.front());
                queue_.pop_front();
            }
            task();
        }
        std::unique_lock<std::mutex> g(j.m);
        j.c.wait(g, [&] { return j.left == 0; });
    }

private:
    static constexpr int kMaxWorkers = 256;
    void loop() {
        for (;;) {
            std::function<void()> task;
            {
                std::unique_lock<std::mutex> lk(mu_);
                ++idle_;
                cv_.wait(lk, [&] { return !queue_.empty(); });
                --idle_;
                task = std::move(queue_.front());
                queue_.pop_front();
            }
            task();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<std::function<void()>> queue_;
    std::vector<std::unique_ptr<std::thread>> workers_;
    int idle_ = 0;
    pid_t owner_ = getpid();
};

template <class F> void parallel_for(int threads, F f) {  // f(thread index)
    if (threads <= 1) { f(0); return; }
    if (getenv("KBBQ_FASTQ_NO_POOL")) {   // a thread per index, as before the pool
        std::vector<std::thread> pool;
        pool.reserve(threads);
        for (int t = 0; t < threads; ++t) pool.emplace_back(f, t);
        for (auto &th : pool) th.join();
        return;
    }
    WorkerPool::get().run(threads - 1, f);
}

inline const char *line_end(const char *p, const char *end) {
    const char *nl = (const char *)memchr(p, '\n', (size_t)(end - p));
    return nl ? nl : end;
}

// the four lines of the record starting at p: [h0,h1) header without '@', [s0,s1) sequence, [q0,q1) quality
struct Rec { const char *h0, *h1, *s0, *s1, *q0, *q1; bool ok; };
inline Rec parse_record(const char *p, const char *end) {
    Rec r{};
    const char *e = line_end(p, end);
    r.ok = p < end && *p == '@';
    r.h0 = p + 1; r.h1 = e;
    p = e < end ? e + 1 : end;
    e = line_end(p, end);
    r.s0 = p; r.s1 = e;
    p = e < end ? e + 1 : end;
    e = line_end(p, end);
    r.ok = r.ok && p < end && *p == '+';
    p = e < end ? e + 1 : end;
    e = line_end(p, end);
    r.q0 = p; r.q1 = e;
    if (r.h1 > r.h0 && r.h1[-1] == '\r') --r.h1;
    if (r.s1 > r.s0 && r.s1[-1] == '\r') --r.s1;
    if (r.q1 > r.q0 && r.q1[-1] == '\r') --r.q1;
    return r;
}

// only the header line of the record starting at p: [h0, h1) without '@' and line end.  What the name-only loops
// (read-group inference, name check) need: parse_record would scan the two long lines of every record as well.
struct Hdr { const char *h0, *h1; };
inline Hdr parse_header(const char *p, const char *end) {
    Hdr r;
    r.h0 = p + 1;
    r.h1 = line_end(p, end);
    if (r.h1 > r.h0 && r.h1[-1] == '\r') --r.h1;
    return r;
}

// name = header up to the first whitespace (pysam's FastxRecord.name)
inline const char *name_end(const char *h0, const char *h1) {
    const char *p = h0;
    while (p < h1 && *p != ' ' && *p != '\t') ++p;
    return p;
}

// The usual file: every record is "@header LF, L bases LF, + LF, L qualities LF".  Once L is known from the first
// record only the header lines have to be scanned: a record that starts at p ends at (end of its header) + 2 L + 5,
// and the three line ends in between sit at fixed offsets.  Every thread finds the first record of its share of the
// bytes (a line that starts with '@' and passes the fixed-offset checks: a quality line that starts with '@' fails
// them, its "+" would have to be the first base of the next record), walks its records, and the walks have to meet:
// thread t must stop exactly where thread t + 1 started.  Anything unusual (CR LF, reads of different lengths,
// multi-line records, a malformed record) -> false, and build_index falls back to the general scan below, which
// also produces the error codes.
bool index_uniform_records(kbbq_fastq *f, int threads) {
    const char *d = f->data;
    const size_t len = f->len;
    if (len < 8 || d[0] != '@') return false;
    const char *end = d + len;
    const char *h1 = (const char *)memchr(d, '\n', len);
    if (!h1) return false;
    const char *s1 = (const char *)memchr(h1 + 1, '\n', (size_t)(end - h1 - 1));
    if (!s1) return false;
    const int64_t L = s1 - h1 - 1;
    if (L < 1) return false;
    // p -> a record?  *next = start of the following record
    auto record_at = [&](const char *p, const char **next) -> bool {
        if (p >= end || *p != '@') return false;
        const char *h = (const char *)memchr(p, '\n', (size_t)(end - p));
        if (!h || h[-1] == '\r') return false;
        const char *last = h + 2 * L + 4;   // the LF behind the qualities (or the end of a file without one)
        if (last > end) return false;
        if (h[L + 1] != '\n' || h[L + 2] != '+' || h[L + 3] != '\n' || h[L] == '\r') return false;
        if (last < end && *last != '\n') return false;
        if (last == end && end[-1] == '\n') return false;   // a short last record
        *next = last < end ? last + 1 : end;
        return true;
    };
    const int T = n_threads(threads, (int64_t)(len >> 20) + 1);
    std::vector<std::vector<int64_t>> starts(T);
    std::vector<const char *> first(T, nullptr), stop(T, nullptr);
    std::vector<int> bad(T, 0);
    parallel_for(T, [&](int t) {
        const char *lo = d + len * (size_t)t / (size_t)T, *hi = d + len * (size_t)(t + 1) / (size_t)T;
        const char *p = lo, *next = nullptr;
        if (t > 0) {   // first line start in [lo, hi) that is a record
            p = nullptr;
            const char *q = lo - 1;
            // a record is at most one header + 2 L + 5 bytes away; give up (empty share) at hi
            while (q < hi) {
                const char *nl = (const char *)memchr(q, '\n', (size_t)(hi - q));
                if (!nl || nl + 1 >= hi) break;
                if (nl[1] == '@' && record_at(nl + 1, &next)) { p = nl + 1; break; }
                q = nl + 1;
            }
            if (!p) { first[t] = stop[t] = nullptr; return; }   // no record starts in this share
        }
        first[t] = p;
        std::vector<int64_t> &v = starts[t];
        v.reserve((size_t)(hi - p) / (size_t)(2 * L + 8) + 16);
        while (p < hi) {
            if (!record_at(p, &next)) { bad[t] = 1; return; }
            v.push_back((int64_t)(p - d));
            p = next;
        }
        stop[t] = p;
    });
    // the walks must meet
    const char *expect = d;
    int64_t n = 0;
    for (int t = 0; t < T; ++t) {
        if (bad[t]) return false;
        if (!first[t]) continue;
        if (first[t] != expect) return false;
        expect = stop[t];
        n += (int64_t)starts[t].size();
    }
    if (expect != end || n == 0) return false;
    f->n = n;
    f->L = (int)L;
    f->rec.resize((size_t)n + 1);
    std::vector<int64_t> base(T + 1, 0);
    for (int t = 0; t < T; ++t) base[t + 1] = base[t] + (int64_t)starts[t].size();
    parallel_for(T, [&](int t) {
        if (!starts[t].empty()) memcpy(f->rec.data() + base[t], starts[t].data(), starts[t].size() * sizeof(int64_t));
    });
    f->rec[(size_t)n] = (int64_t)len;
    return true;
}

int build_index(kbbq_fastq *f, int threads) {
    const char *d = f->data;
    size_t len = f->len;
    // blank lines at the end of the file are not records (pysam ignores them)
    while (len >= 2 && d[len - 1] == '\n' && (d[len - 2] == '\n' || (d[len - 2] == '\r' && len >= 3 && d[len - 3] == '\n'))) {
        len -= d[len - 2] == '\r' ? 2 : 1;
    }
    while (len > 0 && len == 1 && (d[0] == '\n' || d[0] == '\r')) len = 0;
    f->len = len;
    if (len == 0) { f->n = 0; f->L = 0; f->rec.assign(1, 0); return KBBQ_OK; }
    if (!getenv("KBBQ_FASTQ_GENERAL_INDEX") && index_uniform_records(f, threads)) return KBBQ_OK;
    const int T = n_threads(threads, (int64_t)(len >> 20) + 1);
    std::vector<int64_t> lines(T + 1, 0);
    auto lo = [&](int t) { return len * (size_t)t / (size_t)T; };
    // one scan: every thread notes where the newlines of its share are; the line numbers follow from a prefix sum
    std::vector<std::vector<int64_t>> nls(T);
    parallel_for(T, [&](int t) {
        std::vector<int64_t> &v = nls[t];
        const char *p = d + lo(t), *e = d + lo(t + 1);
        v.reserve((size_t)(e - p) / 64 + 16);
        while (p < e) {
            const char *nl = (const char *)memchr(p, '\n', (size_t)(e - p));
            if (!nl) break;
            v.push_back((int64_t)(nl - d));
            p = nl + 1;
        }
        lines[t + 1] = (int64_t)v.size();
    });
    for (int t = 0; t < T; ++t) lines[t + 1] += lines[t];
    int64_t total = lines[T] + (d[len - 1] != '\n' ? 1 : 0);  // last line without a newline
    if (total % 4) return KBBQ_E_FORMAT;
    f->n = total / 4;
    f->rec.assign((size_t)f->n + 1, (int64_t)len);
    // line k starts after the k-th newline; record i starts at line 4 i
    f->rec[0] = 0;
    parallel_for(T, [&](int t) {
        int64_t k = lines[t];  // newlines before this share
        for (const int64_t pos : nls[t]) {
            ++k;  // the line after this newline has index k
            if ((k & 3) == 0 && k / 4 < f->n) f->rec[(size_t)(k / 4)] = pos + 1;
        }
        std::vector<int64_t>().swap(nls[t]);
    });
    // uniform length?
    const Rec r0 = parse_record(d + f->rec[0], d + f->rec[1]);
    if (!r0.ok) return KBBQ_E_FORMAT;
    f->L = (int)(r0.s1 - r0.s0);
    const int T2 = n_threads(threads, f->n);
    std::vector<int> state(T2, 0);  // 1 = format error, 2 = ragged
    parallel_for(T2, [&](int t) {
        const int64_t a = f->n * t / T2, b = f->n * (t + 1) / T2;
        const int64_t L0 = f->L;
        for (int64_t i = a; i < b; ++i) {
            const char *p = d + f->rec[(size_t)i], *e = d + f->rec[(size_t)i + 1];
            // the usual record: header line, then exactly L bases, "+", L qualities, LF line ends -- checked at fixed
            // offsets without scanning the two long lines again
            const char *h1 = (const char *)memchr(p, '\n', (size_t)(e - p));
            if (h1 && *p == '@' && e - h1 == 2 * L0 + 5 && h1[L0 + 1] == '\n' && h1[L0 + 2] == '+' && h1[L0 + 3] == '\n' &&
                e[-1] == '\n' && !memchr(h1 + 1, '\r', 1) && h1[L0] != '\r')
                continue;
            const Rec r = parse_record(p, e);
            if (!r.ok || (r.s1 - r.s0) != (r.q1 - r.q0)) { state[t] |= 1; return; }
            if ((int)(r.s1 - r.s0) != f->L) state[t] |= 2;
        }
    });
    int st = 0;
    for (int v : state) st |= v;
    if (st & 1) return KBBQ_E_FORMAT;
    if (st & 2) f->L = -1;
    return KBBQ_OK;
}

bool ends_with(const std::string &s, const char *suf) {
    const size_t n = strlen(suf);
    return s.size() >= n && s.compare(s.size() - n, n, suf) == 0;
}

}  // namespace

extern "C" {

int kbbq_fastq_open_mem(const void *data, size_t len, int threads, kbbq_fastq **out) {
    if (!out || (!data && len)) return KBBQ_E_ARG;
    kbbq_fastq *f = new kbbq_fastq;
    f->data = (const char *)data;
    f->len = len;
    const int rc = build_index(f, threads);
    if (rc) { delete f; return rc; }
    *out = f;
    return KBBQ_OK;
}

// everything a descriptor yields (pipes, process substitution, files that cannot be mapped)
static int read_all(int fd, std::vector<char> &buf) {
    size_t used = 0;
    for (;;) {
        if (buf.size() - used < (1u << 22)) buf.resize(std::max<size_t>(buf.size() * 2, 1u << 24));
        const ssize_t got = read(fd, buf.data() + used, buf.size() - used);
        if (got < 0) return KBBQ_E_IO;
        if (got == 0) break;
        used += (size_t)got;
    }
    buf.resize(used);
    return KBBQ_OK;
}

int kbbq_fastq_open(const char *path, int threads, kbbq_fastq **out) {
    if (!path || !out) return KBBQ_E_ARG;
    kbbq_fastq *f = new kbbq_fastq;
    // gzip by its magic bytes (pysam's FastxFile does not look at the suffix either); a pipe cannot be sniffed
    // without consuming it, so there the suffix decides.  The path is opened once: a named pipe opened a second time
    // waits for a writer that may have given up when the first reader closed it.
    bool gz = ends_with(path, ".gz");
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { delete f; return KBBQ_E_IO; }
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); delete f; return KBBQ_E_IO; }
    if (S_ISREG(st.st_mode)) {
        unsigned char magic[2] = {0, 0};
        gz = pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
    }
    if (gz) {
        gzFile g = gzdopen(fd, "rb");   // closes fd
        if (!g) { close(fd); delete f; return KBBQ_E_IO; }
        gzbuffer(g, 1 << 20);
        std::vector<char> &buf = f->owned;
        size_t used = 0;
        for (;;) {
            if (buf.size() - used < (1u << 22)) buf.resize(std::max<size_t>(buf.size() * 2, 1u << 24));
            const int got = gzread(g, buf.data() + used, (unsigned)std::min<size_t>(buf.size() - used, 1u << 30));
            if (got < 0) { gzclose(g); delete f; return KBBQ_E_IO; }
            if (got == 0) break;
            used += (size_t)got;
        }
        gzclose(g);
        buf.resize(used);
        f->data = buf.data();
        f->len = used;
    } else {
        void *m = MAP_FAILED;
        if (S_ISREG(st.st_mode) && st.st_size > 0) m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m != MAP_FAILED) {
            madvise(m, (size_t)st.st_size, MADV_SEQUENTIAL);
            f->map = m;
            f->map_len = (size_t)st.st_size;
            f->data = (const char *)m;
            f->len = (size_t)st.st_size;
        } else if (!S_ISREG(st.st_mode) || st.st_size > 0) {   // a pipe, or a file that cannot be mapped
            if (read_all(fd, f->owned) != KBBQ_OK) { close(fd); delete f; return KBBQ_E_IO; }
            f->data = f->owned.data();
            f->len = f->owned.size();
        }
        close(fd);
    }
    const int rc = build_index(f, threads);
    if (rc) { kbbq_fastq_close(f); return rc; }
    *out = f;
    return KBBQ_OK;
}

void kbbq_fastq_close(kbbq_fastq *f) {
    if (!f) return;
    if (f->map) munmap(f->map, f->map_len);
    delete f;
}

int64_t kbbq_fastq_num_reads(const kbbq_fastq *f) { return f ? f->n : -1; }
int kbbq_fastq_read_len(const kbbq_fastq *f) { return f ? f->L : -1; }

int kbbq_fastq_pack(const kbbq_fastq *f, int64_t first, int64_t n, uint8_t *seq, uint8_t *qual, int threads) {
    if (!f || first < 0 || n < 0 || first + n > f->n || (n && !seq)) return KBBQ_E_ARG;   // qual may be NULL (bases only)
    if (f->L < 0) return KBBQ_E_RAGGED;
    const int L = f->L;
    const int T = n_threads(threads, n);
    std::vector<int> bad(T, 0);
    parallel_for(T, [&](int t) {
        const int64_t a = n * t / T, b = n * (t + 1) / T;
        unsigned low = 0;  // thread-local: a shared flag array would bounce its cache line on every base
        for (int64_t i = a; i < b; ++i) {
            const size_t ri = (size_t)(first + i);
            // the index already checked the record: '@' line, sequence, '+' line, quality of L bytes each
            const char *s0 = (const char *)memchr(f->data + f->rec[ri], '\n', (size_t)(f->rec[ri + 1] - f->rec[ri])) + 1;
            const char *q0 = f->data + f->rec[ri + 1] - L - 1;
            if (q0[L] != '\n' || q0[-1] != '\n') {  // no final newline, or CRLF line ends: take the slow path
                const Rec r = parse_record(f->data + f->rec[ri], f->data + f->rec[ri + 1]);
                s0 = r.s0;
                q0 = r.q0;
            }
            memcpy(seq + (size_t)i * L, s0, (size_t)L);
            if (!qual) continue;
            const uint8_t *__restrict q = (const uint8_t *)q0;
            uint8_t *__restrict o = qual + (size_t)i * L;
            unsigned m = 0xFF;
            for (int c = 0; c < L; ++c) {
                m = q[c] < m ? q[c] : m;
                o[c] = (uint8_t)(q[c] - 33);
            }
            low |= m < 33;
        }
        bad[t] = (int)low;
    });
    for (int v : bad) if (v) return KBBQ_E_FORMAT;
    return KBBQ_OK;
}

int kbbq_fastq_name(const kbbq_fastq *f, int64_t i, const char **name, int *len) {
    if (!f || i < 0 || i >= f->n || !name || !len) return KBBQ_E_ARG;
    const Hdr r = parse_header(f->data + f->rec[(size_t)i], f->data + f->rec[(size_t)i + 1]);
    *name = r.h0;
    *len = (int)(name_end(r.h0, r.h1) - r.h0);
    return KBBQ_OK;
}

int kbbq_fastq_infer(kbbq_fastq *f, int infer_rg, uint16_t *rg, uint8_t *second, int *n_rg, int threads) {
    if (!f || !rg || !second || !n_rg) return KBBQ_E_ARG;
    const int64_t n = f->n;
    const int T = n_threads(threads, n);
    std::vector<std::vector<std::string>> keys(T);
    std::vector<int> err(T, 0);
    std::vector<uint32_t> local((size_t)n);
    parallel_for(T, [&](int t) {
        const int64_t a = n * t / T, b = n * (t + 1) / T;
        std::unordered_map<std::string, uint32_t> seen;
        struct Memo { const char *p = nullptr; size_t len = 0; uint32_t id = 0; } memo[64];
        for (int64_t i = a; i < b; ++i) {
            // one header line per ~2 L bytes of file: the loop waits for memory, not for the scan -- fetch ahead
            if (i + 16 < b) __builtin_prefetch(f->data + f->rec[(size_t)i + 16]);
            const Hdr r = parse_header(f->data + f->rec[(size_t)i], f->data + f->rec[(size_t)i + 1]);
            const char *h1 = name_end(r.h0, r.h1);
            // first '_' field: second in pair <=> it ends in "/2" (kbbq/compare_reads.py:304-306)
            const char *u = (const char *)memchr(r.h0, '_', (size_t)(h1 - r.h0));
            const char *f0e = u ? u : h1;
            second[i] = (f0e - r.h0 >= 2 && f0e[-2] == '/' && f0e[-1] == '2') ? 1 : 0;
            if (!infer_rg) { local[(size_t)i] = 0; continue; }
            // second '_' field must exist and start with "RG"; key = text after its last ':' (:308-318)
            if (!u) { err[t] |= 1; return; }  // IndexError in the reference
            const char *f1 = u + 1;
            const char *u2 = (const char *)memchr(f1, '_', (size_t)(h1 - f1));
            const char *f1e = u2 ? u2 : h1;
            if (f1e - f1 < 2 || f1[0] != 'R' || f1[1] != 'G') { err[t] |= 2; return; }  // AssertionError
            const char *k = f1e;
            while (k > f1 && k[-1] != ':') --k;
            // a file has a handful of read groups: a small direct-mapped memo in front of the map (no string is built,
            // nothing is hashed twice) answers all but the first read of each
            const size_t klen = (size_t)(f1e - k);
            uint32_t h = 2166136261u;
            for (size_t c = 0; c < klen; ++c) h = (h ^ (uint8_t)k[c]) * 16777619u;
            Memo &m = memo[(h ^ (h >> 16)) & 63u];
            if (m.p && m.len == klen && memcmp(m.p, k, klen) == 0) { local[(size_t)i] = m.id; continue; }
            std::string key(k, klen);
            auto it = seen.find(key);
            if (it == seen.end()) {
                it = seen.emplace(key, (uint32_t)keys[t].size()).first;
                keys[t].push_back(key);
            }
            m.p = k; m.len = klen; m.id = it->second;
            local[(size_t)i] = it->second;
        }
    });
    int e = 0;
    for (int v : err) e |= v;
    if (e & 1) return KBBQ_E_NAME_FIELD;
    if (e & 2) return KBBQ_E_NAME_RG;
    f->rg_keys.clear();
    if (!infer_rg) {
        std::fill(rg, rg + n, (uint16_t)0);
        *n_rg = 1;
        return KBBQ_OK;
    }
    // first-seen order over the file = thread order, then each thread's own first-seen order
    std::unordered_map<std::string, uint32_t> global;
    std::vector<std::vector<uint32_t>> remap(T);
    for (int t = 0; t < T; ++t) {
        remap[t].resize(keys[t].size());
        for (size_t k = 0; k < keys[t].size(); ++k) {
            auto it = global.find(keys[t][k]);
            if (it == global.end()) {
                it = global.emplace(keys[t][k], (uint32_t)f->rg_keys.size()).first;
                f->rg_keys.push_back(keys[t][k]);
            }
            remap[t][k] = it->second;
        }
    }
    if (f->rg_keys.size() > 65535) return KBBQ_E_ARG;
    parallel_for(T, [&](int t) {
        const int64_t a = n * t / T, b = n * (t + 1) / T;
        for (int64_t i = a; i < b; ++i) rg[i] = (uint16_t)remap[t][local[(size_t)i]];
    });
    *n_rg = (int)std::max<size_t>(1, f->rg_keys.size());
    return KBBQ_OK;
}

int kbbq_fastq_rg_key(const kbbq_fastq *f, int k, const char **key, int *len) {
    if (!f || k < 0 || (size_t)k >= f->rg_keys.size() || !key || !len) return KBBQ_E_ARG;
    *key = f->rg_keys[(size_t)k].data();
    *len = (int)f->rg_keys[(size_t)k].size();
    return KBBQ_OK;
}

int kbbq_fastq_check_names(const kbbq_fastq *uncorr, const kbbq_fastq *corr, int64_t n, int threads,
                           int64_t *first_bad) {
    if (!uncorr || !corr || n < 0 || n > uncorr->n || n > corr->n) return KBBQ_E_ARG;
    const int T = n_threads(threads, n);
    std::vector<int64_t> bad(T, -1);
    parallel_for(T, [&](int t) {
        const int64_t a = n * t / T, b = n * (t + 1) / T;
        for (int64_t i = a; i < b; ++i) {
            if (i + 16 < b) {
                __builtin_prefetch(uncorr->data + uncorr->rec[(size_t)i + 16]);
                __builtin_prefetch(corr->data + corr->rec[(size_t)i + 16]);
            }
            const Hdr u = parse_header(uncorr->data + uncorr->rec[(size_t)i], uncorr->data + uncorr->rec[(size_t)i + 1]);
            const Hdr c = parse_header(corr->data + corr->rec[(size_t)i], corr->data + corr->rec[(size_t)i + 1]);
            const size_t ul = (size_t)(name_end(u.h0, u.h1) - u.h0), cl = (size_t)(name_end(c.h0, c.h1) - c.h0);
            if (cl < ul || memcmp(u.h0, c.h0, ul) != 0) { bad[t] = i; return; }  // corr.name.startswith(uncorr.name)
        }
    });
    for (int64_t v : bad)
        if (v >= 0) {
            if (first_bad) *first_bad = v;
            return KBBQ_E_NAME_MISMATCH;
        }
    return KBBQ_OK;
}

int kbbq_fastq_format_size(const kbbq_fastq *f, int64_t first, int64_t n, int threads, int64_t *bytes) {
    if (!f || first < 0 || n < 0 || first + n > f->n || !bytes) return KBBQ_E_ARG;
    if (f->L < 0) return KBBQ_E_RAGGED;
    const int L = f->L;
    const int T = n_threads(threads, (n >> 12) + 1);
    std::vector<int64_t> part(T, 0);
    parallel_for(T, [&](int t) {  // names vary, the rest is 2 L + 6 per record
        const int64_t a = n * t / T, b = n * (t + 1) / T;
        int64_t sum = 0;
        for (int64_t i = a; i < b; ++i) {
            const char *h0 = f->data + f->rec[(size_t)(first + i)] + 1;
            const char *h1 = line_end(h0, f->data + f->rec[(size_t)(first + i) + 1]);
            sum += (int64_t)(name_end(h0, h1) - h0) + 2 * (int64_t)L + 6;
        }
        part[t] = sum;
    });
    *bytes = 0;
    for (int64_t v : part) *bytes += v;
    return KBBQ_OK;
}

// one record: '@' name '\n' seq '\n+\n' (q + 33) '\n'; returns the byte after it
static inline char *format_record(const kbbq_fastq *f, size_t ri, const uint8_t *__restrict q, int L, char *__restrict w) {
    const char *p = f->data + f->rec[ri], *e = f->data + f->rec[ri + 1];
    const char *h0 = p + 1, *h1 = (const char *)memchr(p, '\n', (size_t)(e - p)), *s0;
    if (h1 && e - h1 >= 2 * (int64_t)L + 4 && h1[-1] != '\r') {
        s0 = h1 + 1;   // LF line ends: the bases follow the header line (the index checked the record)
    } else {
        const Rec r = parse_record(p, e);
        h0 = r.h0; h1 = r.h1; s0 = r.s0;
    }
    const size_t nl = (size_t)(name_end(h0, h1) - h0);
    *w++ = '@';
    memcpy(w, h0, nl); w += nl;   // the comment is dropped (kbbq/recalibrate.py:153)
    *w++ = '\n';
    memcpy(w, s0, (size_t)L); w += L;
    *w++ = '\n'; *w++ = '+'; *w++ = '\n';
    for (int c = 0; c < L; ++c) w[c] = (char)(q[c] + 33);
    w[L] = '\n';
    return w + L + 1;
}

int kbbq_fastq_format(const kbbq_fastq *f, int64_t first, int64_t n, const uint8_t *out_qual, char *dst, int64_t dst_bytes,
                      int threads) {
    if (!f || first < 0 || n < 0 || first + n > f->n || (n && (!out_qual || !dst))) return KBBQ_E_ARG;
    if (f->L < 0) return KBBQ_E_RAGGED;
    const int L = f->L;
    const int T = n_threads(threads, (n >> 12) + 1);
    std::vector<int64_t> bytes(T + 1, 0);
    parallel_for(T, [&](int t) {
        const int64_t a = n * t / T, b = n * (t + 1) / T;
        int64_t sum = 0;
        for (int64_t i = a; i < b; ++i) {
            const char *h0 = f->data + f->rec[(size_t)(first + i)] + 1;
            const char *h1 = line_end(h0, f->data + f->rec[(size_t)(first + i) + 1]);
            sum += (int64_t)(name_end(h0, h1) - h0) + 2 * (int64_t)L + 6;
        }
        bytes[t + 1] = sum;
    });
    for (int t = 0; t < T; ++t) bytes[t + 1] += bytes[t];
    if (bytes[T] != dst_bytes) return KBBQ_E_ARG;
    parallel_for(T, [&](int t) {
        const int64_t a = n * t / T, b = n * (t + 1) / T;
        char *w = dst + bytes[t];
        for (int64_t i = a; i < b; ++i) w = format_record(f, (size_t)(first + i), out_qual + (size_t)i * L, L, w);
    });
    return KBBQ_OK;
}

int kbbq_fastq_write(int fd, const kbbq_fastq *f, int64_t first, int64_t n, const uint8_t *out_qual, int threads) {
    if (!f || fd < 0 || first < 0 || n < 0 || first + n > f->n || (n && !out_qual)) return KBBQ_E_ARG;
    if (f->L < 0) return KBBQ_E_RAGGED;
    const int L = f->L;
    const int T = n_threads(threads, (n >> 12) + 1);
    const int64_t wave = 1 << 15;  // reads per thread and wave: bounds the formatting buffers
    std::vector<std::vector<char>> buf(T);

    // A regular file (stdout redirected, not a pipe, not O_APPEND): the records are formatted straight into a shared
    // mapping of the output file, every thread its own contiguous share.  write() / pwrite() on ONE file serialise
    // on the inode lock however many threads call them (3 - 4 GB/s into a tmpfs); page faults on a mapping do not.
    // The descriptor is usually write-only (shell redirection), so the file is reopened read-write through /proc.
    const off_t pos0 = lseek(fd, 0, SEEK_CUR);
    const int fl = fcntl(fd, F_GETFL);
    struct stat st;
    if (pos0 >= 0 && fl >= 0 && !(fl & O_APPEND) && T > 1 && n > 0 && fstat(fd, &st) == 0 && S_ISREG(st.st_mode) &&
        !getenv("KBBQ_FASTQ_NO_MMAP")) {
        int64_t total = 0;
        int rc = kbbq_fastq_format_size(f, first, n, threads, &total);
        if (rc) return rc;
        char link[64];
        snprintf(link, sizeof(link), "/proc/self/fd/%d", fd);
        const int rw = open(link, O_RDWR);
        if (rw >= 0) {
            const long page = sysconf(_SC_PAGESIZE);
            const off_t base = pos0 / page * page;
            const size_t span = (size_t)(pos0 - base) + (size_t)total;
            // the file only grows: bytes already behind the records stay, as write() leaves them
            void *m = MAP_FAILED;
            const off_t end = pos0 + (off_t)total;
            if (end <= st.st_size || ftruncate(rw, end) == 0) m = mmap(nullptr, span, PROT_READ | PROT_WRITE, MAP_SHARED, rw, base);
            close(rw);
            if (m != MAP_FAILED) {
                rc = kbbq_fastq_format(f, first, n, out_qual, (char *)m + (pos0 - base), total, threads);
                munmap(m, span);
                if (rc) return rc;
                if (lseek(fd, pos0 + (off_t)total, SEEK_SET) < 0) return KBBQ_E_IO;
                return KBBQ_OK;
            }
        }
    }

    // A seekable descriptor that cannot be mapped: every thread formats its own contiguous share of the reads and
    // writes it at its own offset.
    if (pos0 >= 0 && fl >= 0 && !(fl & O_APPEND) && T > 1) {
        std::vector<int64_t> bytes(T + 1, 0);
        parallel_for(T, [&](int t) {  // size of every share: names vary, the rest is 2 L + 6 per record
            const int64_t a = n * t / T, b = n * (t + 1) / T;
            int64_t sum = 0;
            for (int64_t i = a; i < b; ++i) {
                const char *h0 = f->data + f->rec[(size_t)(first + i)] + 1;
                const char *h1 = line_end(h0, f->data + f->rec[(size_t)(first + i) + 1]);
                sum += (int64_t)(name_end(h0, h1) - h0) + 2 * (int64_t)L + 6;
            }
            bytes[t + 1] = sum;
        });
        for (int t = 0; t < T; ++t) bytes[t + 1] += bytes[t];
        std::vector<int> failed(T, 0);
        parallel_for(T, [&](int t) {
            const int64_t a = n * t / T, b = n * (t + 1) / T;
            off_t at = pos0 + (off_t)bytes[t];
            std::vector<char> &o = buf[t];
            for (int64_t c0 = a; c0 < b; c0 += 4096) {
                const int64_t c1 = std::min(b, c0 + 4096);
                int64_t need = 0;
                for (int64_t i = c0; i < c1; ++i) {
                    const char *h0 = f->data + f->rec[(size_t)(first + i)] + 1;
                    const char *h1 = line_end(h0, f->data + f->rec[(size_t)(first + i) + 1]);
                    need += (int64_t)(name_end(h0, h1) - h0) + 2 * (int64_t)L + 6;
                }
                o.resize((size_t)need);
                char *w = o.data();
                for (int64_t i = c0; i < c1; ++i) w = format_record(f, (size_t)(first + i), out_qual + (size_t)i * L, L, w);
                const char *p = o.data();
                size_t left = o.size();
                while (left) {
                    const ssize_t k = pwrite(fd, p, left, at);
                    if (k < 0) { failed[t] = 1; return; }
                    p += k; at += k; left -= (size_t)k;
                }
            }
        });
        for (int v : failed) if (v) return KBBQ_E_IO;
        if (lseek(fd, pos0 + (off_t)bytes[T], SEEK_SET) < 0) return KBBQ_E_IO;
        return KBBQ_OK;
    }

    for (int64_t base = 0; base < n; base += wave * T) {
        parallel_for(T, [&](int t) {
            const int64_t a = std::min(n, base + wave * t), b = std::min(n, a + wave);
            std::vector<char> &o = buf[t];
            o.clear();
            for (int64_t i = a; i < b; ++i) {
                const size_t ri = (size_t)(first + i);
                const Rec r = parse_record(f->data + f->rec[ri], f->data + f->rec[ri + 1]);
                const size_t nl = (size_t)(name_end(r.h0, r.h1) - r.h0);
                const size_t at = o.size();
                o.resize(at + nl + 2 * (size_t)L + 6);
                char *w = o.data() + at;
                *w++ = '@';
                memcpy(w, r.h0, nl); w += nl;  // the comment is dropped (kbbq/recalibrate.py:153)
                *w++ = '\n';
                memcpy(w, r.s0, (size_t)L); w += L;
                *w++ = '\n'; *w++ = '+'; *w++ = '\n';
                const uint8_t *q = out_qual + (size_t)i * L;
                for (int c = 0; c < L; ++c) w[c] = (char)(q[c] + 33);
                w[L] = '\n';
            }
        });
        for (int t = 0; t < T; ++t) {
            const char *p = buf[t].data();
            size_t left = buf[t].size();
            while (left) {
                const ssize_t k = write(fd, p, left);
                if (k < 0) return KBBQ_E_IO;
                p += k;
                left -= (size_t)k;
            }
        }
    }
    return KBBQ_OK;
}

}  // extern "C"
