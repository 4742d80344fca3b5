// kmer.cuh -- sequencing errors from the reads' own k-mer spectrum (kbbq_kmer_*, include/kbbq_b200.h).
//
// The rule (DESIGN.md, "Errors from k-mer counts"): a window of k bases is valid when all of them are A/C/G/T; its key
// is the smaller of its forward and reverse-complement 2-bit codes (first base in the most significant bits).  count(x)
// is the number of valid windows of the batch with key x; a window is solid when count >= t.  A base is uncovered when
// no solid window covers it; in every maximal run [a, b] of uncovered bases, an inner run flags a and b, a run at the
// read start flags b, a run at the read end flags a, and a run that is the whole read (no solid window) flags nothing.
// A flagged byte that is not A/C/G/T is not flagged.
//
// Table: open addressing over `capacity` (a power of two) 16-byte slots {u64 key, u64 count}, empty key = all ones
// (keys have 62 bits, so it cannot occur), home slot = splitmix64(key) & (capacity - 1), linear probing.  Insert: CAS
// the key into an empty slot, then add 1 to the count -- one 32-byte sector per probe.  A probe that has walked the
// whole table raises KBBQ_FLAG_KMER_FULL and gives up.  The counts, and so the flags, do not depend on where a key
// lands, so any schedule gives the same bits.
//
// Sieved table (DESIGN.md §10, "Streaming"): the same slots, filled in two passes over all reads so that the table
// only has to hold the keys seen at least twice.  Pass A (kmer_sieve_kernel) ORs a pattern of bits into ONE 64-bit
// word of a filter per window and inserts the key with count 0 when the word already held the whole pattern; the
// occurrences of a key meet at one word and the atomics on it are serialised, so every occurrence after the first sees
// the full pattern: every key with count >= 2 is in the table, whatever the schedule (a key seen once lands there only
// through a false positive).  Pass B (kmer_count_present_kernel) adds 1 to the keys present and counts the valid
// windows W.  Then h[c] for c >= 2 is binned from the table and h[1] = W - sum of the counts >= 2
// (kmer_hist_sieved_kernel + kmer_hist_tail_kernel): the exact histogram, so the exact threshold and, for t >= 2,
// the exact flags from the unchanged kmer_flag_kernel (an absent key has count <= 1 < t); t = 1 needs no lookup.
//
// The correcting walk (kmer_correct_kernel, below; DESIGN.md §10): an opt-in second rule on the same table that finds
// every error of a cluster and those at read ends by correcting each read against its trusted k-mers.
//
// Several GPUs (the _part / _parts kernels; DESIGN.md §10, "Several GPUs"): the sieved table split by key into
// partitions, each filled by the same two passes restricted to the keys it owns, and looked up in the owner's table.
#pragma once
#include "common.cuh"

namespace kbbq {

constexpr unsigned long long KMER_EMPTY = ~0ull;

__device__ __forceinline__ unsigned long long kmer_mix(unsigned long long x) {   // splitmix64 finaliser
    x ^= x >> 30;
    x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27;
    x *= 0x94D049BB133111EBull;
    x ^= x >> 31;
    return x;
}

// A=0 C=1 G=2 T=3, anything else (N, lowercase) -1
__device__ __forceinline__ int kmer_code(uint8_t b) {
    return b == 'A' ? 0 : b == 'C' ? 1 : b == 'G' ? 2 : b == 'T' ? 3 : -1;
}

// Rolling codes of the window that ends at the base just pushed.  valid() once the last k bases were all A/C/G/T.
struct KmerRoll {
    unsigned long long fwd = 0, rc = 0, mask;
    int shift, k, run = 0;
    __device__ KmerRoll(int k_) : mask((1ull << (2 * k_)) - 1), shift(2 * (k_ - 1)), k(k_) {}
    __device__ __forceinline__ void push(uint8_t b) {
        const int c = kmer_code(b);
        if (c < 0) { run = 0; return; }
        fwd = ((fwd << 2) | (unsigned)c) & mask;
        rc = (rc >> 2) | ((unsigned long long)(3 - c) << shift);
        ++run;
    }
    __device__ __forceinline__ bool valid() const { return run >= k; }
    __device__ __forceinline__ unsigned long long key() const { return fwd < rc ? fwd : rc; }
};

__global__ void kmer_clear_kernel(ulonglong2 *table, unsigned long long capacity) {
    for (unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; s < capacity;
         s += (unsigned long long)gridDim.x * blockDim.x)
        table[s] = make_ulonglong2(KMER_EMPTY, 0ull);
}

// One thread per read: roll the codes along the read, one insert per valid window.  Counts accumulate.
__global__ void kmer_count_kernel(const uint8_t *seq, long long N, int L, int k, unsigned long long *table,
                                  unsigned long long mask, int *status) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= N) return;
    const uint8_t *s = seq + r * L;
    KmerRoll roll(k);
    for (int e = 0; e < L; ++e) {
        roll.push(s[e]);
        if (!roll.valid()) continue;
        const unsigned long long key = roll.key();
        unsigned long long slot = kmer_mix(key) & mask;
        bool done = false;
        for (unsigned long long p = 0; p <= mask; ++p) {
            unsigned long long *kp = table + 2 * slot;
            unsigned long long cur = __ldcg(kp);   // a key never changes once set: a stale EMPTY only costs the CAS
            if (cur == KMER_EMPTY) {
                cur = atomicCAS(kp, KMER_EMPTY, key);
                if (cur == KMER_EMPTY) cur = key;
            }
            if (cur == key) {
                atomicAdd(kp + 1, 1ull);
                done = true;
                break;
            }
            slot = (slot + 1) & mask;
        }
        if (!done) {
            atomicOr(status, KBBQ_FLAG_KMER_FULL);
            return;
        }
    }
}

// 256-bin histogram of the counts of the occupied slots (count >= 255 in bin 255), privatised in shared memory.
__global__ void kmer_hist_kernel(const ulonglong2 *table, unsigned long long capacity, unsigned long long *hist) {
    __shared__ unsigned int h[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) h[i] = 0;
    __syncthreads();
    for (unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; s < capacity;
         s += (unsigned long long)gridDim.x * blockDim.x) {
        const ulonglong2 v = __ldg(table + s);
        if (v.x != KMER_EMPTY && v.y) atomicAdd(&h[v.y < 255 ? v.y : 255], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        if (h[i]) atomicAdd(hist + i, (unsigned long long)h[i]);
}

// count of `key` in a table whose probe for it starts at `slot` (0 when absent)
__device__ __forceinline__ unsigned long long kmer_probe(const ulonglong2 *table, unsigned long long mask,
                                                         unsigned long long slot, unsigned long long key, bool *full) {
    for (unsigned long long p = 0; p <= mask; ++p) {
        const ulonglong2 v = __ldg(table + slot);
        if (v.x == key) return v.y;
        if (v.x == KMER_EMPTY) return 0;
        slot = (slot + 1) & mask;
    }
    *full = true;
    return 0;
}

__device__ __forceinline__ unsigned long long kmer_lookup(const ulonglong2 *table, unsigned long long mask,
                                                          unsigned long long key, bool *full) {
    return kmer_probe(table, mask, kmer_mix(key) & mask, key, full);
}

// ---- a table split by key across partitions (DESIGN.md §10, "Several GPUs") ----
//
// With h = kmer_mix(key) and n partitions, partition owner(key) = ((h >> 32) * n) >> 32 holds the key, at the home
// slot h & (capacity - 1) of its own table.  For n > 1 a partition has at most 2^32 slots, so the owner and the home
// slot come from disjoint bits of h; n = 1 puts every key in partition 0 and is the single table.  Passes A and B of
// partition p see every window and skip the ones it does not own before touching memory, so all occurrences of a key
// meet in its owner's filter word and table: each partition's table, counts and W_p are those of a single table fed
// only its keys, and the sum of the partitions' sieved histograms is the exact one.  A lookup reads the owner's table.
constexpr int KMER_MAX_PARTS = 16;

__device__ __forceinline__ unsigned kmer_owner(unsigned long long h, unsigned n) {   // h = kmer_mix(key)
    return (unsigned)(((h >> 32) * n) >> 32);
}

// the windows a counting pass takes: all of them (one table), or those partition `part` of `n` owns
struct KmerAllKeys {
    __device__ __forceinline__ bool owns(unsigned long long) const { return true; }
};
struct KmerOwnedKeys {
    unsigned part, n;
    __device__ __forceinline__ bool owns(unsigned long long key) const { return kmer_owner(kmer_mix(key), n) == part; }
};

// the tables a lookup reads: one table, or the partitions' tables (those of other devices are peer memory, read
// over NVLink) -- the owner and the home slot from one kmer_mix
struct KmerTable {
    const ulonglong2 *table;
    unsigned long long mask;
    __device__ __forceinline__ unsigned long long lookup(unsigned long long key, bool *full) const {
        return kmer_lookup(table, mask, key, full);
    }
};
struct KmerParts {
    const ulonglong2 *t[KMER_MAX_PARTS];
    unsigned long long mask;
    unsigned n;
    __device__ __forceinline__ unsigned long long lookup(unsigned long long key, bool *full) const {
        const unsigned long long h = kmer_mix(key);
        return kmer_probe(t[kmer_owner(h, n)], mask, h & mask, key, full);
    }
};

// One thread per read, one warp per 32 consecutive reads.  Each window's count is looked up once; base i is covered
// when the last solid window that starts at or before i starts at i - k + 1 or later (the running form of "one of the
// k windows over i is solid").  A base's coverage is final once the window that starts at it has been looked up, so
// the run rule runs one window behind the lookups.  The 32 reads of a warp are 32 L bits = L whole words of the
// map, starting at word (first read / 32) * L: the warp assembles them in shared memory and stores whole words.
// ALL_SOLID: every valid window is solid (t = 1 on a sieved table, where a key seen once may be absent); no lookups.
template <bool ALL_SOLID, class Tables>
__device__ __forceinline__ void kmer_flag_reads(const uint8_t *seq, long long N, int L, int k, Tables tables,
                                                unsigned long long t, uint32_t *bits, int *status) {
    extern __shared__ uint32_t kmer_words[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long r0 = ((long long)blockIdx.x * (blockDim.x >> 5) + warp) * 32;
    if (r0 >= N) return;
    uint32_t *wb = kmer_words + (size_t)warp * L;
    for (int w = lane; w < L; w += 32) wb[w] = 0;
    __syncwarp();
    const long long r = r0 + lane;
    if (r < N && L >= k) {
        const uint8_t *s = seq + r * L;
        const int base_bit = lane * L;
        auto flag = [&](int i) {
            if (kmer_code(s[i]) >= 0) atomicOr(&wb[(base_bit + i) >> 5], 1u << ((base_bit + i) & 31));
        };
        int last = -L - k;   // start of the last solid window so far
        int run = -1;        // start of the open uncovered run, -1: none
        auto settle = [&](int i) {   // coverage of base i is final
            if (last < i - k + 1) {
                if (run < 0) run = i;
            } else if (run >= 0) {
                if (run > 0) flag(run);   // an inner run flags both ends, one at the read start only its end
                flag(i - 1);
                run = -1;
            }
        };
        KmerRoll roll(k);
        bool full = false;
        for (int e = 0; e < L; ++e) {
            roll.push(s[e]);
            if (e < k - 1) continue;
            const int j = e - k + 1;
            if (roll.valid() && (ALL_SOLID || tables.lookup(roll.key(), &full) >= t)) last = j;
            settle(j);
        }
        for (int i = L - k + 1; i < L; ++i) settle(i);
        if (run > 0) flag(run);   // a run at the read end flags its start; a run of the whole read flags nothing
        if (full) atomicOr(status, KBBQ_FLAG_KMER_FULL);
    }
    __syncwarp();
    const long long nreads = N - r0 < 32 ? N - r0 : 32;
    const int nwords = (int)((nreads * L + 31) / 32);
    uint32_t *out = bits + (r0 / 32) * L;
    for (int w = lane; w < nwords; w += 32) out[w] = wb[w];
}

template <bool ALL_SOLID>
__global__ void kmer_flag_kernel(const uint8_t *seq, long long N, int L, int k, const ulonglong2 *table,
                                 unsigned long long mask, unsigned long long t, uint32_t *bits, int *status) {
    kmer_flag_reads<ALL_SOLID>(seq, N, L, k, KmerTable{table, mask}, t, bits, status);
}

// the boundary rule on a table split across partitions (t >= 2; t = 1 is kmer_flag_kernel<true>).  The set goes to
// the body by reference, so that it stays in parameter space (the owner's pointer is one LDC; a copy would be a local
// array); the single table goes by value, as the two parameters it was.
__global__ void kmer_flag_parts_kernel(const uint8_t *seq, long long N, int L, int k, const KmerParts tables,
                                       unsigned long long t, uint32_t *bits, int *status) {
    kmer_flag_reads<false, const KmerParts &>(seq, N, L, k, tables, t, bits, status);
}

// Filter word and bit pattern of a key for the sieve: splitmix64 of the key plus a constant, so independent of the
// home slot (splitmix64 of the key).  Word: the low bits; pattern: five bit positions from the top 30 bits.
__device__ __forceinline__ void kmer_sieve_hash(unsigned long long key, unsigned long long fmask, unsigned long long *w,
                                                unsigned long long *pattern) {
    const unsigned long long h = kmer_mix(key + 0x9E3779B97F4A7C15ull);
    *w = h & fmask;
    *pattern = (1ull << ((h >> 34) & 63)) | (1ull << ((h >> 40) & 63)) | (1ull << ((h >> 46) & 63)) |
               (1ull << ((h >> 52) & 63)) | (1ull << (h >> 58));
}

// Whether some thread has found the table full: a table without an empty slot makes every probe for an absent key
// walk all of it, so once the flag is up the passes stop probing (the host then reports KBBQ_E_DATA).
__device__ __forceinline__ bool kmer_table_full(const int *status) {
    return (*(const volatile int *)status & KBBQ_FLAG_KMER_FULL) != 0;
}

// Pass A.  One thread per read as kmer_count_kernel; per valid window one 64-bit atomicOr on one filter word, and
// when the old word held the whole pattern, the key is claimed (count 0) or found in the table.  A thread stops once
// the table is full.  Keys: the windows it takes (KmerAllKeys, or those one partition owns).
template <class Keys>
__device__ __forceinline__ void kmer_sieve_reads(const uint8_t *seq, long long N, int L, int k,
                                                 unsigned long long *filter, unsigned long long fmask,
                                                 unsigned long long *table, unsigned long long mask, int *status,
                                                 Keys keys) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= N) return;
    const uint8_t *s = seq + r * L;
    KmerRoll roll(k);
    for (int e = 0; e < L; ++e) {
        roll.push(s[e]);
        if (!roll.valid()) continue;
        const unsigned long long key = roll.key();
        if (!keys.owns(key)) continue;
        unsigned long long w, pattern;
        kmer_sieve_hash(key, fmask, &w, &pattern);
        if ((atomicOr(filter + w, pattern) & pattern) != pattern) continue;   // first sight (or so it seems)
        if (kmer_table_full(status)) return;
        unsigned long long slot = kmer_mix(key) & mask;
        bool done = false;
        for (unsigned long long p = 0; p <= mask; ++p) {
            unsigned long long *kp = table + 2 * slot;
            unsigned long long cur = __ldcg(kp);
            if (cur == KMER_EMPTY) {
                cur = atomicCAS(kp, KMER_EMPTY, key);
                if (cur == KMER_EMPTY) cur = key;
            }
            if (cur == key) {
                done = true;
                break;
            }
            slot = (slot + 1) & mask;
        }
        if (!done) {
            atomicOr(status, KBBQ_FLAG_KMER_FULL);
            return;
        }
    }
}

__global__ void kmer_sieve_kernel(const uint8_t *seq, long long N, int L, int k, unsigned long long *filter,
                                  unsigned long long fmask, unsigned long long *table, unsigned long long mask,
                                  int *status) {
    kmer_sieve_reads(seq, N, L, k, filter, fmask, table, mask, status, KmerAllKeys{});
}

// pass A of partition `part` of `n`: only the windows it owns
__global__ void kmer_sieve_part_kernel(const uint8_t *seq, long long N, int L, int k, unsigned long long *filter,
                                       unsigned long long fmask, unsigned long long *table, unsigned long long mask,
                                       int *status, unsigned part, unsigned n) {
    kmer_sieve_reads(seq, N, L, k, filter, fmask, table, mask, status, KmerOwnedKeys{part, n});
}

// Pass B.  One thread per read: a key present in the table gets 1 added, an absent one nothing (its count is <= 1).
// The valid windows of the batch are added to *windows: a warp sum, one atomic per warp.  A probe that walks the
// whole table (no empty slot: every absent key would cost `capacity` loads) raises KBBQ_FLAG_KMER_FULL, and a thread
// stops once the flag is up; W is then incomplete, but the table is reported full anyway.  Keys: as in pass A; a
// partition counts only the windows it owns, in W too.
template <class Keys>
__device__ __forceinline__ void kmer_count_present_reads(const uint8_t *seq, long long N, int L, int k,
                                                         unsigned long long *table, unsigned long long mask,
                                                         unsigned long long *windows, int *status, Keys keys) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int valid = 0;
    if (r < N) {
        const uint8_t *s = seq + r * L;
        KmerRoll roll(k);
        for (int e = 0; e < L; ++e) {
            roll.push(s[e]);
            if (!roll.valid()) continue;
            if (!keys.owns(roll.key())) continue;
            if (kmer_table_full(status)) break;   // not return: the whole warp takes part in the sum below
            ++valid;
            const unsigned long long key = roll.key();
            unsigned long long slot = kmer_mix(key) & mask;
            bool done = false;
            for (unsigned long long p = 0; p <= mask; ++p) {
                unsigned long long *kp = table + 2 * slot;
                const unsigned long long cur = __ldcg(kp);   // no key is inserted in this pass
                if (cur == key) atomicAdd(kp + 1, 1ull);
                if (cur == key || cur == KMER_EMPTY) {
                    done = true;
                    break;
                }
                slot = (slot + 1) & mask;
            }
            if (!done) {
                atomicOr(status, KBBQ_FLAG_KMER_FULL);
                break;
            }
        }
    }
    valid = __reduce_add_sync(0xffffffffu, valid);
    if ((threadIdx.x & 31) == 0 && valid) atomicAdd(windows, (unsigned long long)valid);
}

__global__ void kmer_count_present_kernel(const uint8_t *seq, long long N, int L, int k, unsigned long long *table,
                                          unsigned long long mask, unsigned long long *windows, int *status) {
    kmer_count_present_reads(seq, N, L, k, table, mask, windows, status, KmerAllKeys{});
}

// pass B of partition `part` of `n`
__global__ void kmer_count_present_part_kernel(const uint8_t *seq, long long N, int L, int k, unsigned long long *table,
                                               unsigned long long mask, unsigned long long *windows, int *status,
                                               unsigned part, unsigned n) {
    kmer_count_present_reads(seq, N, L, k, table, mask, windows, status, KmerOwnedKeys{part, n});
}

// h[c] for c >= 2 from the slots of a sieved table (count >= 255 in bin 255, as kmer_hist_kernel bins), and the sum of
// those counts, unclipped, into hist[1]; the singletons a false positive let in are not binned.  kmer_hist_tail_kernel
// then turns hist[1] into W - that sum: the number of keys seen once.
__global__ void kmer_hist_sieved_kernel(const ulonglong2 *table, unsigned long long capacity, unsigned long long *hist) {
    __shared__ unsigned int h[256];
    __shared__ unsigned long long sum;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) h[i] = 0;
    if (threadIdx.x == 0) sum = 0;
    __syncthreads();
    unsigned long long mine = 0;
    for (unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; s < capacity;
         s += (unsigned long long)gridDim.x * blockDim.x) {
        const ulonglong2 v = __ldg(table + s);
        if (v.x != KMER_EMPTY && v.y >= 2) {
            atomicAdd(&h[v.y < 255 ? v.y : 255], 1u);
            mine += v.y;
        }
    }
    for (int o = 16; o; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&sum, mine);
    __syncthreads();
    for (int i = 2 + threadIdx.x; i < 256; i += blockDim.x)
        if (h[i]) atomicAdd(hist + i, (unsigned long long)h[i]);
    if (threadIdx.x == 0 && sum) atomicAdd(hist + 1, sum);
}

__global__ void kmer_hist_tail_kernel(const unsigned long long *windows, unsigned long long *hist) {
    hist[1] = *windows - hist[1];
}

// ---- the correcting walk (kbbq_kmer_correct, DESIGN.md §10 "The correcting walk") ----
//
// The rule, per read (nw = L - k + 1 windows; L < k flags nothing); counts, keys, validity and solid (count >= t) as
// above:
//   1. solid[j] for every window of the read.  No solid window: nothing is flagged.
//   2. Anchor: the longest maximal run [a0, a1] of solid windows, the leftmost of equal ones.
//   3. Right walk over a copy w of the read, j = a1 + 1 .. nw - 1: a solid window j of w goes on to j + 1.  Otherwise
//      e = j + k - 1 (the one base of window j not in the solid window j - 1); w[e] not A/C/G/T stops the walk.  For
//      each c in A, C, G, T with c != w[e], score(c) = the number of consecutive solid windows j, j + 1, ... of w with
//      w[e] = c, at most min(k, nw - j).  e is flagged; a best score >= 1 that exactly one c reaches sets w[e] = c and
//      goes on to j + 1, anything else (a tie, no candidate) stops.
//   4. Left walk, the mirror image: j = a0 - 1 down to 0, e = j, scores over windows j, j - 1, ..., at most
//      min(k, j + 1).  The right walk changes bases >= a1 + k, the left walk bases < a0: the order does not matter.
// Every flagged base is A/C/G/T.  The bits depend only on the counts, so any schedule gives the same bits; on a sieved
// table with t >= 2 an absent key has count <= 1 < t, so it gives the exact table's bits.  With t = 1 every valid
// window is solid and nothing is flagged (the host writes a zero map and launches nothing).
//
// The kernel: one thread per read, one warp per 32 reads and the map words in shared memory, as kmer_flag_kernel.
// The first pass looks every window up once and keeps its solid bit in shared memory next to the warp's map words
// (word i of a lane at [32 i + lane]: no bank conflict) while it tracks the anchor.  The walks need no copy of the
// read: the right walk keeps the code of window j - 1 of w, a candidate's windows are that code rolled with c and then
// with the read's own bases beyond e (everything right of e is unchanged), and the left walk prepends.  A window that
// holds no corrected base reuses its first-pass bit.  After a correction the windows its score counted are known
// solid, and when that score is below k the next one is known not to be: the walk moves past them without a lookup.

// forward and reverse-complement 2-bit codes of one window, rolled at either end
struct KmerCode {
    unsigned long long fwd, rc;
    __device__ __forceinline__ void append(int c, unsigned long long kmask, int shift) {
        fwd = ((fwd << 2) | (unsigned)c) & kmask;
        rc = (rc >> 2) | ((unsigned long long)(3 - c) << shift);
    }
    __device__ __forceinline__ void prepend(int c, unsigned long long kmask, int shift) {
        fwd = (fwd >> 2) | ((unsigned long long)c << shift);
        rc = ((rc << 2) | (unsigned)(3 - c)) & kmask;
    }
    __device__ __forceinline__ unsigned long long key() const { return fwd < rc ? fwd : rc; }
};

// shared-memory words a warp of kmer_correct_kernel uses: the L map words of its 32 reads, then ceil(nw / 32) words
// of solid bits per read
__host__ __device__ __forceinline__ int kmer_correct_warp_words(int L, int k) {
    return L + (L >= k ? 32 * ((L - k + 1 + 31) >> 5) : 0);
}

template <class Tables>
__device__ __forceinline__ void kmer_correct_reads(const uint8_t *seq, long long N, int L, int k, Tables tables,
                                                   unsigned long long t, uint32_t *bits, int *status) {
    extern __shared__ uint32_t kmer_words[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long r0 = ((long long)blockIdx.x * (blockDim.x >> 5) + warp) * 32;
    if (r0 >= N) return;
    uint32_t *wb = kmer_words + (size_t)warp * kmer_correct_warp_words(L, k);
    for (int w = lane; w < L; w += 32) wb[w] = 0;
    __syncwarp();
    const long long r = r0 + lane;
    const int nw = L - k + 1;
    if (r < N && nw > 0) {
        const uint8_t *s = seq + r * L;
        const int base_bit = lane * L;
        uint32_t *sol = wb + L + lane;   // solid bit of window j: bit j & 31 of sol[32 * (j >> 5)]
        const unsigned long long kmask = (1ull << (2 * k)) - 1;
        const int shift = 2 * (k - 1);
        bool full = false;
        auto flag = [&](int i) { atomicOr(&wb[(base_bit + i) >> 5], 1u << ((base_bit + i) & 31)); };
        auto solid = [&](const KmerCode &x) { return tables.lookup(x.key(), &full) >= t; };
        auto was_solid = [&](int j) { return (sol[32 * (j >> 5)] >> (j & 31)) & 1u; };
        auto code_at = [&](int p) {   // window p of the read, all A/C/G/T
            KmerCode x{0, 0};
            for (int i = 0; i < k; ++i) x.append(kmer_code(s[p + i]), kmask, shift);
            return x;
        };

        // first pass: solid bits and the anchor
        KmerRoll roll(k);
        int a0 = 0, best = 0, run = 0;
        uint32_t word = 0;
        for (int e = 0; e < L; ++e) {
            roll.push(s[e]);
            if (e < k - 1) continue;
            const int j = e - k + 1;
            const bool ok = roll.valid() && tables.lookup(roll.key(), &full) >= t;
            word |= (uint32_t)ok << (j & 31);
            if ((j & 31) == 31 || j == nw - 1) {
                sol[32 * (j >> 5)] = word;
                word = 0;
            }
            run = ok ? run + 1 : 0;
            if (run > best) {
                best = run;
                a0 = j - run + 1;
            }
        }

        if (best > 0) {
            // right walk: x is window j - 1 of w; known_bad: window j holds the last correction and is not solid
            const int a1 = a0 + best - 1;
            KmerCode x = code_at(a1);
            bool known_bad = false;
            for (int j = a1 + 1; j < nw;) {
                const int e = j + k - 1;
                const int b = kmer_code(s[e]);
                if (!known_bad && b >= 0 && was_solid(j)) {
                    x.append(b, kmask, shift);
                    ++j;
                    continue;
                }
                if (b < 0) break;
                flag(e);
                const int m = min(k, nw - j);
                int best_c = -1, best_n = 0;
                bool tie = false;
                for (int c = 0; c < 4; ++c) {
                    if (c == b) continue;
                    KmerCode y = x;
                    y.append(c, kmask, shift);
                    int n = 0;
                    while (solid(y) && ++n < m) {
                        const int nb = kmer_code(s[e + n]);
                        if (nb < 0) break;
                        y.append(nb, kmask, shift);
                    }
                    if (n > best_n) {
                        best_n = n;
                        best_c = c;
                        tie = false;
                    } else if (n == best_n && n > 0) {
                        tie = true;
                    }
                }
                if (best_n == 0 || tie) break;
                x.append(best_c, kmask, shift);
                for (int i = 1; i < best_n; ++i) x.append(kmer_code(s[e + i]), kmask, shift);
                j += best_n;
                known_bad = best_n < k;
            }

            // left walk: x is window j + 1 of w
            x = code_at(a0);
            known_bad = false;
            for (int j = a0 - 1; j >= 0;) {
                const int e = j;
                const int b = kmer_code(s[e]);
                if (!known_bad && b >= 0 && was_solid(j)) {
                    x.prepend(b, kmask, shift);
                    --j;
                    continue;
                }
                if (b < 0) break;
                flag(e);
                const int m = min(k, j + 1);
                int best_c = -1, best_n = 0;
                bool tie = false;
                for (int c = 0; c < 4; ++c) {
                    if (c == b) continue;
                    KmerCode y = x;
                    y.prepend(c, kmask, shift);
                    int n = 0;
                    while (solid(y) && ++n < m) {
                        const int nb = kmer_code(s[e - n]);
                        if (nb < 0) break;
                        y.prepend(nb, kmask, shift);
                    }
                    if (n > best_n) {
                        best_n = n;
                        best_c = c;
                        tie = false;
                    } else if (n == best_n && n > 0) {
                        tie = true;
                    }
                }
                if (best_n == 0 || tie) break;
                x.prepend(best_c, kmask, shift);
                for (int i = 1; i < best_n; ++i) x.prepend(kmer_code(s[e - i]), kmask, shift);
                j -= best_n;
                known_bad = best_n < k;
            }
        }
        if (full) atomicOr(status, KBBQ_FLAG_KMER_FULL);
    }
    __syncwarp();
    const long long nreads = N - r0 < 32 ? N - r0 : 32;
    const int nwords = (int)((nreads * L + 31) / 32);
    uint32_t *out = bits + (r0 / 32) * L;
    for (int w = lane; w < nwords; w += 32) out[w] = wb[w];
}

__global__ void kmer_correct_kernel(const uint8_t *seq, long long N, int L, int k, const ulonglong2 *table,
                                    unsigned long long mask, unsigned long long t, uint32_t *bits, int *status) {
    kmer_correct_reads(seq, N, L, k, KmerTable{table, mask}, t, bits, status);
}

// the correcting walk on a table split across partitions
__global__ void kmer_correct_parts_kernel(const uint8_t *seq, long long N, int L, int k, const KmerParts tables,
                                          unsigned long long t, uint32_t *bits, int *status) {
    kmer_correct_reads<const KmerParts &>(seq, N, L, k, tables, t, bits, status);
}

}  // namespace kbbq
