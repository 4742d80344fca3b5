/*
 * kmer_correct_oracle.c -- CPU restatement of the correcting walk (DESIGN.md section 10, "The correcting walk"), the
 * reference the GPU tests of kbbq_kmer_correct compare against.
 *
 * TEST INFRASTRUCTURE ONLY: tests/kmer_correct_oracle.py compiles it into a temporary directory and loads it; the
 * product (kbbq-py_b200/) never links it, and it shares no code with the library.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* A=0 C=1 G=2 T=3, anything else (N, lowercase) -1 */
static int kmer_base(uint8_t b) {
    switch (b) {
    case 'A': return 0;
    case 'C': return 1;
    case 'G': return 2;
    case 'T': return 3;
    default: return -1;
    }
}

/* canonical code of the window of k bases at s, or -1 when one of them is not A/C/G/T */
static int64_t kmer_window_key(const uint8_t *s, int k) {
    uint64_t f = 0, r = 0;
    for (int i = 0; i < k; ++i) {
        int c = kmer_base(s[i]);
        if (c < 0) return -1;
        f = (f << 2) | (uint64_t)c;
        r |= (uint64_t)(3 - c) << (2 * i);   /* the reverse complement reads the window backwards */
    }
    return (int64_t)(f < r ? f : r);
}

static int cmp_u64(const void *a, const void *b) {
    uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b;
    return x < y ? -1 : x > y;
}

/* ---- the correcting walk (DESIGN.md section 10, "The correcting walk") -------------------------------------------
 * A literal restatement of the rule on a working copy w of each read: every window's key is recomputed from scratch
 * with kmer_window_key and its count looked up by binary search in the sorted codes of the batch.  Counts, histogram
 * and threshold as oracle_kmer_errors of tests/kmer_oracle.c.  Returns -1 on a bad argument or when out of memory. */
static int64_t kmer_count_of(const uint64_t *keys, int64_t nk, int64_t key) {
    if (key < 0) return 0;
    int64_t lo = 0, hi = nk;
    while (lo < hi) { int64_t m = (lo + hi) / 2; if (keys[m] < (uint64_t)key) lo = m + 1; else hi = m; }
    int64_t a = lo;
    hi = nk;
    while (lo < hi) { int64_t m = (lo + hi) / 2; if (keys[m] <= (uint64_t)key) lo = m + 1; else hi = m; }
    return lo - a;
}

/* window j of w is solid */
static int kmer_w_solid(const uint8_t *w, int64_t j, int k, const uint64_t *keys, int64_t nk, int t) {
    return kmer_count_of(keys, nk, kmer_window_key(w + j, k)) >= t;
}

/* lookups of valid windows: every one of the first pass, and those the walks score -- what kmer_correct_kernel looks
 * up, as it reuses the first-pass bit of every other window.  Counted for tools/kmer_bench.py only. */
static uint64_t kmer_score_lookups;

/* score(c) of the walk: the consecutive solid windows j, j + dir, ... of w with w[e] = c, at most m */
static int kmer_w_score(uint8_t *w, int64_t e, uint8_t c, int64_t j, int dir, int64_t m, int k, const uint64_t *keys,
                        int64_t nk, int t) {
    uint8_t keep = w[e];
    int n = 0;
    w[e] = c;
    while (n < m) {
        if (kmer_window_key(w + j + dir * n, k) >= 0) ++kmer_score_lookups;
        if (!kmer_w_solid(w, j + dir * n, k, keys, nk, t)) break;
        ++n;
    }
    w[e] = keep;
    return n;
}

/* the walk from the anchor in direction dir (+1 right, -1 left), flagging into bits at row offset `row` */
static void kmer_walk(uint8_t *w, int64_t nw, int k, int64_t j, int dir, const uint64_t *keys, int64_t nk, int t,
                      uint32_t *bits, uint64_t row) {
    static const uint8_t ACGT[4] = {'A', 'C', 'G', 'T'};
    for (; j >= 0 && j < nw; j += dir) {
        if (kmer_w_solid(w, j, k, keys, nk, t)) continue;
        int64_t e = dir > 0 ? j + k - 1 : j;
        if (kmer_base(w[e]) < 0) return;
        int64_t m = dir > 0 ? nw - j : j + 1;
        if (m > k) m = k;
        int best = 0, nbest = 0;
        uint8_t best_c = 0;
        for (int i = 0; i < 4; ++i) {
            if (ACGT[i] == w[e]) continue;
            int sc = kmer_w_score(w, e, ACGT[i], j, dir, m, k, keys, nk, t);
            if (sc > best) { best = sc; nbest = 1; best_c = ACGT[i]; }
            else if (sc == best) ++nbest;
        }
        bits[(row + (uint64_t)e) / 32] |= 1u << ((row + (uint64_t)e) % 32);
        if (best < 1 || nbest != 1) return;
        w[e] = best_c;
    }
}

int oracle_kmer_corrections(const uint8_t *seq, int64_t N, int L, int k, int min_count, uint32_t *bits, uint64_t *hist,
                            int *t_out) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || min_count < 0 || !bits || !hist || !t_out) return -1;
    int64_t nw = L >= k ? (int64_t)(L - k + 1) : 0;
    uint64_t *keys = malloc((size_t)(N * nw + 1) * 8);
    uint8_t *w = malloc((size_t)L);
    unsigned char *solid = malloc((size_t)(nw + 1));
    if (!keys || !w || !solid) { free(keys); free(w); free(solid); return -1; }
    int64_t nk = 0;
    for (int64_t r = 0; r < N; ++r)
        for (int64_t j = 0; j < nw; ++j) {
            int64_t key = kmer_window_key(seq + r * L + j, k);
            if (key >= 0) keys[nk++] = (uint64_t)key;
        }
    qsort(keys, (size_t)nk, 8, cmp_u64);
    memset(hist, 0, 256 * 8);
    for (int64_t i = 0; i < nk;) {
        int64_t e = i;
        while (e < nk && keys[e] == keys[i]) ++e;
        int64_t c = e - i;
        hist[c < 255 ? c : 255] += 1;
        i = e;
    }
    int t = min_count;
    if (t <= 0) {
        t = 255;
        for (int c = 2; c <= 254; ++c)
            if (hist[c] <= hist[c + 1]) { t = c; break; }
    }
    *t_out = t;

    memset(bits, 0, (size_t)(((uint64_t)N * L + 31) / 32) * 4);
    for (int64_t r = 0; r < N; ++r) {
        const uint8_t *s = seq + r * L;
        /* 1-2: the solid windows and the anchor, the longest maximal run of them (the leftmost of equal ones) */
        int64_t a0 = -1, best = 0;
        for (int64_t j = 0; j < nw; ++j) solid[j] = (unsigned char)kmer_w_solid(s, j, k, keys, nk, t);
        for (int64_t j = 0; j < nw;) {
            if (!solid[j]) { ++j; continue; }
            int64_t b = j;
            while (b < nw && solid[b]) ++b;
            if (b - j > best) { best = b - j; a0 = j; }
            j = b;
        }
        for (int64_t j = 0; j < nw; ++j) kmer_score_lookups += kmer_window_key(s + j, k) >= 0;   /* the first pass */
        if (best == 0) continue;
        /* 3-4: the two walks on a working copy; they change disjoint bases */
        memcpy(w, s, (size_t)L);
        kmer_walk(w, nw, k, a0 + best, +1, keys, nk, t, bits, (uint64_t)r * L);
        kmer_walk(w, nw, k, a0 - 1, -1, keys, nk, t, bits, (uint64_t)r * L);
    }
    free(keys); free(w); free(solid);
    return 0;
}

/* the table lookups kmer_correct_kernel makes on the batch for t >= 2 (t = 1 makes none): every valid window in its
 * first pass, then the valid windows the walks score */
int oracle_kmer_correct_lookups(const uint8_t *seq, int64_t N, int L, int k, int min_count, uint64_t *lookups) {
    uint32_t *bits = malloc((size_t)(((uint64_t)N * L + 31) / 32 + 1) * 4);
    uint64_t hist[256];
    int t = 0;
    if (!bits || !lookups) { free(bits); return -1; }
    kmer_score_lookups = 0;
    int rc = oracle_kmer_corrections(seq, N, L, k, min_count, bits, hist, &t);
    free(bits);
    *lookups = kmer_score_lookups;
    return rc;
}
