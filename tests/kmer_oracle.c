/*
 * kmer_oracle.c -- CPU restatement of the k-mer error rule (DESIGN.md section 10), the reference the GPU tests of
 * kbbq_kmer_* compare against.
 *
 * TEST INFRASTRUCTURE ONLY: tests/kmer_oracle.py compiles it into a temporary directory and loads it; the product
 * (kbbq-py_b200/) never links it, and it shares no code with the library.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* ---- errors from k-mer counts (DESIGN.md, "Errors from k-mer counts") --------------------------------------------
 * A plain restatement of the rule: exact counts by sorting the canonical codes of all valid windows, counts looked up
 * by binary search, coverage of every base by scanning the k windows over it.  bits: ceil(N*L/32) words, bit i of the
 * flattened batch in word i/32, LSB first.  hist u64[256].  *t: the threshold used.  Returns -1 on a bad argument or
 * when out of memory. */
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

int oracle_kmer_errors(const uint8_t *seq, int64_t N, int L, int k, int min_count, uint32_t *bits, uint64_t *hist,
                       int *t_out) {
    if (N < 0 || L < 1 || k < 1 || k > 31 || min_count < 0 || !bits || !hist || !t_out) return -1;
    int64_t nw = L >= k ? (int64_t)(L - k + 1) : 0;
    uint64_t *keys = malloc((size_t)(N * nw + 1) * 8);
    int64_t *wkey = malloc((size_t)(N * nw + 1) * 8);
    unsigned char *solid = malloc((size_t)(nw + 1));
    if (!keys || !wkey || !solid) { free(keys); free(wkey); free(solid); return -1; }
    int64_t nk = 0;
    for (int64_t r = 0; r < N; ++r)
        for (int64_t j = 0; j < nw; ++j) {
            int64_t key = kmer_window_key(seq + r * L + j, k);
            wkey[r * nw + j] = key;
            if (key >= 0) keys[nk++] = (uint64_t)key;
        }
    qsort(keys, (size_t)nk, 8, cmp_u64);

    /* histogram of the counts of the distinct codes */
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
        int any_solid = 0;
        for (int64_t j = 0; j < nw; ++j) {
            int64_t key = wkey[r * nw + j];
            int64_t count = 0;
            if (key >= 0) {
                /* count = upper bound - lower bound of key in the sorted codes */
                int64_t lo = 0, hi = nk;
                while (lo < hi) { int64_t m = (lo + hi) / 2; if (keys[m] < (uint64_t)key) lo = m + 1; else hi = m; }
                int64_t a = lo;
                hi = nk;
                while (lo < hi) { int64_t m = (lo + hi) / 2; if (keys[m] <= (uint64_t)key) lo = m + 1; else hi = m; }
                count = lo - a;
            }
            solid[j] = count >= t;
            any_solid |= solid[j];
        }
        if (!any_solid) continue;   /* a read from a region the batch does not cover is left alone */
        int a = -1;                 /* start of the current run of uncovered bases */
        for (int i = 0; i <= L; ++i) {
            int uncovered = 0;
            if (i < L) {
                uncovered = 1;
                for (int64_t j = i - k + 1; j <= i; ++j)
                    if (j >= 0 && j < nw && solid[j]) { uncovered = 0; break; }
            }
            if (uncovered && a < 0) a = i;
            if (!uncovered && a >= 0) {
                int b = i - 1, f[2] = {-1, -1};
                if (a > 0 && b < L - 1) { f[0] = a; f[1] = b; }   /* inner run: both ends */
                else if (a == 0) f[0] = b;                       /* at the read start: its end */
                else f[0] = a;                                   /* at the read end: its start */
                for (int m = 0; m < 2; ++m) {
                    if (f[m] < 0 || kmer_base(s[f[m]]) < 0) continue;   /* an N is never an error */
                    uint64_t bit = (uint64_t)r * L + (uint64_t)f[m];
                    bits[bit / 32] |= 1u << (bit % 32);
                }
                a = -1;
            }
        }
    }
    free(keys); free(wkey); free(solid);
    return 0;
}
