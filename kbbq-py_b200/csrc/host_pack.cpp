// host_pack.cpp -- host-side packing for the PCIe-bound host-buffer entry point.
//
// kbbq_recalibrate_host spends its time on PCIe (4.5 GB up, 1.5 GB down per 10 M x 150 bp, the
// kernels take 2 ms).  The corrected reads are only ever compared with the reads
// (find_corrected_sites, kbbq/recalibrate.py:13-20), so one bit per base carries everything the build
// needs from them: the host cores reduce (seq, corrected) to a mismatch bit map while the copy engine
// moves seq and qual, the map (1/8 of the bytes) follows, and expand_corr_kernel (expand.cuh) turns
// it back into a byte array that differs from seq exactly where the corrected read did.
// kbbq_host_pack_nibbles goes one step further and folds the read itself into the same pass: 4 bits per
// base (3-bit base code | mismatch), so that seq + corrected cross PCIe as 0.5 B per base instead of 1.125 and
// only the qualities travel as they are; expand_nibbles_kernel (expand.cuh) rebuilds both byte arrays in HBM.
// Plain host C++ (no CUDA).  AVX2 when the CPU has it (32 bases per compare + movemask), portable
// 64-bit SWAR otherwise.
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <thread>
#include <vector>

#include "../../include/kbbq_b200.h"

#if defined(__x86_64__)
#include <immintrin.h>
#endif

namespace {

#if defined(__x86_64__)
__attribute__((target("avx2"))) void bits_avx2(const uint8_t *a, const uint8_t *b, size_t words, uint32_t *out) {
    for (size_t i = 0; i < words; ++i) {
        const __m256i x = _mm256_loadu_si256((const __m256i *)(a + 32 * i));
        const __m256i y = _mm256_loadu_si256((const __m256i *)(b + 32 * i));
        out[i] = ~(uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(x, y));
    }
}
#endif

// bit j of out[i] = (a[32 i + j] != b[32 i + j])
void bits_portable(const uint8_t *a, const uint8_t *b, size_t words, uint32_t *out) {
    for (size_t i = 0; i < words; ++i) {
        uint32_t w = 0;
        for (int k = 0; k < 4; ++k) {
            uint64_t x, y;
            memcpy(&x, a + 32 * i + 8 * k, 8);
            memcpy(&y, b + 32 * i + 8 * k, 8);
            uint64_t d = x ^ y;
            // bit 7 of every non-zero byte, then gather the eight flags into one byte
            d = (((d & 0x7F7F7F7F7F7F7F7Full) + 0x7F7F7F7F7F7F7F7Full) | d) & 0x8080808080808080ull;
            w |= (uint32_t)(((d >> 7) * 0x0102040810204080ull) >> 56) << (8 * k);
        }
        out[i] = w;
    }
}

// ---- 4 bits per base: 3-bit base code | mismatch << 3 ----
// code = (base >> 1) & 7 tells A (0), C (1), T (2), G (3) and N (7) apart; any other byte fails the round trip
// through the 8-entry table below, which is the reference's TypeError for a base outside ACGTN
// (kbbq/compare_reads.py:289-302) found on the host, since the device never sees the byte itself.
const uint8_t kCodeToBase[16] = {'A', 'C', 'T', 'G', 0, 0, 0, 'N', 'A', 'C', 'T', 'G', 0, 0, 0, 'N'};

#if defined(__x86_64__)
__attribute__((target("avx2"))) uint32_t nibbles_avx2(const uint8_t *a, const uint8_t *b, size_t blocks, uint8_t *out, bool stream_stores) {
    const __m256i lut = _mm256_broadcastsi128_si256(_mm_loadu_si128((const __m128i *)kCodeToBase));
    const __m256i seven = _mm256_set1_epi8(7), eight = _mm256_set1_epi8(8), w = _mm256_set1_epi16(0x1001);
    __m256i bad = _mm256_setzero_si256();
    const bool nt = (((uintptr_t)out) & 31u) == 0 && stream_stores;
    for (size_t i = 0; i < blocks; ++i) {   // 64 bases -> 32 bytes
        const __m256i x0 = _mm256_loadu_si256((const __m256i *)(a + 64 * i)), x1 = _mm256_loadu_si256((const __m256i *)(a + 64 * i + 32));
        const __m256i y0 = _mm256_loadu_si256((const __m256i *)(b + 64 * i)), y1 = _mm256_loadu_si256((const __m256i *)(b + 64 * i + 32));
        const __m256i c0 = _mm256_and_si256(_mm256_srli_epi16(x0, 1), seven), c1 = _mm256_and_si256(_mm256_srli_epi16(x1, 1), seven);
        bad = _mm256_or_si256(bad, _mm256_or_si256(_mm256_xor_si256(_mm256_shuffle_epi8(lut, c0), x0),
                                                   _mm256_xor_si256(_mm256_shuffle_epi8(lut, c1), x1)));
        const __m256i n0 = _mm256_or_si256(c0, _mm256_andnot_si256(_mm256_cmpeq_epi8(x0, y0), eight));
        const __m256i n1 = _mm256_or_si256(c1, _mm256_andnot_si256(_mm256_cmpeq_epi8(x1, y1), eight));
        // even nibble + 16 * odd nibble in every 16-bit lane, then the low bytes of the sixteen-bit lanes
        const __m256i p = _mm256_permute4x64_epi64(_mm256_packus_epi16(_mm256_maddubs_epi16(n0, w), _mm256_maddubs_epi16(n1, w)), 0xD8);
        if (nt) _mm256_stream_si256((__m256i *)(out + 32 * i), p);
        else _mm256_storeu_si256((__m256i *)(out + 32 * i), p);
    }
    if (nt) _mm_sfence();
    return _mm256_testz_si256(bad, bad) ? 0u : 1u;
}
#endif

uint32_t nibbles_portable(const uint8_t *a, const uint8_t *b, size_t first, size_t last, uint8_t *out) {
    uint32_t bad = 0;
    for (size_t j = first; j < last; ++j) {   // bases; `first` is even
        const uint8_t c = (a[j] >> 1) & 7;
        bad |= (uint32_t)(kCodeToBase[c] ^ a[j]);
        const uint8_t nib = (uint8_t)(c | ((a[j] != b[j]) << 3));
        if (j & 1) out[j >> 1] |= (uint8_t)(nib << 4);
        else out[j >> 1] = nib;
    }
    return bad ? 1u : 0u;
}

}  // namespace

extern "C" int kbbq_host_pack_nibbles(const uint8_t *seq, const uint8_t *corr, int64_t n, uint8_t *packed, int threads,
                                      int *bad_base) {
    if (n < 0 || (n > 0 && (!seq || !corr || !packed))) return KBBQ_E_ARG;
    const size_t blocks = (size_t)n / 64;
    int T = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (T < 1) T = 1;
    if ((size_t)T > blocks / 2048 + 1) T = (int)(blocks / 2048 + 1);
#if defined(__x86_64__)
    const bool avx2 = __builtin_cpu_supports("avx2");
#else
    const bool avx2 = false;
#endif
    std::vector<uint32_t> bad((size_t)T * 16, 0);   // one cache line per thread
    // the packed form is read next by the copy engine, not by a core: streaming stores (KBBQ_PACK_NT=0: plain ones)
    const char *nt_env = getenv("KBBQ_PACK_NT");
    const bool stream_stores = !nt_env || atoi(nt_env) != 0;
    auto run = [&](int t) {
        const size_t lo = blocks * t / T, hi = blocks * (t + 1) / T;
#if defined(__x86_64__)
        if (avx2) { bad[(size_t)t * 16] = nibbles_avx2(seq + 64 * lo, corr + 64 * lo, hi - lo, packed + 32 * lo, stream_stores); return; }
#endif
        bad[(size_t)t * 16] = nibbles_portable(seq, corr, 64 * lo, 64 * hi, packed);
    };
    if (T == 1) run(0);
    else {
        std::vector<std::thread> pool;
        pool.reserve(T);
        for (int t = 0; t < T; ++t) pool.emplace_back(run, t);
        for (auto &th : pool) th.join();
    }
    uint32_t any = nibbles_portable(seq, corr, blocks * 64, (size_t)n, packed);
    for (int t = 0; t < T; ++t) any |= bad[(size_t)t * 16];
    if (bad_base) *bad_base = any ? 1 : 0;
    return KBBQ_OK;
}

extern "C" int kbbq_host_mismatch_bits(const uint8_t *seq, const uint8_t *corr, int64_t n, uint32_t *bits, int threads) {
    if (n < 0 || (n > 0 && (!seq || !corr || !bits))) return KBBQ_E_ARG;
    const size_t words = (size_t)n / 32;
    int T = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (T < 1) T = 1;
    if ((size_t)T > words / 4096 + 1) T = (int)(words / 4096 + 1);
#if defined(__x86_64__)
    const bool avx2 = __builtin_cpu_supports("avx2");
#else
    const bool avx2 = false;
#endif
    auto run = [&](int t) {
        const size_t lo = words * t / T, hi = words * (t + 1) / T;
#if defined(__x86_64__)
        if (avx2) { bits_avx2(seq + 32 * lo, corr + 32 * lo, hi - lo, bits + lo); return; }
#endif
        bits_portable(seq + 32 * lo, corr + 32 * lo, hi - lo, bits + lo);
    };
    if (T == 1) run(0);
    else {
        std::vector<std::thread> pool;
        pool.reserve(T);
        for (int t = 0; t < T; ++t) pool.emplace_back(run, t);
        for (auto &th : pool) th.join();
    }
    if ((size_t)n % 32) {  // last partial word
        uint32_t w = 0;
        for (size_t j = words * 32; j < (size_t)n; ++j) w |= (uint32_t)(seq[j] != corr[j]) << (j - words * 32);
        bits[words] = w;
    }
    return KBBQ_OK;
}
