// expand.cuh -- the packed forms of (seq, corrected) that cross PCIe (host_pack.cpp) back into byte arrays in HBM.
#pragma once
#include "common.cuh"

namespace kbbq {

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

}  // namespace kbbq
