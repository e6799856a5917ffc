// Noise of the sampling decoding (DESIGN.md section 15), shared by the fused classifier epilogue (gemm_tcgen05.cu) and the
// fallback kernel over fp32 logits (sampling.cu), so that both draw from the same bits.
//   Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011; the Random123 constants),
//   counter (t, s, v >> 2, 0) and key (lo32(key_b), hi32(key_b)): column t of sample s of source b, token v takes output
//   word v & 3, so one call serves four consecutive tokens.
//   u = ((x >> 9) * 2 + 1) * 2^-24: an odd multiple of 2^-24, strictly inside (0, 1) and exact in fp32.
//   g = -log(-log(u)): standard Gumbel, so argmax_v (logit_v / T + g_v) is distributed as softmax(logits / T).
#pragma once
#include <cstdint>

namespace ttb {

struct Philox4 { uint32_t x[4]; };

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += W0;
        k1 += W1;
    }
    return Philox4{{c0, c1, c2, c3}};
}

__device__ __forceinline__ float philox_uniform(uint32_t x) { return (float)((x >> 9) * 2u + 1u) * 5.9604644775390625e-8f; }   // 2^-24
__device__ __forceinline__ float gumbel(uint32_t x) { return -logf(-logf(philox_uniform(x))); }

// The four noise values of tokens 4 j .. 4 j + 3 at column t of sample s, source key `key`.
__device__ __forceinline__ Philox4 sample_noise_bits(int t, int s, int j, unsigned long long key) {
    return philox4x32_10((uint32_t)t, (uint32_t)s, (uint32_t)j, 0u, (uint32_t)key, (uint32_t)(key >> 32));
}

// Word i of a Philox output, without a local-memory array for a run-time index.
__device__ __forceinline__ uint32_t philox_word(const Philox4& p, int i) {
    return i == 0 ? p.x[0] : (i == 1 ? p.x[1] : (i == 2 ? p.x[2] : p.x[3]));
}

// Draw order: larger z wins, equal z go to the lower token id.
__device__ __forceinline__ bool sample_better(float z, int v, float bz, int bv) { return z > bz || (z == bz && v < bv); }

// Candidate-list insertion of classifier_stats_kernel: (v, col) enters a list sorted descending when it beats the last entry;
// equal values stay behind earlier (lower) columns.
template <int KT>
__device__ __forceinline__ void topk_list_insert(float (&tv)[KT], int (&ti)[KT], float v, int col) {
    if (v > tv[KT - 1]) {
        float cv = v;
        int ci = col;
#pragma unroll
        for (int i = 0; i < KT; ++i) {
            if (cv > tv[i]) {
                const float t0 = tv[i]; tv[i] = cv; cv = t0;
                const int t1 = ti[i]; ti[i] = ci; ci = t1;
            }
        }
    }
}

}  // namespace ttb
