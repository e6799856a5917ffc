// Fused embedding + positional encoding, residual + LayerNorm, argmax and small conversion kernels.
// All of these are memory-bound row kernels: one warp per row, lanes stride the row so that every
// global access of a warp is a contiguous 128-byte line.
#include "kernels.cuh"

namespace ttb {

__global__ void i64_to_i32_kernel(const long long* __restrict__ in, int* __restrict__ out, long long n) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int)in[i];
}
__global__ void i32_to_i64_kernel(const int* __restrict__ in, long long* __restrict__ out, long long n) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = (long long)in[i];
}
__global__ void mask_to_tokens_kernel(const unsigned char* __restrict__ m, int* __restrict__ out, long long n, int pad_id) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = m[i] ? pad_id : pad_id + 1;
}
__global__ void f32_to_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, long long n) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = __float2bfloat16_rn(in[i]);
}
void launch_f32_to_bf16(const float* in, __nv_bfloat16* out, long long n, cudaStream_t s) {
    if (n > 0) f32_to_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, n);
}
void launch_i64_to_i32(const long long* in, int* out, long long n, cudaStream_t s) {
    if (n > 0) i64_to_i32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, n);
}
void launch_i32_to_i64(const int* in, long long* out, long long n, cudaStream_t s) {
    if (n > 0) i32_to_i64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, n);
}
void launch_mask_to_tokens(const unsigned char* mask, int* out, long long n, int pad_id, cudaStream_t s) {
    if (n > 0) mask_to_tokens_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(mask, out, n, pad_id);
}

// ---- embedding + positional encoding (reference: embeddings.py:7-15 and :53-64) --------------
template <typename ActT>
__global__ void embed_seq_kernel(const int* __restrict__ tok, int T, int L, const float* __restrict__ table,
                                 const float* __restrict__ pe, int E, float* __restrict__ x, ActT* __restrict__ xh) {
    int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= T) return;
    const float* e = table + (long long)tok[row] * E;
    const float* p = pe + (long long)((row % L) + 1) * E;
    for (int c = lane; c < E; c += 32) {
        float v = e[c] + p[c];
        x[(long long)row * E + c] = v;
        if (xh) xh[(long long)row * E + c] = from_f32<ActT>(v);
    }
}
template <typename ActT>
void launch_embed_seq(const int* tok, int T, int L, const float* table, const float* pe, int E,
                      float* x, ActT* xh, cudaStream_t s) {
    if (T <= 0) return;
    embed_seq_kernel<ActT><<<(T + 7) / 8, 256, 0, s>>>(tok, T, L, table, pe, E, x, xh);
}
template void launch_embed_seq<float>(const int*, int, int, const float*, const float*, int, float*, float*, cudaStream_t);
template void launch_embed_seq<__nv_bfloat16>(const int*, int, int, const float*, const float*, int, float*, __nv_bfloat16*, cudaStream_t);

// ---- residual add + LayerNorm (post-norm layers, modules.py:56-80; eps 1e-5) ----------------
// Row statistics follow torch's CPU LayerNorm: mean, then biased variance of (x - mean).
template <typename ActT, int MAXPL>
__global__ void add_layernorm_kernel(const float* __restrict__ resid, const float* __restrict__ y,
                                     const float* __restrict__ g, const float* __restrict__ b,
                                     const float* __restrict__ g2, const float* __restrict__ b2,
                                     float* __restrict__ out, ActT* __restrict__ outh, RowCount rows, int E) {
    int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= rows.live()) return;
    const long long base = (long long)row * E;
    float v[MAXPL];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < MAXPL; ++k) {
        int c = lane + 32 * k;
        float t = 0.f;
        if (c < E) {
            t = resid[base + c];
            if (y) t += y[base + c];
        }
        v[k] = t;
        sum += t;
    }
    const float inv_e = 1.0f / (float)E;
    float mean = warp_sum(sum) * inv_e;
    float sq = 0.f;
#pragma unroll
    for (int k = 0; k < MAXPL; ++k) {
        int c = lane + 32 * k;
        float d = (c < E) ? v[k] - mean : 0.f;
        sq += d * d;
    }
    float rstd = rsqrtf(warp_sum(sq) * inv_e + 1e-5f);
#pragma unroll
    for (int k = 0; k < MAXPL; ++k) {
        int c = lane + 32 * k;
        if (c < E) v[k] = (v[k] - mean) * rstd * g[c] + b[c];
    }
    if (g2) {  // final LayerNorm of the stack fused on top (modules.py:67 / :79)
        sum = 0.f;
#pragma unroll
        for (int k = 0; k < MAXPL; ++k) sum += (lane + 32 * k < E) ? v[k] : 0.f;
        mean = warp_sum(sum) * inv_e;
        sq = 0.f;
#pragma unroll
        for (int k = 0; k < MAXPL; ++k) {
            float d = (lane + 32 * k < E) ? v[k] - mean : 0.f;
            sq += d * d;
        }
        rstd = rsqrtf(warp_sum(sq) * inv_e + 1e-5f);
#pragma unroll
        for (int k = 0; k < MAXPL; ++k) {
            int c = lane + 32 * k;
            if (c < E) v[k] = (v[k] - mean) * rstd * g2[c] + b2[c];
        }
    }
#pragma unroll
    for (int k = 0; k < MAXPL; ++k) {
        int c = lane + 32 * k;
        if (c < E) {
            out[base + c] = v[k];
            if (outh) outh[base + c] = from_f32<ActT>(v[k]);
        }
    }
}
// E == 256 fast path: one warp per row, each lane owns 8 consecutive columns (two 16-byte loads per
// operand, one 16-byte bf16 store), i.e. every warp instruction moves a whole 1 KB / 512 B row.
template <typename ActT>
__global__ void __launch_bounds__(256)
add_layernorm256_kernel(const float* __restrict__ resid, const float* __restrict__ y,
                        const float* __restrict__ g, const float* __restrict__ b,
                        const float* __restrict__ g2, const float* __restrict__ b2,
                        float* __restrict__ out, ActT* __restrict__ outh, RowCount rows) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows.live()) return;
    const long long base = (long long)row * 256 + lane * 8;
    float v[8];
    {
        const float4 r0 = *reinterpret_cast<const float4*>(resid + base), r1 = *reinterpret_cast<const float4*>(resid + base + 4);
        v[0] = r0.x; v[1] = r0.y; v[2] = r0.z; v[3] = r0.w; v[4] = r1.x; v[5] = r1.y; v[6] = r1.z; v[7] = r1.w;
        if (y) {
            const float4 y0 = *reinterpret_cast<const float4*>(y + base), y1 = *reinterpret_cast<const float4*>(y + base + 4);
            v[0] += y0.x; v[1] += y0.y; v[2] += y0.z; v[3] += y0.w; v[4] += y1.x; v[5] += y1.y; v[6] += y1.z; v[7] += y1.w;
        }
    }
    auto normalise = [&](const float* gg, const float* bb) {
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) sum += v[k];
        const float mean = warp_sum(sum) * (1.0f / 256.0f);
        float sq = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const float d = v[k] - mean; sq += d * d; }
        const float rstd = rsqrtf(warp_sum(sq) * (1.0f / 256.0f) + 1e-5f);
        const float4 g0 = *reinterpret_cast<const float4*>(gg + lane * 8), g1 = *reinterpret_cast<const float4*>(gg + lane * 8 + 4);
        const float4 b0 = *reinterpret_cast<const float4*>(bb + lane * 8), b1 = *reinterpret_cast<const float4*>(bb + lane * 8 + 4);
        const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = (v[k] - mean) * rstd * gv[k] + bv[k];
    };
    normalise(g, b);
    if (g2) normalise(g2, b2);
    *reinterpret_cast<float4*>(out + base) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(out + base + 4) = make_float4(v[4], v[5], v[6], v[7]);
    if (outh) {
        if constexpr (sizeof(ActT) == 2) {
            __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
            __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
            uint4 u;
            u.x = *reinterpret_cast<uint32_t*>(&p0); u.y = *reinterpret_cast<uint32_t*>(&p1);
            u.z = *reinterpret_cast<uint32_t*>(&p2); u.w = *reinterpret_cast<uint32_t*>(&p3);
            *reinterpret_cast<uint4*>(outh + base) = u;
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) outh[base + k] = from_f32<ActT>(v[k]);
        }
    }
}

template <typename ActT>
void launch_add_layernorm(const float* resid, const float* y, const float* g, const float* b,
                          const float* g2, const float* b2, float* out, ActT* outh,
                          RowCount rows, int E, cudaStream_t s) {
    if (rows.max_rows <= 0) return;
    int grid = (rows.max_rows + 7) / 8;
    if (E == 256)
        add_layernorm256_kernel<ActT><<<grid, 256, 0, s>>>(resid, y, g, b, g2, b2, out, outh, rows);
    else if (E <= 256)
        add_layernorm_kernel<ActT, 8><<<grid, 256, 0, s>>>(resid, y, g, b, g2, b2, out, outh, rows, E);
    else
        add_layernorm_kernel<ActT, 32><<<grid, 256, 0, s>>>(resid, y, g, b, g2, b2, out, outh, rows, E);
}
template void launch_add_layernorm<float>(const float*, const float*, const float*, const float*, const float*, const float*, float*, float*, RowCount, int, cudaStream_t);
template void launch_add_layernorm<__nv_bfloat16>(const float*, const float*, const float*, const float*, const float*, const float*, float*, __nv_bfloat16*, RowCount, int, cudaStream_t);

__global__ void row_lengths_kernel(const int* __restrict__ tok, int L, int pad_id, int* __restrict__ out) {
    __shared__ int s_len;
    if (threadIdx.x == 0) s_len = 0;
    __syncthreads();
    int last = 0;
    for (int j = threadIdx.x; j < L; j += blockDim.x)
        if (tok[(long long)blockIdx.x * L + j] != pad_id) last = j + 1;
    if (last) atomicMax(&s_len, last);
    __syncthreads();
    if (threadIdx.x == 0) out[blockIdx.x] = s_len;
}
void launch_row_lengths(const int* tok, int B, int L, int pad_id, int* out, cudaStream_t s) {
    if (B > 0) row_lengths_kernel<<<B, 128, 0, s>>>(tok, L, pad_id, out);
}

// ---- argmax over the vocabulary (first maximal index, like torch.argmax) ----------------------
__global__ void argmax_rows_kernel(const float* __restrict__ logits, int ld, int V, int* __restrict__ out, RowCount rows) {
    int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    pdl_launch_dependents();
    pdl_wait();
    if (row >= rows.live()) return;
    const float* p = logits + (long long)row * ld;
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int c = lane; c < V; c += 32) {
        float v = p[c];
        if (v > best || (v == best && c < bi) || bi == 0x7fffffff) { best = v; bi = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, best, o);
        int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi != 0x7fffffff && (bi == 0x7fffffff || ov > best || (ov == best && oi < bi))) { best = ov; bi = oi; }
    }
    if (lane == 0) out[row] = bi;
}
void launch_argmax_rows(const float* logits, int ld, int V, int* out, RowCount rows, cudaStream_t s) {
    if (rows.max_rows <= 0) return;
    launch_pdl(argmax_rows_kernel, dim3((rows.max_rows + 7) / 8), dim3(256), 0, s, logits, ld, V, out, rows);
}

}  // namespace ttb
