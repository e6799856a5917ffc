// Teacher-forced scoring of given targets (ttb_score_targets, DESIGN.md section 14): the bookkeeping kernels around one
// decoder pass over every (candidate, position) row.  Row r = g * Lt + t of a call holds candidate g's prefix up to column t
// and predicts column t + 1.
#include "kernels.cuh"

namespace ttb {

__global__ void score_prepare_kernel(const int* __restrict__ tgt, int G, int Lt, int K, int* __restrict__ kvmap, int* __restrict__ row_tok) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < G) kvmap[i] = (int)(i / K);
    if (i < (long long)G * Lt) row_tok[i] = (i % Lt) + 1 < Lt ? tgt[i + 1] : -1;
}
void launch_score_prepare(const int* tgt, int G, int Lt, int K, int* kvmap, int* row_tok, cudaStream_t s) {
    const long long n = (long long)G * Lt;
    if (n > 0) score_prepare_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(tgt, G, Lt, K, kvmap, row_tok);
}

// One warp per row of fp32 logits: the (tokv, lmax, lsum) triple classifier_stats_kernel writes on the bf16 path.
__global__ void logprob_stats_kernel(const float* __restrict__ logits, int ld, int V, const int* __restrict__ row_tok, int rows,
                                     float* __restrict__ tokv, float* __restrict__ lmax, float* __restrict__ lsum) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float* p = logits + (long long)row * ld;
    float mx = -INFINITY;
    for (int c = lane; c < V; c += 32) mx = fmaxf(mx, p[c]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int c = lane; c < V; c += 32) sum += expf(p[c] - mx);
    sum = warp_sum(sum);
    if (lane == 0) {
        const int tok = row_tok[row];
        tokv[row] = tok >= 0 ? p[tok] : 0.f;
        lmax[row] = mx;
        lsum[row] = sum;
    }
}
void launch_logprob_stats(const float* logits, int ld, int V, const int* row_tok, int rows, float* tokv, float* lmax, float* lsum,
                          cudaStream_t s) {
    if (rows > 0) logprob_stats_kernel<<<(rows + 7) / 8, 256, 0, s>>>(logits, ld, V, row_tok, rows, tokv, lmax, lsum);
}

// One warp per candidate.  Scored columns are 1 .. n: up to and including the first EOS, or up to but not including the
// first PAD, whichever comes first.  Every lane sums its columns in order and the lanes meet in a fixed butterfly, so the
// result does not depend on scheduling (no atomics).
__global__ void score_reduce_kernel(const int* __restrict__ tgt, int G, int Lt, int pad, int eos, const float* __restrict__ tokv,
                                    const float* __restrict__ lmax, const float* __restrict__ lsum, float* __restrict__ logp_out,
                                    int* __restrict__ ntok_out, float* __restrict__ token_logp_out) {
    const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (g >= G) return;
    const int* row = tgt + (long long)g * Lt;
    int n = Lt - 1;
    for (int t0 = 1; t0 < Lt; t0 += 32) {
        const int t = t0 + lane;
        const int tok = t < Lt ? row[t] : pad;
        const unsigned stop = __ballot_sync(0xffffffffu, t < Lt && (tok == pad || tok == eos));
        if (stop) {
            const int first = __ffs(stop) - 1;
            const int tf = t0 + first;
            n = __shfl_sync(0xffffffffu, tok, first) == eos ? tf : tf - 1;
            break;
        }
    }
    const long long r0 = (long long)g * Lt;
    float sum = 0.f;
    for (int t = 1 + lane; t < Lt; t += 32) {
        float v = 0.f;
        if (t <= n) {
            const long long r = r0 + t - 1;
            v = tokv[r] - lmax[r] - logf(lsum[r]);
            sum += v;
        }
        if (token_logp_out) token_logp_out[(long long)g * (Lt - 1) + t - 1] = v;
    }
    sum = warp_sum(sum);
    if (lane == 0) {
        logp_out[g] = sum;
        ntok_out[g] = n;
    }
}
void launch_score_reduce(const int* tgt, int G, int Lt, int pad, int eos, const float* tokv, const float* lmax, const float* lsum,
                         float* logp_out, int* ntok_out, float* token_logp_out, cudaStream_t s) {
    if (G > 0) score_reduce_kernel<<<(G + 7) / 8, 256, 0, s>>>(tgt, G, Lt, pad, eos, tokv, lmax, lsum, logp_out, ntok_out, token_logp_out);
}

}  // namespace ttb
