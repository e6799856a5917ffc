// Sampling decoding (ttb_sample_generate, DESIGN.md section 15): the bookkeeping kernels of the KV-cached loop run with
// S sample rows per source, and the draw over fp32 logits where the fused classifier epilogue does not run.
//   Slot r = b * S + s is sample s of source b.  Every slot starts from BOS, appends one drawn token per step and ends at
//   its first drawn EOS or PAD (kept) or when it holds max_len tokens; slots end individually.
#include "kernels.cuh"
#include "philox.cuh"

namespace ttb {

// ---- per-source key: FNV-1a-64 over the 8 little-endian bytes of the seed, then the 4 little-endian bytes of every
// non-PAD source token in column order (the key ignores where the PAD sits, so padded widths do not matter) ----------
__global__ void sample_keys_kernel(const int* __restrict__ src32, int B, int Ls, int pad, unsigned long long seed,
                                   unsigned long long* __restrict__ keys) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    constexpr unsigned long long P = 0x100000001b3ull;
    unsigned long long h = 0xcbf29ce484222325ull;
    for (int i = 0; i < 8; ++i) h = (h ^ ((seed >> (8 * i)) & 0xffull)) * P;
    const int* row = src32 + (long long)b * Ls;
    for (int c = 0; c < Ls; ++c) {
        const unsigned int tok = (unsigned int)row[c];
        if ((int)tok == pad) continue;
        for (int i = 0; i < 4; ++i) h = (h ^ ((tok >> (8 * i)) & 0xffu)) * P;
    }
    keys[b] = h;
}
void launch_sample_keys(const int* src32, int B, int Ls, int pad, unsigned long long seed, unsigned long long* keys, cudaStream_t s) {
    sample_keys_kernel<<<(B + 127) / 128, 128, 0, s>>>(src32, B, Ls, pad, seed, keys);
}

// ---- loop state before the first step: every slot holds BOS, the output is PAD ----------------------------------------
__global__ void __launch_bounds__(1024) sample_init_kernel(GreedyState st, SampleLoop sl) {
    const int R = st.B;
    for (long long i = threadIdx.x; i < (long long)R * st.gen_ld; i += blockDim.x) st.gen[i] = (i % st.gen_ld == 0) ? st.bos : st.pad;
    for (long long i = threadIdx.x; i < (long long)R * st.max_len; i += blockDim.x) st.out[i] = st.pad;
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        const int b = r / sl.S, len = st.src_len[b];
        st.front[r] = 0;
        st.active[r] = r;
        st.desc[r] = make_int4(r, 0, st.bos, len);
        sl.kvsrc[r] = b;
        sl.xdesc[r] = make_int4(b, 0, 0, len);
    }
    if (threadIdx.x < CTRL_COUNT) st.ctrl[threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        st.ctrl[CTRL_N_ACTIVE] = R;
        st.ctrl[CTRL_LS] = st.Ls;
    }
}
void launch_sample_init(const GreedyState& st, const SampleLoop& sl, cudaStream_t s) {
    sample_init_kernel<<<1, 1024, 0, s>>>(st, sl);
}

// ---- one step: append the drawn tokens, retire ended slots, compact the live list ---------------------------------------
// Runs in place of greedy_std_step_kernel.  pred[g] is the token drawn for live position g, whose slot holds f + 1 tokens
// (f = desc[g].y).  An ended slot is written to out[slot] (tokens 0 .. f + 1; the PAD behind them is there since the
// init) and leaves the live list; the others keep their order.
__global__ void __launch_bounds__(1024) sample_step_kernel(GreedyState st, SampleLoop sl) {
    pdl_launch_dependents();
    pdl_wait();
    if (st.ctrl[CTRL_DONE]) return;
    const int n_active = st.ctrl[CTRL_N_ACTIVE];
    const int iter = st.ctrl[CTRL_ITERS];
    int kept = 0, unfinished = 0;
    for (int g0 = 0; g0 < n_active; g0 += blockDim.x) {   // uniform loop: block_scan2 needs every thread
        const int g = g0 + threadIdx.x;
        const bool in = g < n_active;
        int r = 0, f = 0, tok = 0;
        bool keep = false;
        if (in) {
            const int4 d = st.desc[g];
            r = d.x;
            f = d.y;
            tok = st.pred[g];
            st.gen[(long long)r * st.gen_ld + f + 1] = tok;
            st.front[r] = f + 1;
            const bool drew_end = tok == st.eos || tok == st.pad;
            keep = !drew_end && f + 2 < st.max_len;
            if (!keep && !drew_end) ++unfinished;
            // K/V of the step's input token (cache position f) is appended by the next advance kernel for kept slots only
            reinterpret_cast<int4*>(st.sel)[g] = make_int4(r, f, 0, keep ? 0 : -1);
            if (!keep) {
                long long* o = st.out + (long long)r * st.max_len;
                const int* row = st.gen + (long long)r * st.gen_ld;
                for (int c = 0; c <= f + 1; ++c) o[c] = row[c];
            }
        }
        int pos, dummy, total, dummy_t;
        block_scan2(keep ? 1 : 0, 0, pos, dummy, total, dummy_t);   // its barriers order every read above before the writes below
        if (keep) {
            const int p = kept + pos, b = r / sl.S, len = st.src_len[b];
            st.active[p] = r;
            st.desc[p] = make_int4(r, f + 1, tok, len);
            sl.kvsrc[p] = b;
            sl.xdesc[p] = make_int4(b, 0, 0, len);
        }
        kept += total;
    }
    for (int o = 16; o > 0; o >>= 1) unfinished += __shfl_xor_sync(0xffffffffu, unfinished, o);
    if ((threadIdx.x & 31) == 0 && unfinished) atomicAdd(&st.ctrl[CTRL_N_LEFT], unfinished);
    if (threadIdx.x == 0) {
        if (st.hist) st.hist[iter] = n_active;
        st.ctrl[CTRL_N_SEL] = n_active;
        st.ctrl[CTRL_N_ACTIVE] = kept;
        st.ctrl[CTRL_ITERS] = iter + 1;
        st.ctrl[CTRL_TOKENS] += n_active;
        st.ctrl[CTRL_DONE] = kept == 0 ? 1 : 0;
    }
}
void launch_sample_step(const GreedyState& st, const SampleLoop& sl, cudaStream_t s) {
    launch_pdl(sample_step_kernel, dim3(1), dim3(st.B < 1024 ? ((st.B + 31) / 32 * 32) : 1024), 0, s, st, sl);
}

// ---- the draw over fp32 logits: one warp per live row ---------------------------------------------------------------
// Candidate set (top_k in [1, V)): the top_k largest logits, ties at the boundary to the lower token id.  theta = the
// top_k-th largest value is found by a bisection over the order-preserving integer image of the floats; the values equal
// to theta are admitted in token order up to top_k.  Then z = logit / T + g over the candidates, larger z wins, equal z
// go to the lower id -- the rule of the fused epilogue.
__device__ __forceinline__ unsigned int float_order_key(float v) {
    const unsigned int u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__global__ void sample_rows_kernel(const float* __restrict__ logits, int ld, int V, RowCount rows, SampleArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows.live()) return;
    const float* p = logits + (long long)row * ld;
    const int4 d = a.desc[row];
    const int slot = d.x, t = d.y + 1, s = slot % a.S;
    const unsigned long long key = a.keys[slot / a.S];
    unsigned int theta = 0u;
    int id_thr = V;   // values equal to theta are candidates up to this token id
    const bool restrict_k = a.top_k > 0 && a.top_k < V;
    if (restrict_k) {
        for (int bit = 31; bit >= 0; --bit) {
            const unsigned int cand = theta | (1u << bit);
            int cnt = 0;
            for (int c = lane; c < V; c += 32) cnt += float_order_key(p[c]) >= cand ? 1 : 0;
            for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            if (cnt >= a.top_k) theta = cand;
        }
        int gt = 0;
        for (int c = lane; c < V; c += 32) gt += float_order_key(p[c]) > theta ? 1 : 0;
        for (int o = 16; o > 0; o >>= 1) gt += __shfl_xor_sync(0xffffffffu, gt, o);
        int need = a.top_k - gt;   // >= 1: theta is the top_k-th largest value
        for (int c0 = 0; c0 < V; c0 += 32) {
            const int c = c0 + lane;
            const unsigned m = __ballot_sync(0xffffffffu, c < V && float_order_key(p[c]) == theta);
            if (__popc(m) >= need) {
                unsigned mm = m;
                for (int i = 1; i < need; ++i) mm &= mm - 1;
                id_thr = c0 + __ffs(mm) - 1;
                break;
            }
            need -= __popc(m);
        }
    }
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int j = lane; 4 * j < V; j += 32) {
        const Philox4 nz = sample_noise_bits(t, s, j, key);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = 4 * j + u;
            if (c >= V) break;
            const float v = p[c];
            if (restrict_k) {
                const unsigned int k = float_order_key(v);
                if (k < theta || (k == theta && c > id_thr)) continue;
            }
            const float z = v / a.temperature + gumbel(nz.x[u]);
            if (sample_better(z, c, best, bi)) { best = z; bi = c; }
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const float oz = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (sample_better(oz, oi, best, bi)) { best = oz; bi = oi; }
    }
    if (lane == 0) a.pred[row] = bi < V ? bi : 0;   // no candidate only with NaN logits
}
void launch_sample_rows(const float* logits, int ld, int V, RowCount rows, const SampleArgs& a, cudaStream_t s) {
    if (rows.max_rows > 0) launch_pdl(sample_rows_kernel, dim3((rows.max_rows + 7) / 8), dim3(256), 0, s, logits, ld, V, rows, a);
}

}  // namespace ttb
