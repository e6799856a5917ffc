// Device side of the standard beam search.
// Reference: /root/reference/src/decoding/standard_decoding.py:90-174 (TranslationInferenceBeamSearch.generate).
//
// Per step the engine runs
//   sbeam_prepare -> finished flag of every hypothesis (contains EOS), compact list of live hypotheses,
//                    row -> query map for the cross-attention
//   sbeam_embed_last -> embedding of the last token of every live hypothesis
//   decoder stack on those rows (the prefix comes from the hypothesis' KV cache), classifier GEMM
//   sbeam_scores  -> log(softmax(logits)) per hypothesis (artificial logits for finished ones: 35 on the PAD
//                    column, 0 elsewhere, :132-135) added to the hypothesis score
//   sbeam_select  -> per query: the beam_size best of the (beam x vocab) continuations, sorted, and the new
//                    token rows (parent prefix + chosen token); counts hypotheses that contain EOS
#include "kernels.cuh"
#include "topk_emul.cuh"

namespace ttb {

// Control words: [0] live rows of the step, [1] hypotheses that contain EOS after the step's selection, [2] DONE: every
// hypothesis contains EOS (raised by the CTA of sbeam_select that finishes last; the reference's stop test, :169) -- a step the
// host has enqueued ahead of reading [1] is then a no-op --, [3] steps that really ran, [4] ticket of the select CTAs
__global__ void __launch_bounds__(1024) sbeam_prepare_kernel(StdBeamState st, int C, int beam, int W) {
    if (st.ctrl[2]) {
        if (threadIdx.x == 0) st.ctrl[0] = 0;   // no live rows: the decoder kernels of this step exit at once
        return;
    }
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int* row = st.y_cur + (long long)c * st.ldw;
        int fin = 0;
        for (int j = 0; j < W; ++j) fin |= (row[j] == st.eos) ? 1 : 0;
        st.fin[c] = fin;
    }
    __syncthreads();
    if (threadIdx.x == 0) {   // order-preserving compaction (boolean indexing in the reference)
        int run = 0;
        for (int c = 0; c < C; ++c) {
            if (st.fin[c]) { st.cand_row[c] = -1; continue; }
            st.cand_row[c] = run;
            st.row_cand[run] = c;
            st.row_query[run] = c / beam;
            // W - 1 cached positions, the token at W - 1 is this step's input
            st.desc_self[run] = make_int4(c, W - 1, st.y_cur[(long long)c * st.ldw + W - 1], 0x7fffffff);
            st.desc_cross[run] = make_int4(c / beam, 0, 0, st.src_len[c / beam]);
            ++run;
        }
        st.ctrl[0] = run;
        st.ctrl[1] = 0;       // hypotheses with EOS after the coming selection (sbeam_select counts them)
    }
    for (int c = threadIdx.x; c < C; c += blockDim.x) st.c_front[c] = W - 1;
}
void launch_sbeam_prepare(const StdBeamState& st, int C, int beam, int W, cudaStream_t s) {
    sbeam_prepare_kernel<<<1, 1024, 0, s>>>(st, C, beam, W);
}

// One warp per hypothesis: total[c][v] = score[c] + log(softmax(logits_c)[v])   (softmax first, then log, like
// `torch.log(torch.softmax(x, -1))` at :111 / :150)
__global__ void __launch_bounds__(256) sbeam_scores_kernel(StdBeamState st, int C, const float* __restrict__ logits) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= C || st.ctrl[2]) return;
    const int V = st.V, r = st.cand_row[c];
    const float* p = r >= 0 ? logits + (long long)r * V : nullptr;
    auto val = [&](int v) { return p ? p[v] : (v == st.pad ? 35.0f : 0.0f); };
    float mx = -INFINITY;
    for (int v = lane; v < V; v += 32) mx = fmaxf(mx, val(v));
    mx = warp_max(mx);
    float sum = 0.f;
    for (int v = lane; v < V; v += 32) sum += expf(val(v) - mx);
    sum = warp_sum(sum);
    const float base = st.score_cur[c];
    float* out = st.total + (long long)c * V;
    for (int v = lane; v < V; v += 32) out[v] = base + logf(expf(val(v) - mx) / sum);
}
void launch_sbeam_scores(const StdBeamState& st, int C, const float* logits, cudaStream_t s) {
    sbeam_scores_kernel<<<(C + 7) / 8, 256, 0, s>>>(st, C, logits);
}

// One CTA per query: the beam_size best of the beam * V continuation scores in the order torch.topk(sorted=True)
// returns them on the CPU backend (ties between exactly equal scores — the "-35" continuations of finished
// hypotheses — are decided by libstdc++'s partial_sort / nth_element, emulated in topk_emul.cuh), then the new
// token rows.
__global__ void __launch_bounds__(256) sbeam_select_kernel(StdBeamState st, int beam, int W) {
    extern __shared__ __align__(8) unsigned char s_sel_raw[];
    if (st.ctrl[2]) return;                          // step enqueued behind the end of the search
    VF* s_e = reinterpret_cast<VF*>(s_sel_raw);      // [beam * V] (score, flat index)
    const int b = blockIdx.x, V = st.V, K = st.K, n = beam * V;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* tot = st.total + (long long)b * beam * V;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { s_e[i].v = tot[i]; s_e[i].i = i; }
    __syncthreads();
    if (threadIdx.x == 0) topk_sorted_torch_cpu_(s_e, n, K);
    __syncthreads();
    int n_fin = 0;
    for (int j = warp; j < K; j += 8) {
        const int idx = s_e[j].i;
        const int parent = idx / V, ch = idx % V;
        const int* src = st.y_cur + (long long)(b * beam + parent) * st.ldw;
        int* dst = st.y_next + (long long)(b * K + j) * st.ldw;
        int fin = (ch == st.eos) ? 1 : 0;
        for (int c = lane; c < W; c += 32) {
            const int t = src[c];
            dst[c] = t;
            fin |= (t == st.eos) ? 1 : 0;
        }
        if (lane == 0) { dst[W] = ch; st.score_next[b * K + j] = s_e[j].v; if (st.parent) st.parent[b * K + j] = b * beam + parent; }
        fin = __any_sync(0xffffffffu, fin);
        if (lane == 0 && fin) ++n_fin;
    }
    if (lane == 0 && n_fin) atomicAdd(&st.ctrl[1], n_fin);
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&st.ctrl[4], 1) == (int)gridDim.x - 1) {   // last CTA of the step: stop test, step count
            __threadfence();
            st.ctrl[4] = 0;
            st.ctrl[3] += 1;
            if (W > 1 && atomicAdd(&st.ctrl[1], 0) == st.B * st.K) st.ctrl[2] = 1;   // the first step (W = 1) never stops (:106-125)
        }
    }
}
int launch_sbeam_select(const StdBeamState& st, int beam, int W, cudaStream_t s) {
    const size_t smem = (size_t)beam * st.V * sizeof(VF);
    if (smem > 200 * 1024) return -1;
    if (smem > 48 * 1024 && ensure_dyn_smem(sbeam_select_kernel, 200 * 1024)) return 1;
    sbeam_select_kernel<<<st.B, 256, smem, s>>>(st, beam, W);
    return 0;
}

// ---- KV caches --------------------------------------------------------------------------------------------------------
template <typename ActT>
__global__ void sbeam_embed_last_kernel(StdBeamState st, int W, const float* __restrict__ table, const float* __restrict__ pe, int E,
                                        float* __restrict__ x, ActT* __restrict__ xh) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= st.ctrl[0]) return;
    const int tok = st.y_cur[(long long)st.row_cand[r] * st.ldw + W - 1];
    const float* e = table + (long long)tok * E;
    const float* p = pe + (long long)W * E;          // position W - 1 -> row W of the table (row 0 = zeros, embeddings.py:47)
    for (int c = lane; c < E; c += 32) {
        const float v = e[c] + p[c];
        x[(long long)r * E + c] = v;
        if (xh) xh[(long long)r * E + c] = from_f32<ActT>(v);
    }
}
template <typename ActT>
void launch_sbeam_embed_last(const StdBeamState& st, int max_rows, int W, const float* table, const float* pe, int E, float* x, ActT* xh,
                             cudaStream_t s) {
    if (max_rows <= 0) return;
    sbeam_embed_last_kernel<ActT><<<(max_rows + 7) / 8, 256, 0, s>>>(st, W, table, pe, E, x, xh);
}
template void launch_sbeam_embed_last<float>(const StdBeamState&, int, int, const float*, const float*, int, float*, float*, cudaStream_t);
template void launch_sbeam_embed_last<__nv_bfloat16>(const StdBeamState&, int, int, const float*, const float*, int, float*, __nv_bfloat16*, cudaStream_t);

template <typename ActT>
__global__ void sbeam_cache_update_kernel(StdBeamState st, int W, const ActT* __restrict__ qkv_all, long long qkv_layer_stride, int qkv_ld, int E,
                                          const ActT* __restrict__ kc_cur, const ActT* __restrict__ vc_cur, ActT* __restrict__ kc_next,
                                          ActT* __restrict__ vc_next, long long cache_layer_stride, long long cache_cand_stride) {
    const int cn = blockIdx.x, l = blockIdx.y;
    if (st.ctrl[2]) return;                          // the search has ended: the caches are not read again
    const int parent = st.parent[cn];
    const int r = st.cand_row[parent];
    if (r < 0) return;                               // continuation of a finished hypothesis: never decoded again
    const long long lo = (long long)l * cache_layer_stride;
    const ActT* ks = kc_cur + lo + (long long)parent * cache_cand_stride;
    const ActT* vs = vc_cur + lo + (long long)parent * cache_cand_stride;
    ActT* kd = kc_next + lo + (long long)cn * cache_cand_stride;
    ActT* vd = vc_next + lo + (long long)cn * cache_cand_stride;
    constexpr int VEC = 16 / (int)sizeof(ActT);
    const long long nvec = (long long)(W - 1) * E / VEC;
    const uint4* ks4 = reinterpret_cast<const uint4*>(ks);
    const uint4* vs4 = reinterpret_cast<const uint4*>(vs);
    uint4* kd4 = reinterpret_cast<uint4*>(kd);
    uint4* vd4 = reinterpret_cast<uint4*>(vd);
    for (long long i = threadIdx.x; i < nvec; i += blockDim.x) { kd4[i] = ks4[i]; vd4[i] = vs4[i]; }
    const ActT* src = qkv_all + (long long)l * qkv_layer_stride + (long long)r * qkv_ld;
    for (int col = threadIdx.x; col < E; col += blockDim.x) {
        kd[(long long)(W - 1) * E + col] = src[E + col];
        vd[(long long)(W - 1) * E + col] = src[2 * E + col];
    }
}
template <typename ActT>
void launch_sbeam_cache_update(const StdBeamState& st, int W, const ActT* qkv_all, long long qkv_layer_stride, int n_layers, int qkv_ld, int E,
                               const ActT* kc_cur, const ActT* vc_cur, ActT* kc_next, ActT* vc_next, long long cache_layer_stride,
                               long long cache_cand_stride, cudaStream_t s) {
    sbeam_cache_update_kernel<ActT><<<dim3(st.B * st.K, n_layers), 256, 0, s>>>(st, W, qkv_all, qkv_layer_stride, qkv_ld, E, kc_cur, vc_cur, kc_next, vc_next,
                                                                               cache_layer_stride, cache_cand_stride);
}
template void launch_sbeam_cache_update<float>(const StdBeamState&, int, const float*, long long, int, int, int, const float*, const float*, float*, float*,
                                               long long, long long, cudaStream_t);
template void launch_sbeam_cache_update<__nv_bfloat16>(const StdBeamState&, int, const __nv_bfloat16*, long long, int, int, int, const __nv_bfloat16*,
                                                       const __nv_bfloat16*, __nv_bfloat16*, __nv_bfloat16*, long long, long long, cudaStream_t);

__global__ void sbeam_init_kernel(StdBeamState st) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < st.B; b += gridDim.x * blockDim.x) {
        st.y_cur[(long long)b * st.ldw] = st.bos;
        st.score_cur[b] = 0.f;
    }
    if (blockIdx.x == 0 && threadIdx.x < 8) st.ctrl[threadIdx.x] = 0;
}
void launch_sbeam_init(const StdBeamState& st, cudaStream_t s) { sbeam_init_kernel<<<8, 256, 0, s>>>(st); }

}  // namespace ttb
