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
// The continuous loop (ttb_beam_search_generate_batches) runs the same step with group-aware prepare / select kernels.
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
// `torch.log(torch.softmax(x, -1))` at :111 / :150).  Absent hypotheses (continuous loop: cand_row -2) are skipped.
__global__ void __launch_bounds__(256) sbeam_scores_kernel(StdBeamState st, int C, const float* __restrict__ logits) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= C || st.ctrl[2]) return;
    const int V = st.V, r = st.cand_row[c];
    if (r == -2) return;
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

// Selection of one query (the whole CTA): the K best of its n = beam * V continuation scores `tot` in the order
// torch.topk(sorted=True) returns them on the CPU backend (ties between exactly equal scores — the "-35" continuations of
// finished hypotheses — are decided by libstdc++'s partial_sort / nth_element, emulated in topk_emul.cuh), then the new
// hypotheses dst0 + j = hypothesis src0 + parent (W tokens) + chosen token; with `out` also its rows [K][W + 1] there.
// Returns, in thread 0, how many of the new hypotheses contain EOS.
__device__ int sbeam_select_query(const StdBeamState& st, VF* s_e, const float* tot, int n, int src0, int dst0, int W, long long* out) {
    __shared__ int s_fin;
    const int V = st.V, K = st.K;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { s_e[i].v = tot[i]; s_e[i].i = i; }
    if (threadIdx.x == 0) s_fin = 0;
    __syncthreads();
    if (threadIdx.x == 0) topk_sorted_torch_cpu_(s_e, n, K);
    __syncthreads();
    int n_fin = 0;
    for (int j = warp; j < K; j += n_warps) {
        const int idx = s_e[j].i;
        const int parent = idx / V, ch = idx % V;
        const int* src = st.y_cur + (long long)(src0 + parent) * st.ldw;
        int* dst = st.y_next + (long long)(dst0 + j) * st.ldw;
        long long* o = out ? out + (long long)j * (W + 1) : nullptr;
        int fin = (ch == st.eos) ? 1 : 0;
        for (int c = lane; c < W; c += 32) {
            const int t = src[c];
            dst[c] = t;
            if (o) o[c] = t;
            fin |= (t == st.eos) ? 1 : 0;
        }
        if (lane == 0) {
            dst[W] = ch;
            if (o) o[W] = ch;
            st.score_next[dst0 + j] = s_e[j].v;
            if (st.parent) st.parent[dst0 + j] = src0 + parent;
        }
        fin = __any_sync(0xffffffffu, fin);
        if (lane == 0 && fin) ++n_fin;
    }
    if (lane == 0 && n_fin) atomicAdd(&s_fin, n_fin);
    __syncthreads();
    return s_fin;
}

// One CTA per query (generate(): query b holds hypotheses b beam .. and writes b K ..)
__global__ void __launch_bounds__(256) sbeam_select_kernel(StdBeamState st, int beam, int W) {
    extern __shared__ __align__(8) unsigned char s_sel_raw[];
    if (st.ctrl[2]) return;                          // step enqueued behind the end of the search
    const int b = blockIdx.x;
    const int n_fin = sbeam_select_query(st, reinterpret_cast<VF*>(s_sel_raw), st.total + (long long)b * beam * st.V, beam * st.V, b * beam,
                                         b * st.K, W, nullptr);
    if (threadIdx.x == 0) {
        if (n_fin) atomicAdd(&st.ctrl[1], n_fin);
        __threadfence();
        if (atomicAdd(&st.ctrl[4], 1) == (int)gridDim.x - 1) {   // last CTA of the step: stop test, step count
            __threadfence();
            st.ctrl[4] = 0;
            st.ctrl[3] += 1;
            if (W > 1 && atomicAdd(&st.ctrl[1], 0) == st.B * st.K) st.ctrl[2] = 1;   // the first step (W = 1) never stops (:106-125)
        }
    }
}
constexpr size_t kSelectSmemMax = 200 * 1024;
bool sbeam_select_fits(int beam, int V) { return (size_t)beam * V * sizeof(VF) <= kSelectSmemMax; }
int launch_sbeam_select(const StdBeamState& st, int beam, int W, cudaStream_t s) {
    const size_t smem = (size_t)beam * st.V * sizeof(VF);
    if (!sbeam_select_fits(beam, st.V)) return -1;
    if (smem > 48 * 1024 && ensure_dyn_smem(sbeam_select_kernel, (int)kSelectSmemMax)) return 1;
    sbeam_select_kernel<<<st.B, 256, smem, s>>>(st, beam, W);
    return 0;
}

// ---- KV caches --------------------------------------------------------------------------------------------------------
template <typename ActT>
__global__ void sbeam_embed_last_kernel(StdBeamState st, const float* __restrict__ table, const float* __restrict__ pe, int E,
                                        float* __restrict__ x, ActT* __restrict__ xh) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= st.ctrl[0]) return;
    const int4 d = st.desc_self[r];                  // {hypothesis, W - 1, token at W - 1, -}
    const float* e = table + (long long)d.z * E;
    const float* p = pe + (long long)(d.y + 1) * E;  // position W - 1 -> row W of the table (row 0 = zeros, embeddings.py:47)
    for (int c = lane; c < E; c += 32) {
        const float v = e[c] + p[c];
        x[(long long)r * E + c] = v;
        if (xh) xh[(long long)r * E + c] = from_f32<ActT>(v);
    }
}
template <typename ActT>
void launch_sbeam_embed_last(const StdBeamState& st, int max_rows, const float* table, const float* pe, int E, float* x, ActT* xh, cudaStream_t s) {
    if (max_rows <= 0) return;
    sbeam_embed_last_kernel<ActT><<<(max_rows + 7) / 8, 256, 0, s>>>(st, table, pe, E, x, xh);
}
template void launch_sbeam_embed_last<float>(const StdBeamState&, int, const float*, const float*, int, float*, float*, cudaStream_t);
template void launch_sbeam_embed_last<__nv_bfloat16>(const StdBeamState&, int, const float*, const float*, int, float*, __nv_bfloat16*, cudaStream_t);

template <typename ActT>
__global__ void sbeam_cache_update_kernel(StdBeamState st, const ActT* __restrict__ qkv_all, long long qkv_layer_stride, int qkv_ld, int E,
                                          const ActT* __restrict__ kc_cur, const ActT* __restrict__ vc_cur, ActT* __restrict__ kc_next,
                                          ActT* __restrict__ vc_next, long long cache_layer_stride, long long cache_cand_stride) {
    const int cn = blockIdx.x, l = blockIdx.y;
    if (st.ctrl[2]) return;                          // the search has ended: the caches are not read again
    const int parent = st.parent[cn];
    if (parent < 0) return;                          // continuous loop: no hypothesis here
    const int r = st.cand_row[parent];
    if (r < 0) return;                               // continuation of a finished hypothesis: never decoded again
    const int f = st.desc_self[r].y;                 // cached positions of the parent = W - 1
    const long long lo = (long long)l * cache_layer_stride;
    const ActT* ks = kc_cur + lo + (long long)parent * cache_cand_stride;
    const ActT* vs = vc_cur + lo + (long long)parent * cache_cand_stride;
    ActT* kd = kc_next + lo + (long long)cn * cache_cand_stride;
    ActT* vd = vc_next + lo + (long long)cn * cache_cand_stride;
    constexpr int VEC = 16 / (int)sizeof(ActT);
    const long long nvec = (long long)f * E / VEC;
    const uint4* ks4 = reinterpret_cast<const uint4*>(ks);
    const uint4* vs4 = reinterpret_cast<const uint4*>(vs);
    uint4* kd4 = reinterpret_cast<uint4*>(kd);
    uint4* vd4 = reinterpret_cast<uint4*>(vd);
    for (long long i = threadIdx.x; i < nvec; i += blockDim.x) { kd4[i] = ks4[i]; vd4[i] = vs4[i]; }
    const ActT* src = qkv_all + (long long)l * qkv_layer_stride + (long long)r * qkv_ld;
    for (int col = threadIdx.x; col < E; col += blockDim.x) {
        kd[(long long)f * E + col] = src[E + col];
        vd[(long long)f * E + col] = src[2 * E + col];
    }
}
template <typename ActT>
void launch_sbeam_cache_update(const StdBeamState& st, const ActT* qkv_all, long long qkv_layer_stride, int n_layers, int qkv_ld, int E,
                               const ActT* kc_cur, const ActT* vc_cur, ActT* kc_next, ActT* vc_next, long long cache_layer_stride,
                               long long cache_cand_stride, cudaStream_t s) {
    sbeam_cache_update_kernel<ActT><<<dim3(st.B * st.K, n_layers), 256, 0, s>>>(st, qkv_all, qkv_layer_stride, qkv_ld, E, kc_cur, vc_cur, kc_next, vc_next,
                                                                               cache_layer_stride, cache_cand_stride);
}
template void launch_sbeam_cache_update<float>(const StdBeamState&, const float*, long long, int, int, int, const float*, const float*, float*, float*,
                                               long long, long long, cudaStream_t);
template void launch_sbeam_cache_update<__nv_bfloat16>(const StdBeamState&, const __nv_bfloat16*, long long, int, int, int, const __nv_bfloat16*,
                                                       const __nv_bfloat16*, __nv_bfloat16*, __nv_bfloat16*, long long, long long, cudaStream_t);

__global__ void sbeam_init_kernel(StdBeamState st) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < st.B; b += gridDim.x * blockDim.x) {
        st.y_cur[(long long)b * st.ldw] = st.bos;
        st.score_cur[b] = 0.f;
    }
    if (blockIdx.x == 0 && threadIdx.x < 8) st.ctrl[threadIdx.x] = 0;
}
void launch_sbeam_init(const StdBeamState& st, cudaStream_t s) { sbeam_init_kernel<<<8, 256, 0, s>>>(st); }

// ---- continuous batching: several batches share the query slots of one loop ----------------------------------------
// Slot q holds query cb.slots.slot_q[q] of batch cb.slots.slot_group[q] (-1: free) and hypotheses q K .. q K + K - 1.  A batch keeps in
// its SbGroup what the reference couples across the queries of a batch: width, hypotheses per query, step count and the
// stop rule.  In a query's first step only hypothesis 0 exists (the reference starts from the BOS column, beam = 1): the
// others are absent (cand_row -2), with no decoder rows and no continuations, so its selection sees the V scores
// generate() sees, in the same order.

// Admission of batch `grp` (Bi queries) into the first Bi free slots: BOS hypothesis with score 0 (both buffer sets: the
// coming step reads one of them), source lengths and the batch's record.  One CTA, between two steps.
__global__ void __launch_bounds__(1024) sbeam_admit_kernel(StdBeamState st, SbTable cb, int grp, int Bi, const int* __restrict__ srclen_in,
                                                           long long* out) {
    extern __shared__ int s_slots[];   // [Bi] slots taken, in batch order
    __shared__ int s_nfree;
    const int K = st.K;
    if ((threadIdx.x >> 5) == 0) {
        const int taken = take_free_slots(cb.slots.slot_group, st.B, Bi, s_slots);
        if (threadIdx.x == 0) s_nfree = taken;
    }
    __syncthreads();
    if (s_nfree < Bi) {
        if (threadIdx.x == 0) st.ctrl[SBC_ADM_ERR] = 1;
        return;
    }
    for (int j = threadIdx.x; j < Bi; j += blockDim.x) {
        const int q = s_slots[j];
        const long long c = (long long)q * K;
        cb.slots.adm_slots[j] = q;
        cb.slots.slot_group[q] = grp;
        cb.slots.slot_q[q] = j;
        const_cast<int*>(st.src_len)[q] = srclen_in[j];
        st.y_cur[c * st.ldw] = st.bos;
        st.y_next[c * st.ldw] = st.bos;
        st.score_cur[c] = 0.f;
        st.score_next[c] = 0.f;
    }
    if (threadIdx.x == 0) {
        SbGroup g{};
        g.out = out;
        g.B = Bi; g.W = 1; g.beam = 1;
        cb.groups[grp] = g;
        st.ctrl[SBC_USED] += Bi;
    }
}
int launch_sbeam_admit(const StdBeamState& st, const SbTable& cb, int grp, int Bi, const int* srclen_in, long long* out, cudaStream_t s) {
    const size_t smem = (size_t)Bi * sizeof(int);
    if (ensure_dyn_smem(sbeam_admit_kernel, (int)smem)) return 1;   // error recorded by ensure_dyn_smem
    sbeam_admit_kernel<<<1, 1024, smem, s>>>(st, cb, grp, Bi, srclen_in, out);
    return 0;
}

// Prepare step of the continuous loop: sbeam_prepare per hypothesis with the width of its batch (one warp each), live rows
// by a block-wide scan in hypothesis order.  st.fin: 0 live, 1 contains EOS, 2 absent.
__global__ void __launch_bounds__(1024) sbeam_prepare_groups_kernel(StdBeamState st, SbTable cb) {
    const int K = st.K, C = st.B * K;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
    for (int c = warp; c < C; c += n_warps) {
        const int g = cb.slots.slot_group[c / K];
        if (g < 0 || c % K >= cb.groups[g].beam) {
            if (lane == 0) st.fin[c] = 2;
            continue;
        }
        const int W = cb.groups[g].W;
        const int* row = st.y_cur + (long long)c * st.ldw;
        int fin = 0;
        for (int j = lane; j < W; j += 32) fin |= (row[j] == st.eos) ? 1 : 0;
        fin = __any_sync(0xffffffffu, fin);
        if (lane == 0) { st.fin[c] = fin; st.c_front[c] = W - 1; }
    }
    __syncthreads();
    __shared__ int s_rows;
    if (threadIdx.x == 0) s_rows = 0;
    __syncthreads();
    for (int c0 = 0; c0 < C; c0 += blockDim.x) {
        const int c = c0 + threadIdx.x;
        const int f = c < C ? st.fin[c] : 2;
        const int live = f == 0 ? 1 : 0;
        int e, e2, t, t2;
        block_scan2(live, 0, e, e2, t, t2);
        if (c < C) st.cand_row[c] = live ? s_rows + e : (f == 2 ? -2 : -1);
        if (live) {
            const int r = s_rows + e, q = c / K, w1 = st.c_front[c];
            st.row_cand[r] = c;
            st.row_query[r] = q;
            st.desc_self[r] = make_int4(c, w1, st.y_cur[(long long)c * st.ldw + w1], 0x7fffffff);
            st.desc_cross[r] = make_int4(q, 0, 0, st.src_len[q]);
        }
        __syncthreads();
        if (threadIdx.x == 0) s_rows += t;
        __syncthreads();
    }
    if (threadIdx.x == 0) st.ctrl[0] = s_rows;
}
void launch_sbeam_prepare_groups(const StdBeamState& st, const SbTable& cb, cudaStream_t s) { sbeam_prepare_groups_kernel<<<1, 1024, 0, s>>>(st, cb); }

// Select step of the continuous loop: one CTA per slot, the selection of its query with its batch's width and beam, the new
// hypotheses also written to the batch's output at its new width.  The CTA that arrives last closes the step of every open
// batch with the reference's stop rule (:106-127, :169: after a step with W > 1 in which every hypothesis of the batch
// contains EOS, or after max_len - 1 steps), frees the slots of the batches that stopped and posts the loop's word.
__global__ void __launch_bounds__(256) sbeam_select_groups_kernel(StdBeamState st, SbTable cb) {
    extern __shared__ __align__(8) unsigned char s_sel_raw[];
    __shared__ int s_last, s_live;
    const int q = blockIdx.x, K = st.K, V = st.V;
    const int g = cb.slots.slot_group[q];
    if (g >= 0) {
        SbGroup* gr = &cb.groups[g];
        const int W = gr->W;
        const int n_fin = sbeam_select_query(st, reinterpret_cast<VF*>(s_sel_raw), st.total + (long long)q * K * V, gr->beam * V, q * K, q * K, W,
                                             gr->out + (long long)cb.slots.slot_q[q] * K * (W + 1));
        if (threadIdx.x == 0 && n_fin) atomicAdd(&gr->n_eos, n_fin);
    } else {
        for (int k = threadIdx.x; k < K; k += blockDim.x) st.parent[q * K + k] = -1;   // no cache to carry
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(&st.ctrl[SBC_TICKET], 1) == (int)gridDim.x - 1;
        s_live = 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int gi = threadIdx.x; gi < cb.n_groups; gi += blockDim.x) {
        SbGroup* gr = &cb.groups[gi];
        if (gr->closed) continue;
        const int n_eos = atomicAdd(&gr->n_eos, 0);
        gr->n_eos = 0;
        gr->steps += 1;
        if ((gr->W > 1 && n_eos == gr->B * K) || gr->steps >= st.max_len - 1) {
            gr->closed = 1;   // W stays the width before the batch's last step: its output is W + 1 wide
            atomicSub(&st.ctrl[SBC_USED], gr->B);
        } else {
            gr->W += 1;
            gr->beam = K;
            atomicAdd(&s_live, gr->B * K - n_eos);
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < st.B; b += blockDim.x) {
        const int gb = cb.slots.slot_group[b];
        if (gb >= 0 && cb.groups[gb].closed) cb.slots.slot_group[b] = -1;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        st.ctrl[SBC_TICKET] = 0;
        const int seq = st.ctrl[SBC_SEQ] + 1;
        st.ctrl[SBC_SEQ] = seq;
        const unsigned long long word = ((unsigned long long)(seq & 0xffffff) << 40) | ((unsigned long long)(st.ctrl[SBC_USED] & 0xffff) << 24) |
                                        (unsigned long long)(s_live & 0xffffff);
        __threadfence_system();
        reinterpret_cast<volatile unsigned long long*>(st.host_ctrl)[seq & 3] = word;
    }
}
int launch_sbeam_select_groups(const StdBeamState& st, const SbTable& cb, int max_beam, cudaStream_t s) {
    const size_t smem = (size_t)max_beam * st.V * sizeof(VF);
    if (!sbeam_select_fits(max_beam, st.V)) return -1;
    if (smem > 48 * 1024 && ensure_dyn_smem(sbeam_select_groups_kernel, (int)kSelectSmemMax)) return 1;
    sbeam_select_groups_kernel<<<st.B, 256, smem, s>>>(st, cb);
    return 0;
}

}  // namespace ttb
