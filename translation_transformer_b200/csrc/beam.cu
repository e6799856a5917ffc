// Device side of the speculative beam search ("try all the drafts" mode).
// Reference: /root/reference/src/decoding/speculative_decoding.py:428-598 (loop), :294-400 (sample),
// :847-869 (accepted lengths), :871-904 (nucleus truncation), :177-238 (top-k per query).
//
// Per iteration the engine runs
//   beam_prepare  -> per-candidate bookkeeping (first free slot, finished flag, live-row prefix)
//   beam_embed_cached -> last token + draft tokens of every live (candidate, draft) row
//   decoder stack on the dl+1 positions of those rows (the prefix comes from the candidate's KV cache),
//   classifier GEMM
//   beam_stats    -> per (row, position): softmax max/sum, the n_best largest logits (sorted), size of
//                    the nucleus-truncated support
//   beam_choose   -> accepted length of every draft, best draft per candidate (torch-CPU topk(1) order)
//   beam_expand   -> per query: scores of all leaves of the continuation trees of its candidates, the
//                    n_best best become the next candidates
//   (loop control: all-finished flag, trailing empty columns, acceptance statistics -> the last CTA of beam_expand)
#include "kernels.cuh"
#include "topk_emul.cuh"

namespace ttb {
// Accumulators of the loop control behind the BC_COUNT control words (reset by the CTA that finalises an iteration), and the
// loop state the device carries itself so that an iteration can be enqueued before the host has read the outcome of the one
// before it: width of the token matrix and number of the CURRENT iteration, advanced by the CTA that closes the iteration
// with the same rule the host applies (engine.cu:beam_api, speculative_decoding.py:452-470)
constexpr int BCX_ALL_FIN = BC_COUNT, BCX_MIN_PAD = BC_COUNT + 1, BCX_ACC = BC_COUNT + 2, BCX_CNT = BC_COUNT + 3, BCX_TICKET = BC_COUNT + 4,
              BCX_W = BC_COUNT + 5, BCX_ITER = BC_COUNT + 6,
              BCX_NLIVE_NEXT = BC_COUNT + 8,   // accumulator: new hypotheses without EOS = live candidates of the next iteration
              BCX_DONE = BC_COUNT + 7;   // the loop has ended (every hypothesis finished, length budget used up, or an error): set by the CTA that
                                         // closes an iteration with the reference's own stop rule, so that an iteration the host has
                                         // enqueued ahead of reading this one's outcome is a no-op on the device


// drafts of candidate c (query q): all N source drafts, or in smart mode the library windows keyed by its last token
__device__ __forceinline__ int cand_n_drafts(const BeamState& st, int c) { return st.smart ? st.c_cnt[c] : st.N; }
__device__ __forceinline__ const int* cand_draft(const BeamState& st, int c, int q, int j) {
    if (!st.smart) return st.drafts + ((long long)q * st.N + j) * st.dl0;
    const int n = st.tok_list[((long long)q * st.V + st.c_last[c]) * st.N + j];
    return st.drafts + ((long long)q * st.n_lib + n) * st.dl0 + 1;      // skip the key token
}

// ---- smart drafts: windows of the library grouped by their first token (get_vocab_tokens_bool_lib, :402-420) ------
__global__ void beam_build_lib_kernel(BeamState st) {
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= st.B * st.V) return;
    const int b = w / st.V, v = w % st.V;
    int* list = st.tok_list + (long long)w * st.N;
    int cnt = 0;
    for (int n0 = 0; n0 < st.n_lib && cnt < st.N; n0 += 32) {
        const int n = n0 + lane;
        const bool hit = n < st.n_lib && st.drafts[((long long)b * st.n_lib + n) * st.dl0] == v;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        const int pos = cnt + __popc(m & ((1u << lane) - 1u));
        if (hit && pos < st.N) list[pos] = n;                 // the first N windows in library order (:419)
        cnt += __popc(m);
    }
    if (lane == 0) {
        if (cnt == 0) { list[0] = 0; cnt = 1; }              // "each line needs at least one draft" (:418)
        st.tok_cnt[w] = cnt < st.N ? cnt : st.N;
    }
}
void launch_beam_build_lib(const BeamState& st, cudaStream_t s) {
    const int warps = st.B * st.V;
    beam_build_lib_kernel<<<(warps + 7) / 8, 256, 0, s>>>(st);
}

// ---- prepare ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) beam_prepare_kernel(BeamState st, int C, int beam, int dl) {
    if (st.ctrl[BCX_DONE]) {   // enqueued ahead of the end of the loop: no live rows, every kernel behind this one exits at once
        if (threadIdx.x == 0) { st.ctrl[BC_NLIVE_ROWS] = 0; st.ctrl[BC_NLIVE_CANDS] = 0; }
        return;
    }
    const int W = st.ctrl[BCX_W];
    // one warp per candidate row, coalesced scan: first PAD column, EOS anywhere, a real token behind the first PAD
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
    for (int c = warp; c < C; c += n_warps) {
        const int* row = st.cand_cur + (long long)c * st.ldw;
        int first_pad = 0x7fffffff, last_real = -1, fin = 0;
        for (int j = lane; j < W; j += 32) {
            const int t = row[j];
            if (t == st.eos) fin = 1;
            if (t == st.pad) first_pad = min(first_pad, j); else last_real = max(last_real, j);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            first_pad = min(first_pad, __shfl_xor_sync(0xffffffffu, first_pad, o));
            last_real = max(last_real, __shfl_xor_sync(0xffffffffu, last_real, o));
            fin |= __shfl_xor_sync(0xffffffffu, fin, o);
        }
        if (lane == 0) {
            const int slot0 = first_pad == 0x7fffffff ? -1 : first_pad;
            const int hole = slot0 >= 0 && last_real > slot0;   // a real token after a PAD: draft slots not contiguous
            st.c_slot0[c] = slot0;
            st.c_fin[c] = fin;
            if (hole || slot0 < 1 || slot0 + dl + 1 > W) atomicExch(&st.ctrl[BC_ERROR], 3);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0, live = 0, lmax = 0;
        for (int c = 0; c < C; ++c) {
            st.c_rowbase[c] = run;
            const int slot0 = st.c_slot0[c];
            st.c_front[c] = max(0, slot0 - 1);   // clamped: an inconsistent hypothesis raises BC_ERROR, its rows are discarded
            int cnt = st.N;
            if (st.smart) {
                // last meaningful token = the one before the first PAD (hypotheses without interior PADs), or the last
                // column when the row has no PAD at all (:693-697)
                const int last = st.cand_cur[(long long)c * st.ldw + (slot0 >= 1 ? slot0 - 1 : (slot0 < 0 ? W - 1 : 0))];
                st.c_last[c] = last;
                cnt = st.tok_cnt[(c / beam) * st.V + last];
                st.c_cnt[c] = cnt;
            }
            lmax = max(lmax, cnt);
            if (!st.c_fin[c]) {
                run += cnt;
                if (!st.smart) {
                    st.live_cand[live] = c;
                    st.live_query[live] = c / beam;
                    const int f = st.c_front[c];
                    st.desc_self[live] = make_int4(c, f, st.cand_cur[(long long)c * st.ldw + f], 0x7fffffff);
                    st.desc_cross[live] = make_int4(c / beam, 0, 0, st.src_len[c / beam]);
                }
                ++live;
            }
        }
        st.ctrl[BC_NLIVE_ROWS] = run;
        st.ctrl[BC_NLIVE_CANDS] = st.smart ? run : live;     // attention groups: candidates, or single rows in smart mode
        st.ctrl[BC_LMAX] = lmax;
    }
    __syncthreads();
    if (st.smart) {   // every live row is its own attention group: row -> (candidate, query, library window)
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            if (st.c_fin[c]) continue;
            const int q = c / beam, base = st.c_rowbase[c], cnt = st.c_cnt[c];
            const int* list = st.tok_list + ((long long)q * st.V + st.c_last[c]) * st.N;
            const int f = st.c_front[c];
            const int4 ds = make_int4(c, f, st.cand_cur[(long long)c * st.ldw + f], 0x7fffffff);
            const int4 dc = make_int4(q, 0, 0, st.src_len[q]);
            for (int j = 0; j < cnt; ++j) {
                st.live_cand[base + j] = c;
                st.live_query[base + j] = q;
                st.row_draft[base + j] = list[j];
                st.desc_self[base + j] = ds;
                st.desc_cross[base + j] = dc;
            }
        }
    }
}
void launch_beam_prepare(const BeamState& st, int C, int beam, int dl, cudaStream_t s) {
    beam_prepare_kernel<<<1, 1024, 0, s>>>(st, C, beam, dl);
}

// ---- decoder input: the candidate's prefix is in its KV cache -----------------------------------------------------
// Row t = (live candidate g, draft n, position i): token = last token of the candidate (i = 0) or draft token i-1,
// sequence position front + i.  Row order matches c_rowbase (rows of live candidate g start at g * N).
template <typename ActT>
__global__ void beam_embed_cached_kernel(BeamState st, int beam, int dl, const float* __restrict__ table, const float* __restrict__ pe,
                                         int E, float* __restrict__ x, ActT* __restrict__ xh) {
    pdl_wait();   // launched with the programmatic attribute: scheduled while the predecessor drains, starts when it is complete
    const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (t >= st.ctrl[BC_NLIVE_ROWS] * (dl + 1)) return;
    const int r = t / (dl + 1), i = t % (dl + 1);
    int c, f, tok;
    if (st.smart) {
        c = st.live_cand[r];
        f = st.c_front[c];
        tok = (i == 0) ? st.cand_cur[(long long)c * st.ldw + f]
                       : st.drafts[((long long)(c / beam) * st.n_lib + st.row_draft[r]) * st.dl0 + i];   // window token i (0 = key)
    } else {
        const int g = r / st.N, n = r % st.N;
        c = st.live_cand[g];
        f = st.c_front[c];
        tok = (i == 0) ? st.cand_cur[(long long)c * st.ldw + f] : st.drafts[((long long)(c / beam) * st.N + n) * st.dl0 + i - 1];
    }
    if (lane == 0) {   // the draft token at input position i is the "next draft token" of scored position i - 1
        if (i >= 1) st.row_tok[t - 1] = tok;
        if (i == dl) st.row_tok[t] = -1;
    }
    const float* e = table + (long long)tok * E;
    const float* p = pe + (long long)(f + i + 1) * E;
    for (int col = lane; col < E; col += 32) {
        const float v = e[col] + p[col];
        x[(long long)t * E + col] = v;
        if (xh) xh[(long long)t * E + col] = from_f32<ActT>(v);
    }
}
template <typename ActT>
void launch_beam_embed_cached(const BeamState& st, int beam, int max_rows, int dl, const float* table, const float* pe, int E,
                              float* x, ActT* xh, cudaStream_t s) {
    const int T = max_rows * (dl + 1);
    if (T <= 0) return;
    launch_pdl(beam_embed_cached_kernel<ActT>, dim3((T + 7) / 8), dim3(256), 0, s, st, beam, dl, table, pe, E, x, xh);
}
template void launch_beam_embed_cached<float>(const BeamState&, int, int, int, const float*, const float*, int, float*, float*, cudaStream_t);
template void launch_beam_embed_cached<__nv_bfloat16>(const BeamState&, int, int, int, const float*, const float*, int, float*, __nv_bfloat16*,
                                                      cudaStream_t);

template <typename ActT>
__global__ void beam_cache_update_kernel(BeamState st, int dl, const ActT* __restrict__ qkv_all, long long qkv_layer_stride, int qkv_ld,
                                         int E, const ActT* __restrict__ kc_cur, const ActT* __restrict__ vc_cur, ActT* __restrict__ kc_next,
                                         ActT* __restrict__ vc_next, long long cache_layer_stride, long long cache_cand_stride) {
    pdl_wait();   // launched with the programmatic attribute: scheduled while the predecessor drains, starts when it is complete
    if (st.ctrl[BCX_DONE]) return;   // the loop has ended (this iteration closed it, or it was enqueued behind the end): the caches are not read again
    const int cn = blockIdx.x, l = blockIdx.y;
    const int parent = st.n_parent[cn];
    if (parent < 0) return;                         // child of a finished hypothesis: never decoded again
    const int f = st.c_front[parent], keep = st.n_keep[cn], r = st.n_row[cn];
    const long long lo = (long long)l * cache_layer_stride;
    const ActT* ks = kc_cur + lo + (long long)parent * cache_cand_stride;
    const ActT* vs = vc_cur + lo + (long long)parent * cache_cand_stride;
    ActT* kd = kc_next + lo + (long long)cn * cache_cand_stride;
    ActT* vd = vc_next + lo + (long long)cn * cache_cand_stride;
    // parent prefix: f rows of E elements, 16-byte vectors (E * sizeof(ActT) is a multiple of 16)
    constexpr int VEC = 16 / (int)sizeof(ActT);
    const long long nvec = (long long)f * E / VEC;
    const uint4* ks4 = reinterpret_cast<const uint4*>(ks);
    const uint4* vs4 = reinterpret_cast<const uint4*>(vs);
    uint4* kd4 = reinterpret_cast<uint4*>(kd);
    uint4* vd4 = reinterpret_cast<uint4*>(vd);
    for (long long i = (long long)blockIdx.z * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.z * blockDim.x) { kd4[i] = ks4[i]; vd4[i] = vs4[i]; }
    if (blockIdx.z != 0) return;
    // positions f .. f + keep from the chosen draft row of this iteration
    const ActT* src = qkv_all + (long long)l * qkv_layer_stride + (long long)r * (dl + 1) * qkv_ld;
    for (int idx = threadIdx.x; idx < (keep + 1) * E; idx += blockDim.x) {
        const int i = idx / E, col = idx % E;
        kd[(long long)(f + i) * E + col] = src[(long long)i * qkv_ld + E + col];
        vd[(long long)(f + i) * E + col] = src[(long long)i * qkv_ld + 2 * E + col];
    }
}
template <typename ActT>
void launch_beam_cache_update(const BeamState& st, int dl, const ActT* qkv_all, long long qkv_layer_stride, int n_layers, int qkv_ld,
                              int E, const ActT* kc_cur, const ActT* vc_cur, ActT* kc_next, ActT* vc_next, long long cache_layer_stride,
                              long long cache_cand_stride, cudaStream_t s) {
    dim3 grid(st.B * st.K, n_layers, 4);   // z: four slices of the parent's prefix
    launch_pdl(beam_cache_update_kernel<ActT>, dim3(grid), dim3(256), 0, s, st, dl, qkv_all, qkv_layer_stride, qkv_ld, E, kc_cur, vc_cur, kc_next, vc_next,
                                                        cache_layer_stride, cache_cand_stride);
}
template void launch_beam_cache_update<float>(const BeamState&, int, const float*, long long, int, int, int, const float*, const float*, float*,
                                              float*, long long, long long, cudaStream_t);
template void launch_beam_cache_update<__nv_bfloat16>(const BeamState&, int, const __nv_bfloat16*, long long, int, int, int,
                                                      const __nv_bfloat16*, const __nv_bfloat16*, __nv_bfloat16*, __nv_bfloat16*, long long,
                                                      long long, cudaStream_t);

// ---- per (row, position) statistics -------------------------------------------------------------------
// One warp per distribution: softmax max / sum, the K largest logits in descending order (ties: lower
// token id first) and the size of the truncated support (exclusive cumulative probability < 0.9975,
// the best token always kept; speculative_decoding.py:886-899).
template <int VPL>
__global__ void __launch_bounds__(256) beam_stats_kernel(BeamState st, const float* __restrict__ logits, int dl) {
    pdl_wait();   // launched with the programmatic attribute: scheduled while the predecessor drains, starts when it is complete
    const int rp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (rp >= st.ctrl[BC_NLIVE_ROWS] * (dl + 1)) return;
    const int V = st.V, K = st.K;
    const float* p = logits + (long long)rp * V;
    float v[VPL];
    float mx = -INFINITY;
    const int want = st.row_tok[rp];
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
        const int c = lane + 32 * k;
        v[k] = c < V ? p[c] : -INFINITY;
        mx = fmaxf(mx, v[k]);
        if (c == want) st.tokv[rp] = v[k];
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) sum += (lane + 32 * k < V) ? expf(v[k] - mx) : 0.f;
    sum = warp_sum(sum);
    float* topv = st.topv + (long long)rp * K;
    int* topi = st.topi + (long long)rp * K;
    float my_v = -INFINITY;
    int my_i = -1;
    for (int j = 0; j < K; ++j) {
        float bv = -INFINITY;
        int bi = 0x7fffffff;
#pragma unroll
        for (int k = 0; k < VPL; ++k) {
            const int c = lane + 32 * k;
            if (c < V && (v[k] > bv || (v[k] == bv && c < bi))) { bv = v[k]; bi = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
#pragma unroll
        for (int k = 0; k < VPL; ++k)
            if (lane + 32 * k == bi) v[k] = -INFINITY;                          // taken
        // every lane holds (bv, bi) after the butterfly: lane j keeps entry j for the support scan below
        if (lane == (j & 31)) { my_v = bv; my_i = bi == 0x7fffffff ? -1 : bi; }
        if (lane == 0) { topv[j] = bv; topi[j] = bi == 0x7fffffff ? -1 : bi; }
    }
    {
        // truncated support: entry j is kept while the exclusive cumulative probability of entries 0..j-1 is < 0.9975
        // (sequential sum in entry order, as the reference's cumsum; K <= 32 entries live one per lane)
        int keep = 1;
        float cum = 0.f;
        for (int j = 1; j < K; ++j) {
            const float pv = __shfl_sync(0xffffffffu, my_v, j - 1);
            const int ij = __shfl_sync(0xffffffffu, my_i, j);
            if (ij < 0) break;
            cum += expf(pv - mx) / sum;
            if (cum < 0.9975f) keep = j + 1; else break;
        }
        if (lane == 0) {
            st.lmax[rp] = mx;
            st.lsum[rp] = sum;
            st.nkeep[rp] = keep;
        }
    }
}
void launch_beam_stats(const BeamState& st, const float* logits, int max_rows, int dl, cudaStream_t s) {
    const int T = max_rows * (dl + 1);
    if (T <= 0) return;
    if (st.V <= 320) launch_pdl(beam_stats_kernel<10>, dim3((T + 7) / 8), dim3(256), 0, s, st, logits, dl);
    else if (st.V <= 512) launch_pdl(beam_stats_kernel<16>, dim3((T + 7) / 8), dim3(256), 0, s, st, logits, dl);
    else launch_pdl(beam_stats_kernel<32>, dim3((T + 7) / 8), dim3(256), 0, s, st, logits, dl);
}

// ---- accepted lengths + best draft per candidate ------------------------------------------------------------
// One CTA per candidate.  "Is draft token a of draft n inside the truncated support of its position?" is evaluated for all
// (draft, position) pairs in parallel (two dependent global loads each instead of a chain of up to 2 dl per draft); the
// accepted length of a draft is the length of its leading run of hits.
// Per-candidate body, shared by the kernel of one batch and the one of the continuous loop: `dl` is the draft length of the
// candidate's batch, `rs` the scored positions per decoder row of the iteration (dl + 1, or more in the continuous loop),
// `lmax` the length the tie-break emulation pads to, tr_nacc / tr_pick the candidate's trace entries (or nullptr).
__device__ __forceinline__ void choose_candidate(const BeamState& st, int c, int q, int dl, int rs, int lmax, int par, unsigned char* s_hit,
                                                 int* s_nacc, int* tr_nacc, int* tr_pick) {
    const int N = st.N, K = st.K;
    const bool fin = st.c_fin[c] != 0;
    const int m = cand_n_drafts(st, c);                      // drafts of this candidate
    const int rb = st.c_rowbase[c];
    auto hit = [&](int n, int a) -> bool {
        const long long rp = (long long)(rb + n) * rs + a;
        const int keep = st.nkeep[rp];
        const int* ti = st.topi + rp * K;
        const int tok = cand_draft(st, c, q, n)[a];
        bool in = false;
        for (int j = 0; j < keep; ++j) in |= (ti[j] == tok);
        return in;
    };
    if (par && !fin) {
        for (int idx = threadIdx.x; idx < m * dl; idx += blockDim.x) s_hit[idx] = hit(idx / dl, idx % dl) ? 1 : 0;
    }
    __syncthreads();
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        int a = -1;
        if (n < m) {
            a = 0;
            if (!fin) {
                if (par) { while (a < dl && s_hit[n * dl + a]) ++a; }
                else { while (a < dl && hit(n, a)) ++a; }
            }
        }
        st.c_nacc[(long long)c * N + n] = a;
        if (n < 64) s_nacc[n] = a;
        if (tr_nacc) tr_nacc[n] = a;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int pick = 0;
        if (st.tie_break == 0 && lmax < 64) {
            pick = topk1_torch_cpu(s_nacc, lmax);
        } else {
            for (int n = 1; n < m; ++n) if (st.c_nacc[(long long)c * N + n] > st.c_nacc[(long long)c * N + pick]) pick = n;
        }
        st.c_pick[c] = pick;
        if (tr_pick) *tr_pick = pick;
    }
}
__global__ void __launch_bounds__(256) beam_choose_kernel(BeamState st, int C, int beam, int dl, int par) {
    pdl_wait();   // launched with the programmatic attribute: scheduled while the predecessor drains, starts when it is complete
    if (st.ctrl[BCX_DONE]) return;   // no-op iteration behind the end of the loop
    const int iter = st.ctrl[BCX_ITER];
    const int c = blockIdx.x;
    __shared__ int s_nacc[64];
    extern __shared__ unsigned char s_hit[];                 // [m][dl] when par
    if (c >= C) return;
    const int lmax = st.smart ? st.ctrl[BC_LMAX] : st.N;     // ragged groups are padded with -1 up to the longest (:206-223)
    const long long tr = (long long)iter * st.B * st.K + c;
    choose_candidate(st, c, c / beam, dl, dl + 1, lmax, par, s_hit, s_nacc, st.trace_nacc ? st.trace_nacc + tr * st.N : nullptr,
                     st.trace_pick ? st.trace_pick + tr : nullptr);
}
void launch_beam_choose(const BeamState& st, int C, int beam, int dl, cudaStream_t s) {
    const size_t smem = (size_t)st.N * (dl > 0 ? dl : 1);
    const int par = smem <= 40 * 1024 ? 1 : 0;
    launch_pdl(beam_choose_kernel, dim3(C), dim3(256), par ? smem : 0, s, st, C, beam, dl, par);
}

// ---- leaves of the continuation trees, n_best best per query, loop control ---------------------------------------
// Accumulators of the loop control behind the BC_COUNT control words (reset by the CTA that finalises an iteration)
// log softmax exactly as the reference evaluates it: log(exp(x - max) / sum)   (:378)
__device__ __forceinline__ float ref_logprob(float logit, float mx, float sum) { return logf(expf(logit - mx) / sum); }

// Per-query body, shared by the kernel of one batch and the one of the continuous loop: scores the leaves of the
// continuation trees of the `beam` candidates q * beam .. of query q (draft length dl of its batch, rs scored positions per
// decoder row, token-matrix width W), keeps the K best and writes them as the query's next candidates.  A candidate with
// c_fin == 2 is absent (continuous loop: a query's first iteration has one candidate): it has no leaves.  `err` receives
// error 4, `out` (optional) the new hypotheses at width W; `tally(k, fin, p, pads, has_eos)` feeds the loop control.
template <typename Tally>
__device__ __forceinline__ void expand_query(const BeamState& st, int q, int beam, int dl, int rs, int W, int* err, long long* out, Tally tally) {
    extern __shared__ float s_score[];                 // [beam][(dl+1)][K] leaf scores, -inf when absent
    __shared__ float s_red_v[256];
    __shared__ int s_red_i[256];
    __shared__ int s_sel[64];
    __shared__ int s_valid;
    const int K = st.K, N = st.N;
    const int per_c = (dl + 1) * K, total = beam * per_c;
    float* s_pre = s_score + total;                    // [beam][dl+2] running log-prob of the accepted path
    if (threadIdx.x == 0) s_valid = 0;
    // accepted-path prefix sums (sequential fp32 adds, same association as the reference's cumsum): one warp per
    // candidate, the terms are fetched by the lanes in parallel and added in order
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
    for (int cb = warp; cb < beam; cb += n_warps) {
        const int c = q * beam + cb;
        float run = 0.f;
        if (lane == 0) s_pre[cb * (dl + 2)] = 0.f;
        if (!st.c_fin[c]) {
            const int n = st.c_pick[c], a = st.c_nacc[(long long)c * N + n], r = st.c_rowbase[c] + n;
            for (int i0 = 0; i0 < a; i0 += 32) {
                float term = 0.f;
                if (i0 + lane < a) {
                    const long long rp = (long long)r * rs + i0 + lane;
                    term = ref_logprob(st.tokv[rp], st.lmax[rp], st.lsum[rp]);
                }
                const int cnt = min(32, a - i0);
                for (int i = 0; i < cnt; ++i) {
                    run += __shfl_sync(0xffffffffu, term, i);
                    if (lane == 0) s_pre[cb * (dl + 2) + i0 + i + 1] = run;
                }
            }
        }
    }
    __syncthreads();
    int my_valid = 0;
    for (int L = threadIdx.x; L < total; L += blockDim.x) {
        const int cb = L / per_c, p = (L % per_c) / K, j = L % K;
        const int c = q * beam + cb;
        const int cf = st.c_fin[c];
        float score = -INFINITY;
        if (cf == 2) {
            // absent candidate: no leaves
        } else if (cf) {
            // finished candidate: the artificial distribution leaves exactly one leaf, PAD at position 0,
            // with log-probability log(1) = 0
            if (p == 0 && j == 0) score = st.logp_cur[c] + 0.f;
        } else {
            const int n = st.c_pick[c], a = st.c_nacc[(long long)c * N + n], r = st.c_rowbase[c] + n;
            if (p <= a) {
                const long long rp = (long long)r * rs + p;
                const int tok = st.topi[rp * K + j];
                const float lg = st.topv[rp * K + j];
                const int* dr = cand_draft(st, c, q, n);
                // excluded: the draft token that continues the accepted path (p < a), BOS in the slot of the first
                // rejected draft token (p == a < dl); entries whose logit is exactly 0.0 vanish in the reference
                const int excl = (p < dl) ? (p < a ? dr[p] : st.bos) : -1;
                if (tok >= 0 && tok != excl && lg != 0.0f)
                    score = st.logp_cur[c] + (s_pre[cb * (dl + 2) + p] + ref_logprob(lg, st.lmax[rp], st.lsum[rp]));
            }
        }
        s_score[L] = score;
        my_valid += score != -INFINITY ? 1 : 0;
    }
    if (my_valid) atomicAdd(&s_valid, my_valid);
    __syncthreads();
    const bool ok = s_valid >= K;
    if (!ok && threadIdx.x == 0) atomicExch(err, 4);   // reference: assert min(group length) >= k (:195)
    for (int k = 0; ok && k < K; ++k) {                // K rounds of block-wide argmax (ties: lower leaf index)
        float bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int L = threadIdx.x; L < total; L += blockDim.x) {
            const float sc = s_score[L];
            if (sc > bv || (sc == bv && sc != -INFINITY && L < bi)) { bv = sc; bi = L; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        if (lane == 0) { s_red_v[warp] = bv; s_red_i[warp] = bi; }
        __syncthreads();
        if (warp == 0) {
            bv = lane < n_warps ? s_red_v[lane] : -INFINITY;
            bi = lane < n_warps ? s_red_i[lane] : 0x7fffffff;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            if (lane == 0) {
                s_sel[k] = bi;
                st.logp_next[q * K + k] = bv;
                s_score[bi] = -INFINITY;
            }
        }
        __syncthreads();
    }
    // materialise the K new candidates: one warp per candidate; the loop control's view of the new rows (PAD columns,
    // EOS anywhere, accepted draft tokens) is accumulated on the way
    for (int k = warp; ok && k < K; k += n_warps) {
        const int L = s_sel[k];
        const int cb = L / per_c, p = (L % per_c) / K, j = L % K;
        const int c = q * beam + cb;
        const int* src = st.cand_cur + (long long)c * st.ldw;
        int* dst = st.cand_next + (long long)(q * K + k) * st.ldw;
        long long* o_row = out ? out + (long long)k * W : nullptr;
        const int slot0 = st.c_slot0[c];
        const bool fin = st.c_fin[c] != 0;
        int n = 0, r = 0;
        if (!fin) { n = st.c_pick[c]; r = st.c_rowbase[c] + n; }
        const int* dr = fin ? st.drafts : cand_draft(st, c, q, n);
        const int tok = fin ? st.pad : st.topi[((long long)r * rs + p) * K + j];
        int pads = 0, has_eos = 0;
        for (int col = lane; col < W; col += 32) {
            int t = src[col];
            if (col >= slot0 && col <= slot0 + dl) {
                const int o = col - slot0;
                t = o < p ? dr[o] : (o == p ? tok : st.pad);
            }
            dst[col] = t;
            if (o_row) o_row[col] = t;
            pads += t == st.pad;
            has_eos |= t == st.eos;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            pads += __shfl_xor_sync(0xffffffffu, pads, o);
            has_eos |= __shfl_xor_sync(0xffffffffu, has_eos, o);
        }
        if (lane == 0) {
            st.acc_stat[q * K + k] = fin ? -1 : p;
            st.n_parent[q * K + k] = fin ? -1 : c;
            st.n_keep[q * K + k] = p;
            st.n_row[q * K + k] = r;
            tally(k, fin, p, pads, has_eos);
        }
    }
}

__global__ void __launch_bounds__(256) beam_expand_kernel(BeamState st, int beam, int dl) {
    pdl_wait();   // launched with the programmatic attribute: scheduled while the predecessor drains, starts when it is complete
    if (st.ctrl[BCX_DONE]) return;   // no-op iteration behind the end of the loop (the word of the last real iteration stays posted)
    const int q = blockIdx.x;
    const int W = st.ctrl[BCX_W];                      // rewritten only by the CTA that closes the iteration, after every CTA has arrived
    int* ctrl = st.ctrl;
    expand_query(st, q, beam, dl, dl + 1, W, &st.ctrl[BC_ERROR], nullptr, [ctrl](int, bool fin, int p, int pads, int has_eos) {
        if (!has_eos) { atomicAnd(&ctrl[BCX_ALL_FIN], 0); atomicAdd(&ctrl[BCX_NLIVE_NEXT], 1); }
        atomicMin(&ctrl[BCX_MIN_PAD], pads);
        if (!fin) { atomicAdd(&ctrl[BCX_ACC], p); atomicAdd(&ctrl[BCX_CNT], 1); }
    });
    // ---- loop control: the CTA that arrives last publishes the control words of the iteration (also into the pinned
    // host mirror, sequence number last) and resets the accumulators
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&st.ctrl[BCX_TICKET], 1) == (int)gridDim.x - 1) {
            __threadfence();
            const int acc = atomicAdd(&st.ctrl[BCX_ACC], 0), cnt = atomicAdd(&st.ctrl[BCX_CNT], 0);
            st.ctrl[BC_ALL_FINISHED] = atomicAdd(&st.ctrl[BCX_ALL_FIN], 0);
            st.ctrl[BC_EMPTY_COLS] = atomicAdd(&st.ctrl[BCX_MIN_PAD], 0);
            st.ctrl[BC_ACCEPTED] += acc;
            st.ctrl[BC_PRODUCED] += acc + cnt;
            const int nlive_next = atomicAdd(&st.ctrl[BCX_NLIVE_NEXT], 0);
            st.ctrl[BCX_ALL_FIN] = 1; st.ctrl[BCX_MIN_PAD] = 0x7fffffff; st.ctrl[BCX_ACC] = 0; st.ctrl[BCX_CNT] = 0; st.ctrl[BCX_TICKET] = 0;
            st.ctrl[BCX_NLIVE_NEXT] = 0;
            // width of the next iteration's token matrix (speculative_decoding.py:452-470, mirrored by the host loop)
            const int seq = st.ctrl[BCX_ITER] + 1;
            {
                const int empty = st.ctrl[BC_EMPTY_COLS], filled = W - empty, budget = st.max_len - filled - 1;
                const int grow = min(budget, dl) + 1 - empty;
                st.ctrl[BCX_W] = W + max(grow, 0);
                st.ctrl[BCX_ITER] = seq;
                // the reference's stop rule (:570-598 break on all finished; :452 while budget >= 1 and filled <= max_len)
                if (atomicAdd(&st.ctrl[BC_ERROR], 0) != 0 || st.ctrl[BC_ALL_FINISHED] != 0 || budget < 1 || filled > st.max_len) st.ctrl[BCX_DONE] = 1;
            }
            if (st.host_ctrl) {
                // what the host needs per iteration, packed into ONE 64-bit word of its own (pinned, mapped) memory:
                // sequence number | error | all finished | empty columns.  One posted store: no copy engine, no stream
                // synchronisation, no system-scope fence between this kernel and the cache update that follows it.
                // sequence (24 bits) | error (4) | all finished (1) | empty columns (12) | live candidates of the next iteration (16)
                const unsigned long long word = ((unsigned long long)(seq & 0xffffff) << 40) |
                                                ((unsigned long long)(atomicAdd(&st.ctrl[BC_ERROR], 0) & 0xf) << 36) |
                                                ((unsigned long long)(st.ctrl[BC_ALL_FINISHED] & 1) << 35) |
                                                ((unsigned long long)(st.ctrl[BC_EMPTY_COLS] & 0xfff) << 23) |
                                                ((unsigned long long)(nlive_next & 0xffff) << 7);
                // ring of four words: the host may read iteration i's word after iteration i + 1 (enqueued ahead) has posted its own
                reinterpret_cast<volatile unsigned long long*>(st.host_ctrl)[seq & 3] = word;
            }
        }
    }
}
void launch_beam_expand(const BeamState& st, int beam, int dl, cudaStream_t s) {
    const size_t smem = ((size_t)beam * (dl + 1) * st.K + (size_t)beam * (dl + 2)) * sizeof(float);
    if (ensure_dyn_smem(beam_expand_kernel, (int)smem)) return;   // error recorded; the launch below fails and cudaGetLastError reports it
    launch_pdl(beam_expand_kernel, dim3(st.B), dim3(256), smem, s, st, beam, dl);
}

// ---- continuous batching: several batches share the query slots of one loop ----------------------------------------
// Slot b holds query cb.slots.slot_q[b] of batch cb.slots.slot_group[b] (-1: free) and candidates b K .. b K + K - 1.  A batch keeps
// in its BcGroup what the reference couples across the queries of a batch: token-matrix width, draft length, iteration,
// the smart-mode padding length, counters, error and stop rule.  Every decoder call runs at the largest draft length of
// the open batches; a batch with a shorter one ignores the extra scored positions (the self-attention over the step
// positions is causal, so its own positions do not see them).  In a query's first iteration only candidate 0 exists (the
// reference starts from one BOS candidate per query): its other candidates are absent (c_fin = 2), with no rows and no
// leaves, so the leaf indices and their tie order are those of generate().
// Loop-level words behind the BCX_* ones: query slots in use; largest draft length of the open batches for the coming
// iteration; set when an admission found too few free slots (host bookkeeping broken)
constexpr int BCC_USED = BC_COUNT + 9, BCC_DLMAX = BC_COUNT + 10, BCC_ADM_ERR = BC_COUNT + 11;

// Admission of batch `grp` (Bi queries) into the first Bi free slots: hypotheses (BOS candidate), scores, drafts or the
// window library (lib_in windows per query in drafts_in), source lengths and the batch's record.  One CTA, between two
// iterations.
__global__ void __launch_bounds__(1024) beam_admit_kernel(BeamState st, BcTable cb, int grp, int Bi, const int* __restrict__ drafts_in, int lib_in,
                                                          const int* __restrict__ tok_cnt_in, const int* __restrict__ tok_list_in,
                                                          const int* __restrict__ srclen_in, long long* out, int* trace_nacc, int* trace_pick, int dl_first) {
    extern __shared__ int s_slots[];   // [Bi] slots taken, in batch order
    __shared__ int s_nfree;
    const int S = st.B, K = st.K, N = st.N, V = st.V, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0) {
        const int taken = take_free_slots(cb.slots.slot_group, S, Bi, s_slots);
        if (lane == 0) s_nfree = taken;
    }
    __syncthreads();
    if (s_nfree < Bi) {
        if (threadIdx.x == 0) st.ctrl[BCC_ADM_ERR] = 1;
        return;
    }
    for (int j = threadIdx.x; j < Bi; j += blockDim.x) {
        const int b = s_slots[j];
        cb.slots.adm_slots[j] = b;
        cb.slots.slot_group[b] = grp;
        cb.slots.slot_q[b] = j;
        const_cast<int*>(st.src_len)[b] = srclen_in[j];
    }
    // both hypothesis buffers (the coming iteration reads one of them and writes the other): BOS row for candidate 0
    const long long per_slot = (long long)K * st.ldw;
    for (long long idx = threadIdx.x; idx < (long long)Bi * per_slot; idx += blockDim.x) {
        const int j = (int)(idx / per_slot);
        const long long r = idx % per_slot;
        const int v = r == 0 ? st.bos : st.pad;
        st.cand_cur[s_slots[j] * per_slot + r] = v;
        st.cand_next[s_slots[j] * per_slot + r] = v;
    }
    for (int idx = threadIdx.x; idx < Bi * K; idx += blockDim.x) {
        const int c = s_slots[idx / K] * K + idx % K;
        st.logp_cur[c] = 0.f;
        st.logp_next[c] = 0.f;
    }
    int* drafts = const_cast<int*>(st.drafts);
    const long long per_in = (long long)(st.smart ? lib_in : N) * st.dl0, per_q = (long long)(st.smart ? st.n_lib : N) * st.dl0;
    for (long long idx = threadIdx.x; idx < (long long)Bi * per_in; idx += blockDim.x)
        drafts[s_slots[idx / per_in] * per_q + idx % per_in] = drafts_in[idx];
    if (st.smart) {
        for (long long idx = threadIdx.x; idx < (long long)Bi * V; idx += blockDim.x) st.tok_cnt[(long long)s_slots[idx / V] * V + idx % V] = tok_cnt_in[idx];
        const long long per_l = (long long)V * N;
        for (long long idx = threadIdx.x; idx < (long long)Bi * per_l; idx += blockDim.x)
            st.tok_list[s_slots[idx / per_l] * per_l + idx % per_l] = tok_list_in[idx];
    }
    if (threadIdx.x == 0) {
        BcGroup g{};
        g.out = out; g.trace_nacc = trace_nacc; g.trace_pick = trace_pick;
        g.B = Bi; g.W = st.w0; g.dl = dl_first;
        g.all_fin = 1; g.min_pad = 0x7fffffff;
        cb.groups[grp] = g;
        st.ctrl[BCC_USED] += Bi;
    }
}
int launch_beam_admit(const BeamState& st, const BcTable& cb, int grp, int Bi, const int* drafts_in, int lib_in, const int* tok_cnt_in,
                      const int* tok_list_in, const int* srclen_in, long long* out, int* trace_nacc, int* trace_pick, int dl_first, cudaStream_t s) {
    const size_t smem = (size_t)Bi * sizeof(int);
    if (ensure_dyn_smem(beam_admit_kernel, (int)smem)) return 1;   // error recorded by ensure_dyn_smem
    beam_admit_kernel<<<1, 1024, smem, s>>>(st, cb, grp, Bi, drafts_in, lib_in, tok_cnt_in, tok_list_in, srclen_in, out, trace_nacc, trace_pick, dl_first);
    return 0;
}

// Prepare step of the continuous loop: beam_prepare per candidate with the width / draft length of its batch; row bases
// and live lists by block-wide scans in candidate order.
__global__ void __launch_bounds__(1024) beam_prepare_groups_kernel(BeamState st, BcTable cb) {
    const int K = st.K, N = st.N, C = st.B * K;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
    for (int c = warp; c < C; c += n_warps) {
        const int g = cb.slots.slot_group[c / K];
        if (g < 0 || (c % K != 0 && cb.groups[g].iter == 0)) {   // free slot, or a candidate that does not exist yet
            if (lane == 0) st.c_fin[c] = 2;
            continue;
        }
        const int W = cb.groups[g].W, dl = cb.groups[g].dl;
        const int* row = st.cand_cur + (long long)c * st.ldw;
        int first_pad = 0x7fffffff, last_real = -1, fin = 0;
        for (int j = lane; j < W; j += 32) {
            const int t = row[j];
            if (t == st.eos) fin = 1;
            if (t == st.pad) first_pad = min(first_pad, j); else last_real = max(last_real, j);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            first_pad = min(first_pad, __shfl_xor_sync(0xffffffffu, first_pad, o));
            last_real = max(last_real, __shfl_xor_sync(0xffffffffu, last_real, o));
            fin |= __shfl_xor_sync(0xffffffffu, fin, o);
        }
        if (lane == 0) {
            const int slot0 = first_pad == 0x7fffffff ? -1 : first_pad;
            const int hole = slot0 >= 0 && last_real > slot0;
            st.c_slot0[c] = slot0;
            st.c_fin[c] = fin;
            if (hole || slot0 < 1 || slot0 + dl + 1 > W) atomicExch(&cb.groups[g].error, 3);
        }
    }
    __syncthreads();
    __shared__ int s_rows, s_live;
    if (threadIdx.x == 0) { s_rows = 0; s_live = 0; }
    __syncthreads();
    for (int c0 = 0; c0 < C; c0 += blockDim.x) {
        const int c = c0 + threadIdx.x, q = c / K;
        int rows = 0, live = 0, rl = 0;
        if (c < C && st.c_fin[c] != 2) {
            const int g = cb.slots.slot_group[q];
            rl = cb.groups[g].dl + 1;   // positions of the candidate's draft rows (the attention's per-group row length)
            const int slot0 = st.c_slot0[c];
            st.c_front[c] = max(0, slot0 - 1);
            int cnt = N;
            if (st.smart) {
                const int W = cb.groups[g].W;
                const int last = st.cand_cur[(long long)c * st.ldw + (slot0 >= 1 ? slot0 - 1 : (slot0 < 0 ? W - 1 : 0))];
                st.c_last[c] = last;
                cnt = st.tok_cnt[(long long)q * st.V + last];
                st.c_cnt[c] = cnt;
                atomicMax(&cb.groups[g].lmax, cnt);
            }
            if (!st.c_fin[c]) { rows = cnt; live = 1; }
        }
        int er, el, tr, tl;
        block_scan2(rows, live, er, el, tr, tl);
        if (c < C) st.c_rowbase[c] = s_rows + er;
        if (live && !st.smart) {
            const int i = s_live + el, f = st.c_front[c];
            st.live_cand[i] = c;
            st.live_query[i] = q;
            st.desc_self[i] = make_int4(c, f, st.cand_cur[(long long)c * st.ldw + f], rl);
            st.desc_cross[i] = make_int4(q, 0, 0, st.src_len[q]);
        }
        __syncthreads();
        if (threadIdx.x == 0) { s_rows += tr; s_live += tl; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        st.ctrl[BC_NLIVE_ROWS] = s_rows;
        st.ctrl[BC_NLIVE_CANDS] = st.smart ? s_rows : s_live;
    }
    if (st.smart) {   // every live row is its own attention group: row -> (candidate, query, library window)
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            if (st.c_fin[c]) continue;
            const int q = c / K, base = st.c_rowbase[c], cnt = st.c_cnt[c];
            const int* list = st.tok_list + ((long long)q * st.V + st.c_last[c]) * N;
            const int f = st.c_front[c];
            const int4 ds = make_int4(c, f, st.cand_cur[(long long)c * st.ldw + f], cb.groups[cb.slots.slot_group[q]].dl + 1);
            const int4 dc = make_int4(q, 0, 0, st.src_len[q]);
            for (int j = 0; j < cnt; ++j) {
                st.live_cand[base + j] = c;
                st.live_query[base + j] = q;
                st.row_draft[base + j] = list[j];
                st.desc_self[base + j] = ds;
                st.desc_cross[base + j] = dc;
            }
        }
    }
}
void launch_beam_prepare_groups(const BeamState& st, const BcTable& cb, cudaStream_t s) { beam_prepare_groups_kernel<<<1, 1024, 0, s>>>(st, cb); }

// Choose step of the continuous loop: beam_choose per candidate with its batch's draft length, padding length and trace
// rows (indexed by the batch's own iteration and its candidate numbering: query in the first iteration, query * K + k after).
__global__ void __launch_bounds__(256) beam_choose_groups_kernel(BeamState st, BcTable cb, int rs, int par) {
    pdl_wait();   // launched with the programmatic attribute: scheduled while the predecessor drains, starts when it is complete
    const int c = blockIdx.x, K = st.K;
    __shared__ int s_nacc[64];
    extern __shared__ unsigned char s_hit[];
    if (st.c_fin[c] == 2) return;
    const int q = c / K;
    const BcGroup& gr = cb.groups[cb.slots.slot_group[q]];
    const int cl = gr.iter == 0 ? cb.slots.slot_q[q] : cb.slots.slot_q[q] * K + c % K;
    const long long tr = (long long)gr.iter * gr.B * K + cl;
    choose_candidate(st, c, q, gr.dl, rs, st.smart ? gr.lmax : st.N, par, s_hit, s_nacc, gr.trace_nacc ? gr.trace_nacc + tr * st.N : nullptr,
                     gr.trace_pick ? gr.trace_pick + tr : nullptr);
}
void launch_beam_choose_groups(const BeamState& st, const BcTable& cb, int dl, cudaStream_t s) {
    const size_t smem = (size_t)st.N * (dl > 0 ? dl : 1);
    const int par = smem <= 40 * 1024 ? 1 : 0;
    launch_pdl(beam_choose_groups_kernel, dim3(st.B * st.K), dim3(256), par ? smem : 0, s, st, cb, dl + 1, par);
}

// Expand step of the continuous loop: beam_expand per occupied slot with its batch's width and draft length, the new
// hypotheses also written to the batch's output at its width.  The CTA that arrives last closes the iteration for every
// open batch with the reference's stop rule (its own counters, error, width and draft length), frees the slots of the
// batches that closed and posts the loop's word: sequence (24 bits) | slots in use (12) | largest draft length of the open
// batches (8) | unfinished candidates of the next iteration (16).
__global__ void __launch_bounds__(256) beam_expand_groups_kernel(BeamState st, BcTable cb, int rs) {
    pdl_wait();   // launched with the programmatic attribute: scheduled while the predecessor drains, starts when it is complete
    const int q = blockIdx.x, K = st.K;
    const int g = cb.slots.slot_group[q];
    if (g >= 0) {
        BcGroup* gr = &cb.groups[g];
        const int W = gr->W;
        int* ctrl = st.ctrl;
        expand_query(st, q, K, gr->dl, rs, W, &gr->error, gr->out + (long long)cb.slots.slot_q[q] * K * W,
                     [gr, ctrl](int, bool fin, int p, int pads, int has_eos) {
                         if (!has_eos) { atomicAnd(&gr->all_fin, 0); atomicAdd(&ctrl[BCX_NLIVE_NEXT], 1); }
                         atomicMin(&gr->min_pad, pads);
                         if (!fin) { atomicAdd(&gr->acc, p); atomicAdd(&gr->cnt, 1); }
                     });
    } else {
        for (int k = threadIdx.x; k < K; k += blockDim.x) st.n_parent[q * K + k] = -1;   // no cache to carry
    }
    __shared__ int s_last, s_dlmax, s_dlmin;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(&st.ctrl[BCX_TICKET], 1) == (int)gridDim.x - 1;
        s_dlmax = 0;
        s_dlmin = 0x7fffffff;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int gi = threadIdx.x; gi < cb.n_groups; gi += blockDim.x) {
        BcGroup* gr = &cb.groups[gi];
        if (gr->closed) continue;
        const int all_fin = atomicAdd(&gr->all_fin, 0), empty = atomicAdd(&gr->min_pad, 0);
        const int acc = atomicAdd(&gr->acc, 0), cnt = atomicAdd(&gr->cnt, 0), err = atomicAdd(&gr->error, 0);
        gr->accepted += acc;
        gr->produced += acc + cnt;
        gr->iter += 1;
        // speculative_decoding.py:452-470 and :570-598, as the CTA that closes an iteration of one batch applies them
        const int W = gr->W, dl = gr->dl, filled = W - empty, budget = st.max_len - filled - 1;
        atomicMin(&s_dlmin, dl);
        if (err != 0 || all_fin != 0 || budget < 1 || filled > st.max_len) {
            gr->closed = 1;   // W stays the width of the batch's last iteration: the width of its output
            atomicSub(&st.ctrl[BCC_USED], gr->B);
        } else {
            gr->W = W + max(min(budget, dl) + 1 - empty, 0);
            gr->dl = min(budget, dl);
            atomicMax(&s_dlmax, gr->dl);
        }
        gr->all_fin = 1; gr->min_pad = 0x7fffffff; gr->acc = 0; gr->cnt = 0; gr->lmax = 0;
    }
    __syncthreads();
    for (int b = threadIdx.x; b < st.B; b += blockDim.x) {
        const int gb = cb.slots.slot_group[b];
        if (gb >= 0 && cb.groups[gb].closed) cb.slots.slot_group[b] = -1;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int nlive_next = st.ctrl[BCX_NLIVE_NEXT];
        st.ctrl[BCX_NLIVE_NEXT] = 0;
        st.ctrl[BCX_TICKET] = 0;
        const int seq = st.ctrl[BCX_ITER] + 1;
        st.ctrl[BCX_ITER] = seq;
        st.ctrl[BCC_DLMAX] = s_dlmax;
        if (cb.dl_min) cb.dl_min[seq - 1] = s_dlmin;
        if (st.host_ctrl) {
            const unsigned long long word = ((unsigned long long)(seq & 0xffffff) << 40) | ((unsigned long long)(st.ctrl[BCC_USED] & 0xfff) << 28) |
                                            ((unsigned long long)(s_dlmax & 0xff) << 20) | ((unsigned long long)(nlive_next & 0xffff) << 4);
            reinterpret_cast<volatile unsigned long long*>(st.host_ctrl)[seq & 3] = word;
        }
    }
}
void launch_beam_expand_groups(const BeamState& st, const BcTable& cb, int dl, cudaStream_t s) {
    const size_t smem = ((size_t)st.K * (dl + 1) * st.K + (size_t)st.K * (dl + 2)) * sizeof(float);
    if (ensure_dyn_smem(beam_expand_groups_kernel, (int)smem)) return;   // error recorded; the launch below fails and cudaGetLastError reports it
    launch_pdl(beam_expand_groups_kernel, dim3(st.B), dim3(256), smem, s, st, cb, dl + 1);
}

__global__ void beam_init_kernel(BeamState st) {
    const long long n = (long long)st.B * st.K * st.ldw;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        st.cand_cur[i] = (i % st.ldw == 0 && i / st.ldw < st.B) ? st.bos : st.pad;
        st.cand_next[i] = st.pad;
    }
    if (blockIdx.x == 0) {
        for (int b = threadIdx.x; b < st.B * st.K; b += blockDim.x) { st.logp_cur[b] = 0.f; st.logp_next[b] = 0.f; }
        if (threadIdx.x < BC_COUNT) st.ctrl[threadIdx.x] = 0;
        if (threadIdx.x == 0) {
            st.ctrl[BCX_ALL_FIN] = 1; st.ctrl[BCX_MIN_PAD] = 0x7fffffff; st.ctrl[BCX_ACC] = 0; st.ctrl[BCX_CNT] = 0; st.ctrl[BCX_TICKET] = 0;
            st.ctrl[BCX_W] = st.w0; st.ctrl[BCX_ITER] = 0; st.ctrl[BCX_DONE] = 0; st.ctrl[BCX_NLIVE_NEXT] = 0;
        }
    }
}
void launch_beam_init(const BeamState& st, cudaStream_t s) { beam_init_kernel<<<64, 256, 0, s>>>(st); }

// (rows, W) int32 with row stride ldw -> dense int64
__global__ void beam_export_kernel(const int* __restrict__ cand, int ldw, int R, int W, long long* __restrict__ out) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx < (long long)R * W) out[idx] = cand[(idx / W) * ldw + idx % W];
}
void launch_beam_export(const int* cand, int ldw, int R, int W, long long* out, cudaStream_t s) {
    const long long n = (long long)R * W;
    if (n > 0) beam_export_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(cand, ldw, R, W, out);
}

}  // namespace ttb
