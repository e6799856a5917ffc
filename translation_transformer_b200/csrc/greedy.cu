// Device-resident state machine of speculative greedy decoding
// (reference: /root/reference/src/decoding/speculative_decoding.py:39-174).
//
// The host never looks at tokens while decoding.  Per iteration the engine launches
//   greedy_embed -> decoder layers -> classifier + argmax -> greedy_accept -> cache_append
// and the accept kernel (a single CTA: the bookkeeping of a whole batch is a few KB) does what the
// reference does with ~40 tensor ops and two host syncs per iteration:
//   * accepted length of every draft  (verification / cumsum / sum, :129-131)
//   * best draft per query            (topk(1), :133; tie-break = torch CPU topk emulation)
//   * token append + front index      (:136-146)
//   * retirement of finished queries into the output buffer and order-preserving compaction of
//     the live list (:149-168)
//   * the width bookkeeping of the reference's shared token matrix (:93-102), which decides when
//     the loop stops and when the reference itself would fail (see oracle/greedy_speculative.py).
#include "kernels.cuh"
#include "topk_emul.cuh"

namespace ttb {

// ---- width plan of the coming iteration (speculative_decoding.py:93-102) -----------------------
// Executed by one CTA after the live list is final.  `W` is the current width of the reference's
// token matrix.  `active` / `front` / `gen` may point to shared-memory copies of the state (accept
// kernel) or to the global arrays (init kernel); `col_live` is [W] ints of shared scratch.
__device__ void plan_next_iteration(const GreedyState& st, const int* active, const int* front, const int* gen,
                                    int n_active, int W, int* /*s_tmp*/, int* /*col_live*/) {
    __syncthreads();
    if (n_active == 0 || W >= st.max_len) {
        if (threadIdx.x == 0) { st.ctrl[CTRL_DONE] = 1; st.ctrl[CTRL_N_LEFT] = n_active; st.ctrl[CTRL_N_ACTIVE] = 0; }
        return;
    }
    // a column is dead when every live row holds PAD there: one column per thread (and pass), rows in the inner loop, the
    // dead columns are counted by the barrier itself
    int dead_total = 0;
    for (int c0 = 0; c0 < W; c0 += blockDim.x) {
        const int c = c0 + threadIdx.x;
        int live = 0;
        if (c < W)
            for (int g = 0; g < n_active; ++g) {
                const int b = active[g];
                live |= (c <= front[b] && gen[(long long)b * st.gen_ld + c] != st.pad) ? 1 : 0;
            }
        dead_total += __syncthreads_count(c < W && !live);
    }
    const int Wn = W + st.D + 1 - dead_total;   // the barrier counts are the same in every thread
    int oob = 0;
    for (int g = threadIdx.x; g < n_active; g += blockDim.x)
        if (front[active[g]] + 1 + st.D > Wn - 1) oob = 1;
    const int any_oob = __syncthreads_or(oob);
    if (threadIdx.x == 0) {
        st.ctrl[CTRL_PREV_WIDTH] = W;
        st.ctrl[CTRL_WIDTH] = Wn;
        if (any_oob) { st.ctrl[CTRL_ERROR] = 1; st.ctrl[CTRL_DONE] = 1; st.ctrl[CTRL_N_LEFT] = n_active; st.ctrl[CTRL_N_ACTIVE] = 0; }
    }
}

__global__ void __launch_bounds__(256) greedy_init_kernel(GreedyState st) {
    __shared__ int s_tmp[2];
    extern __shared__ int s_init_dyn[];   // [gen_ld] column flags
    for (long long idx = threadIdx.x; idx < (long long)st.B * st.gen_ld; idx += blockDim.x)
        st.gen[idx] = (idx % st.gen_ld == 0) ? st.bos : st.pad;
    for (long long idx = threadIdx.x; idx < (long long)st.B * st.max_len; idx += blockDim.x) st.out[idx] = st.pad;
    for (int b = threadIdx.x; b < st.B; b += blockDim.x) {
        st.front[b] = 0;
        st.active[b] = b;
        st.desc[b] = make_int4(b, 0, st.bos, st.src_len ? st.src_len[b] : 0x7fffffff);
    }
    if (threadIdx.x < CTRL_COUNT) st.ctrl[threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        st.ctrl[CTRL_N_ACTIVE] = st.B;
        st.ctrl[CTRL_LS] = st.Ls;
        // the most frequent tie (no draft accepted at all: every length is 0) has a fixed answer per n_drafts
        int pick = 0;
        if (st.tie_break == 0 && st.N > 1 && st.N < 64) {
            for (int n = 0; n < st.N; ++n) s_init_dyn[n] = n;   // value 0, index n
            pick = topk1_torch_cpu_packed(s_init_dyn, st.N);
        }
        st.ctrl[CTRL_ALLEQ_PICK] = pick;
    }
    plan_next_iteration(st, st.active, st.front, st.gen, st.B, 1, s_tmp, s_init_dyn);
}
void launch_greedy_init(const GreedyState& st, cudaStream_t s) {
    greedy_init_kernel<<<1, 256, (size_t)(st.gen_ld > 64 ? st.gen_ld : 64) * sizeof(int), s>>>(st);
}

// ---- first kernel of an iteration: KV-cache append of the previous iteration + step-token embedding ----------
template <typename ActT>
__global__ void greedy_advance_kernel(GreedyState st, const float* __restrict__ table, const float* __restrict__ pe,
                                      int E, float* __restrict__ x, ActT* __restrict__ xh, int n_embed_blocks,
                                      const ActT* __restrict__ qkv_all, long long qkv_layer_stride, int n_layers, int qkv_ld,
                                      ActT* __restrict__ kcache, ActT* __restrict__ vcache, long long cache_layer_stride,
                                      long long cache_query_stride, int cache_ld) {
    // Launched with the programmatic attribute behind the accept kernel (scheduled while it runs, starts when it is
    // complete).  The kernels of the decoding iteration read the control words and descriptor table of the accept kernel
    // ahead of their dependency waits, so none of them may be scheduled before this kernel has SEEN the accept kernel
    // complete: its dependents are released right behind its own wait, not before (their prologues -- barrier set-up,
    // tensor-memory allocation, weight requests -- then overlap this kernel instead of following it).  Nothing this kernel
    // writes (embeddings, the appended K/V rows) is read by a later kernel ahead of that kernel's wait.
    pdl_wait();
#ifndef TTB_ADVANCE_NO_TRIGGER
    pdl_launch_dependents();
#endif
    // the control words and the per-slot records are fetched together, ahead of the tests that use them (as dependent
    // loads they would be three to five global round trips in a row); the slot indices are in range for every CTA
    const int done = st.ctrl[CTRL_DONE], n_sel = st.ctrl[CTRL_N_SEL], n_active = st.ctrl[CTRL_N_ACTIVE];
    if ((int)blockIdx.x >= n_embed_blocks) {
        // K/V of the accepted positions of the chosen draft (recorded in st.sel by the accept kernel) -> cache
        const int idx = blockIdx.x - n_embed_blocks;
        const int g = idx / n_layers, l = idx % n_layers;
        const int4 sel = *reinterpret_cast<const int4*>(st.sel + g * 4);
        // after DONE neither the cache nor the embeddings are read again; a < 0 marks a query that left the live list
        // (continuous batching: its slot may already belong to a newly admitted query)
        if (done || g >= n_sel || sel.w < 0) return;
        const int b = sel.x, f = sel.y, pick = sel.z, a = sel.w;
        const ActT* src = qkv_all + (long long)l * qkv_layer_stride + ((long long)g * st.N + pick) * (st.D + 1) * qkv_ld;
        ActT* kd = kcache + (long long)l * cache_layer_stride + (long long)b * cache_query_stride + (long long)f * cache_ld;
        ActT* vd = vcache + (long long)l * cache_layer_stride + (long long)b * cache_query_stride + (long long)f * cache_ld;
        for (int i2 = threadIdx.x; i2 < (a + 1) * E; i2 += blockDim.x) {
            const int i = i2 / E, c = i2 % E;
            kd[(long long)i * cache_ld + c] = src[(long long)i * qkv_ld + E + c];
            vd[(long long)i * cache_ld + c] = src[(long long)i * qkv_ld + 2 * E + c];
        }
        return;
    }
    const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const int per_q = st.N * (st.D + 1);
    const int g = min(t / per_q, st.B - 1), r = t % per_q, n = r / (st.D + 1), i = r % (st.D + 1);
    const int4 d = st.desc[g];
    if (done || t >= n_active * per_q) return;
    const int b = d.x, f = d.y;
    const int tok = (i == 0) ? d.z : st.drafts[((long long)b * st.N + n) * st.D + i - 1];
    const float* e = table + (long long)tok * E;
    const float* p = pe + (long long)(f + i + 1) * E;
    for (int c = lane; c < E; c += 32) {
        float v = e[c] + p[c];
        x[(long long)t * E + c] = v;
        if (xh) xh[(long long)t * E + c] = from_f32<ActT>(v);
    }
}
template <typename ActT>
void launch_greedy_advance(const GreedyState& st, const float* table, const float* pe, int E, float* x, ActT* xh,
                           const ActT* qkv_all, long long qkv_layer_stride, int n_layers, int qkv_ld, ActT* kcache, ActT* vcache,
                           long long cache_layer_stride, long long cache_query_stride, int cache_ld, cudaStream_t s) {
    const int T = st.B * st.N * (st.D + 1);
    const int n_embed_blocks = (T + 7) / 8;
    // first kernel of the captured iteration: plain launch (its predecessor is the previous graph launch)
    launch_pdl(greedy_advance_kernel<ActT>, dim3(n_embed_blocks + st.B * n_layers), dim3(256), 0, s, st, table, pe, E, x, xh, n_embed_blocks, qkv_all,
                                                                              qkv_layer_stride, n_layers, qkv_ld, kcache, vcache,
                                                                              cache_layer_stride, cache_query_stride, cache_ld);
}
template void launch_greedy_advance<float>(const GreedyState&, const float*, const float*, int, float*, float*, const float*, long long, int, int,
                                           float*, float*, long long, long long, int, cudaStream_t);
template void launch_greedy_advance<__nv_bfloat16>(const GreedyState&, const float*, const float*, int, float*, __nv_bfloat16*,
                                                   const __nv_bfloat16*, long long, int, int, __nv_bfloat16*, __nv_bfloat16*, long long,
                                                   long long, int, cudaStream_t);

// ---- accept / retire / plan ---------------------------------------------------------------------
// One CTA, one warp per live query: lanes score the drafts in parallel (accepted length = leading
// matches between draft tokens and the predictions one position earlier), lane 0 applies the
// tie-break rule, the warp appends the tokens and retires the query if it produced EOS.
// The whole bookkeeping state (live list, fronts, token matrix) is copied to shared memory with one
// round of independent loads at kernel entry, so the dependent chains (live list -> front -> tokens,
// compaction, dead-column scan) never wait on global memory; updates are written through.
constexpr int ACCEPT_MAX_SMEM_INTS = 50 * 1024;   // token matrices larger than 200 KB stay in global memory

// ---- per-query step of the accept kernels: scoring of the drafts, tie-break, token append, retirement row --------------
// Executed by one warp for the query in live slot g (query / slot id b, front f).  `Wn` is the width of the token matrix
// of the iteration (of the query's own batch), `row` / `grow` its token row in shared / global memory (the same row when
// the matrix is not staged).  A finished query's row is written to `out_row` when it fits (the caller flags the shape
// error otherwise).  Returns the accepted length, the chosen draft and whether the query produced EOS.
struct AcceptStep { int a, pick; bool fin; };
__device__ __forceinline__ AcceptStep accept_query(const GreedyState& st, int g, int b, int f, int Wn, int* row, int* grow, bool stage_gen,
                                                   bool keep_pred, int alleq_pick, int* s_nacc, int* s_tokw, long long* out_row) {
    const int D = st.D, N = st.N, lane = threadIdx.x & 31;
    int best_val = -1, best_first = 0x7fffffff;
    int kept[16];
    for (int n = lane; n < N; n += 32) {
        const int* pr = st.pred + ((long long)g * N + n) * (D + 1);
        const int* dr = st.drafts + ((long long)b * N + n) * D;
        int a = 0;
        bool open = true;
        for (int a0 = 0; a0 < D && open; a0 += 16) {         // 32 independent loads per round
            int dv[16], pv[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                dv[u] = (a0 + u < D) ? dr[a0 + u] : -1;
                pv[u] = (a0 + u <= D) ? pr[a0 + u] : -2;   // pr[D]: the token behind a fully accepted draft (dv = -1 there)
            }
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                if (open && dv[u] == pv[u]) ++a; else open = false;
                kept[u] = pv[u];
            }
        }
        if (n < 64) s_nacc[n] = (a << 8) | n;   // packed for the tie-break emulation
        if (a > best_val) { best_val = a; best_first = n; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {   // max accepted length, lowest draft index among equals
        const int ov = __shfl_xor_sync(0xffffffffu, best_val, o), oi = __shfl_xor_sync(0xffffffffu, best_first, o);
        if (ov > best_val || (ov == best_val && oi < best_first)) { best_val = ov; best_first = oi; }
    }
    __syncwarp();
    int pick = best_first;
    if (st.tie_break == 0 && N < 64 && N > 1) {
        // a unique maximum is the answer of any selection algorithm; only ties need the emulation
        int ties = 0;
        for (int n = lane; n < N; n += 32) ties += ((s_nacc[n] >> 8) == best_val) ? 1 : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ties += __shfl_xor_sync(0xffffffffu, ties, o);
        if (ties == N) {
            pick = alleq_pick;            // all lengths equal: answer precomputed by the init kernel
        } else if (ties > 1) {
            if (lane == 0) pick = topk1_torch_cpu_packed(s_nacc, N);
            pick = __shfl_sync(0xffffffffu, pick, 0);
        }
    }
    const int a = best_val;
    const int* pr = st.pred + ((long long)g * N + pick) * (D + 1);
    bool fin_l = false;
    if (keep_pred) {
        if (lane == pick) {
#pragma unroll
            for (int u = 0; u < 16; ++u) s_tokw[u] = kept[u];
        }
        __syncwarp();
    }
    for (int j = lane; j <= D; j += 32) {
        const int t = (j <= a) ? (keep_pred ? s_tokw[j] : pr[j]) : st.pad;
        row[f + 1 + j] = t;
        if (stage_gen) grow[f + 1 + j] = t;
        fin_l |= (j <= a) && (t == st.eos);
    }
    const bool fin = __any_sync(0xffffffffu, fin_l);
    __syncwarp();
    if (fin && Wn <= st.max_len)
        for (int c = lane; c < Wn; c += 32) out_row[c] = (c <= f + a + 1) ? row[c] : st.pad;
    return {a, pick, fin};
}

// Copy of the token matrix [B][gen_ld] to shared memory: all loads of a thread in flight before the first store (a plain
// copy loop waits for every load: seven global round trips for the 27 KB of B = 32, max_len = 200)
__device__ __forceinline__ void stage_token_matrix(const GreedyState& st, int* s_gen) {
    const int total = st.B * st.gen_ld;
    for (int i0 = 0; i0 < total; i0 += 8 * blockDim.x) {
        int tmp[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int idx = i0 + u * blockDim.x + threadIdx.x; tmp[u] = idx < total ? st.gen[idx] : 0; }
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int idx = i0 + u * blockDim.x + threadIdx.x; if (idx < total) s_gen[idx] = tmp[u]; }
    }
}

#ifdef TTB_ACC_TIMELINE
__device__ long long g_acc_ts[16];
#define ACC_TS(i) do { if (threadIdx.x == 0) g_acc_ts[i] = clock64(); } while (0)
#else
#define ACC_TS(i) do { } while (0)
#endif
__global__ void __launch_bounds__(1024) greedy_accept_kernel(GreedyState st, int stage_gen) {
    __shared__ int s_tmp[2];
    __shared__ int s_acc, s_tok, s_err;
    extern __shared__ int s_dyn[];
    const int B = st.B, D = st.D, N = st.N;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
    int* s_active = s_dyn;                       // [B]
    int* s_front = s_active + B;                 // [B]
    int* s_fin = s_front + B;                    // [B]
    int* s_newact = s_fin + B;                   // [B]
    int* s_srclen = s_newact + B;                // [B]
    int* s_nacc_all = s_srclen + B;              // [warps][64]
    int* s_tok_all = s_nacc_all + n_warps * 64;  // [warps][16] predictions of the chosen draft row
    int* col_live = s_tok_all + n_warps * 16;    // [gen_ld]
    int* s_gen = col_live + st.gen_ld;           // [B][gen_ld] when stage_gen
    int* s_nacc = s_nacc_all + warp * 64;
    int* s_tokw = s_tok_all + warp * 16;
    // every lane scores one draft and D + 1 <= 16: the predictions of the chosen row are still in its lane's registers,
    // the token append takes them from there (through shared memory) instead of a second global round trip
    const bool keep_pred = N <= 32 && D + 1 <= 16;
    ACC_TS(0);
    pdl_launch_dependents();
#ifdef TTB_ACC_LATE_LOADS
    pdl_wait();   // A/B build: everything behind the dependency wait
#endif
    // ---- round 1: independent loads, AHEAD of the dependency wait.  Everything read here (control words, live list, fronts,
    // token matrix) was written by the accept kernel of the previous iteration (or by the init kernel), and the first kernel
    // of every iteration (greedy_advance_kernel) releases its dependents only behind its own wait: no kernel of this iteration
    // is scheduled before it has seen that accept kernel complete.  Only the predictions of the classifier (st.pred) need the wait.
    const int done = st.ctrl[CTRL_DONE];
    const int n_active = st.ctrl[CTRL_N_ACTIVE];
    const int Wn = st.ctrl[CTRL_WIDTH];
    const int iter = st.ctrl[CTRL_ITERS];
    const int alleq_pick = st.ctrl[CTRL_ALLEQ_PICK];
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        s_active[b] = st.active[b];
        s_front[b] = st.front[b];
        s_srclen[b] = st.src_len ? st.src_len[b] : 0x7fffffff;
    }
    if (stage_gen) stage_token_matrix(st, s_gen);
    ACC_TS(1);
#ifndef TTB_ACC_LATE_LOADS
    pdl_wait();
#endif
    if (done) return;
    int* G = stage_gen ? s_gen : st.gen;
    if (threadIdx.x == 0) { s_acc = 0; s_tok = 0; s_err = 0; if (st.hist) st.hist[iter] = n_active; }
    __syncthreads();
    ACC_TS(2);
    for (int g = warp; g < n_active; g += n_warps) {
        const int b = s_active[g];
        const int f = s_front[b];
        const AcceptStep r = accept_query(st, g, b, f, Wn, G + (long long)b * st.gen_ld, st.gen + (long long)b * st.gen_ld, stage_gen, keep_pred,
                                          alleq_pick, s_nacc, s_tokw, st.out + (long long)b * st.max_len);
        const int a = r.a, pick = r.pick;
        const bool fin = r.fin;
        if (lane == 0) {
            s_front[b] = f + a + 1;
            st.front[b] = f + a + 1;
            st.sel[g * 4 + 0] = b; st.sel[g * 4 + 1] = f; st.sel[g * 4 + 2] = pick; st.sel[g * 4 + 3] = a;
            if (st.trace) {
                int* tr = st.trace + ((long long)iter * st.B + g) * 4;
                tr[0] = b; tr[1] = a; tr[2] = pick; tr[3] = Wn;
            }
            atomicAdd(&s_acc, a);
            atomicAdd(&s_tok, a + 1);
            s_fin[g] = fin ? 1 : 0;
            if (fin && Wn > st.max_len) s_err = 2;  // the reference cannot store a finished row wider than max_len (:158)
        }
    }
    ACC_TS(3);
    __syncthreads();
    ACC_TS(4);
    // order-preserving compaction of the live list (boolean masking in the reference): warp 0, ballot prefix sums
    if (warp == 0) {
        int w = 0;
        for (int g0 = 0; g0 < n_active; g0 += 32) {
            const int g = g0 + lane;
            const bool alive = g < n_active && !s_fin[g];
            const unsigned m = __ballot_sync(0xffffffffu, alive);
            if (alive) {
                const int pos = w + __popc(m & ((1u << lane) - 1u));
                const int b = s_active[g];
                s_newact[pos] = b;
                st.active[pos] = b;
                const int fb = s_front[b];
                st.desc[pos] = make_int4(b, fb, G[(long long)b * st.gen_ld + fb], s_srclen[b]);
            }
            w += __popc(m);
        }
        if (lane == 0) {
            st.ctrl[CTRL_N_SEL] = n_active;
            st.ctrl[CTRL_N_ACTIVE] = w;
            st.ctrl[CTRL_ITERS] = iter + 1;
            st.ctrl[CTRL_ACCEPTED] += s_acc;
            st.ctrl[CTRL_TOKENS] += s_tok;
            if (s_err) { st.ctrl[CTRL_ERROR] = s_err; st.ctrl[CTRL_DONE] = 1; st.ctrl[CTRL_N_LEFT] = w; st.ctrl[CTRL_N_ACTIVE] = 0; }
            s_tmp[0] = w;
        }
    }
    __syncthreads();
    ACC_TS(5);
    if (s_err) return;
    const int n_left = s_tmp[0];
    plan_next_iteration(st, s_newact, s_front, G, n_left, Wn, s_tmp, col_live);
    ACC_TS(6);
}
void launch_greedy_accept(const GreedyState& st, cudaStream_t s) {
    const int warps = st.B < 32 ? (st.B < 4 ? 4 : st.B) : 32;
    const size_t base_ints = (size_t)5 * st.B + (size_t)warps * 80 + st.gen_ld;
    const size_t gen_ints = (size_t)st.B * st.gen_ld;
    const int stage_gen = base_ints + gen_ints <= (size_t)ACCEPT_MAX_SMEM_INTS ? 1 : 0;
    const size_t smem = (base_ints + (stage_gen ? gen_ints : 0)) * sizeof(int);
    if (smem > 48 * 1024 && ensure_dyn_smem(greedy_accept_kernel, (int)(ACCEPT_MAX_SMEM_INTS * sizeof(int)))) return;   // the launch below then fails loudly
#ifdef TTB_ACC_TIMELINE
    {
        static int n_launch = 0;
        if (++n_launch == 100) {
            cudaStreamSynchronize(s);
            long long h[16];
            cudaMemcpyFromSymbol(h, g_acc_ts, sizeof(h));
            FILE* f = fopen("gpurun_out/acc_timeline.txt", "w");
            if (f) { for (int i = 0; i < 7; ++i) fprintf(f, "%d %lld\n", i, h[i] - h[1]); fclose(f); }
        }
    }
#endif
    launch_pdl(greedy_accept_kernel, dim3(1), dim3(warps * 32), smem, s, st, stage_gen);
}

// ---- continuous batching: several batches share the live slots of one loop -------------------------------------
// Every slot belongs to the batch it was admitted with (cb.slots.slot_group) and holds that batch's query cb.slots.slot_q.  A batch
// keeps its own token-matrix width, iteration count, counters and error (CbGroup): the only quantities of the
// reference that couple the queries of a batch.  The live list keeps the members of a batch contiguous and in batch
// order (admission appends, compaction preserves the order), so a batch's live queries are one run of the list.

// Width plan of one batch, executed by one warp: `list` holds its n live slots after retirement, W the width of the
// iteration just done.  Same rule as plan_next_iteration: dead columns (PAD in every live row) shrink the growth.
__device__ void plan_width_warp(const GreedyState& st, const int* list, const int* front, const int* gen, int n, int W, int& Wn, bool& oob) {
    const int lane = threadIdx.x & 31;
    int dead = 0;
    for (int c0 = 0; c0 < W; c0 += 32) {
        const int c = c0 + lane;
        int live = 0;
        if (c < W)
            for (int r = 0; r < n; ++r) {
                const int b = list[r];
                live |= (c <= front[b] && gen[(long long)b * st.gen_ld + c] != st.pad) ? 1 : 0;
            }
        dead += __popc(__ballot_sync(0xffffffffu, c < W && !live));
    }
    Wn = W + st.D + 1 - dead;
    int o = 0;
    for (int r = lane; r < n; r += 32)
        if (front[list[r]] + 1 + st.D > Wn - 1) o = 1;
    oob = __any_sync(0xffffffffu, o) != 0;
}

// Admission of batch `grp` (Bi queries): takes the first Bi free slots, installs source lengths, drafts, token rows and
// descriptors, PAD-fills the batch's output, plans its first width and appends its slots to the live list.  One CTA,
// launched between two iterations.  Raises CTRL_ERROR = 3 when fewer than Bi slots are free (host bookkeeping broken).
__global__ void __launch_bounds__(1024) greedy_admit_kernel(GreedyState st, CbTable cb, int grp, int Bi, const int* __restrict__ drafts_in,
                                                            const int* __restrict__ srclen_in, long long* out, int* trace, int Ls_cap) {
    extern __shared__ int s_adm[];
    int* s_occ = s_adm;             // [S] -1 = free: the slots outside the live list (slot_group keeps stale entries)
    int* s_slots = s_adm + st.B;    // [Bi] slots taken, in batch order
    __shared__ int s_nfree;
    __shared__ int s_pick[64];      // scratch of the tie-break emulation
    const int S = st.B, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_active = st.ctrl[CTRL_N_ACTIVE];
    for (int i = threadIdx.x; i < S; i += blockDim.x) s_occ[i] = -1;
    __syncthreads();
    for (int g = threadIdx.x; g < n_active; g += blockDim.x) s_occ[st.active[g]] = 0;
    __syncthreads();
    if (warp == 0) {
        const int taken = take_free_slots(s_occ, S, Bi, s_slots);
        if (lane == 0) s_nfree = taken;
    }
    __syncthreads();
    if (s_nfree < Bi) {
        if (threadIdx.x == 0) st.ctrl[CTRL_ERROR] = 3;
        return;
    }
    const int D = st.D, N = st.N;
    for (int j = threadIdx.x; j < Bi; j += blockDim.x) {
        const int b = s_slots[j];
        cb.slots.adm_slots[j] = b;
        cb.slots.slot_group[b] = grp;
        cb.slots.slot_q[b] = j;
        st.front[b] = 0;
        const_cast<int*>(st.src_len)[b] = srclen_in[j];
    }
    for (long long idx = threadIdx.x; idx < (long long)Bi * st.gen_ld; idx += blockDim.x) {
        const int j = (int)(idx / st.gen_ld), c = (int)(idx % st.gen_ld);
        st.gen[(long long)s_slots[j] * st.gen_ld + c] = c == 0 ? st.bos : st.pad;
    }
    int* drafts = const_cast<int*>(st.drafts);
    for (long long idx = threadIdx.x; idx < (long long)Bi * N * D; idx += blockDim.x) {
        const int j = (int)(idx / (N * D)), r = (int)(idx % (N * D));
        drafts[(long long)s_slots[j] * N * D + r] = drafts_in[idx];
    }
    for (long long idx = threadIdx.x; idx < (long long)Bi * st.max_len; idx += blockDim.x) out[idx] = st.pad;
    __syncthreads();
    __shared__ int s_open;
    if (warp == 0) {
        int Wn = 1;
        bool oob = false;
        const bool short_loop = st.max_len <= 1;   // the reference's loop does not run at all
        // the standard loop (D = 0) has no token-matrix width to plan: with BOS = PAD the plan would close the batch
        if (!short_loop && D > 0) plan_width_warp(st, s_slots, st.front, st.gen, Bi, 1, Wn, oob);
        if (lane == 0) {
            const bool open = !short_loop && !oob;
            CbGroup gr{};
            gr.out = out; gr.trace = trace; gr.B = Bi; gr.W = open ? Wn : 1; gr.live = open ? Bi : 0;
            gr.error = oob ? 1 : 0; gr.n_left = open ? 0 : Bi; gr.closed = open ? 0 : 1;
            cb.groups[grp] = gr;
            s_open = open ? 1 : 0;
            // the most frequent tie (no draft accepted at all) has a fixed answer per n_drafts (as in greedy_init_kernel)
            int pick = 0;
            if (st.tie_break == 0 && N > 1 && N < 64) {
                for (int n = 0; n < N; ++n) s_pick[n] = n;
                pick = topk1_torch_cpu_packed(s_pick, N);
            }
            st.ctrl[CTRL_ALLEQ_PICK] = pick;
            st.ctrl[CTRL_LS] = Ls_cap;
        }
    }
    __syncthreads();
    if (!s_open) return;
    for (int j = threadIdx.x; j < Bi; j += blockDim.x) {
        const int b = s_slots[j];
        st.active[n_active + j] = b;
        st.desc[n_active + j] = make_int4(b, 0, st.bos, srclen_in[j]);
    }
    if (threadIdx.x == 0) { st.ctrl[CTRL_N_ACTIVE] = n_active + Bi; st.ctrl[CTRL_DONE] = 0; }
}
int launch_greedy_admit(const GreedyState& st, const CbTable& cb, int grp, int Bi, const int* drafts_in, const int* srclen_in, long long* out,
                        int* trace, int Ls_cap, cudaStream_t s) {
    const size_t smem = (size_t)(st.B + Bi) * sizeof(int);
    if (ensure_dyn_smem(greedy_admit_kernel, (int)smem)) return 1;   // error recorded by ensure_dyn_smem
    greedy_admit_kernel<<<1, 1024, smem, s>>>(st, cb, grp, Bi, drafts_in, srclen_in, out, trace, Ls_cap);
    return 0;
}

// Cross-attention K/V rows and key tokens of an admitted batch -> its slots (adm_slots, written by the admission kernel of
// any of the three continuous loops just before): rows [0, Ls) of slot b at b * Ls_cap; key tokens PAD behind Ls.  16-byte
// copies, grid-stride.
template <typename ActT>
__global__ void admit_kv_kernel(const int* __restrict__ slots, int Bi, int Ls, int Ls_cap, int n_layers, int row_chunks,
                                       const uint4* __restrict__ stage_kv, long long stage_layer_chunks, uint4* __restrict__ kv,
                                       long long layer_chunks, const int* __restrict__ src32, int* __restrict__ keytok, int pad) {
    const long long per_layer = (long long)Bi * Ls * row_chunks;
    const long long total = per_layer * n_layers;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int l = (int)(idx / per_layer);
        const long long r = idx % per_layer;
        const int row = (int)(r / row_chunks), c = (int)(r % row_chunks);   // row = j * Ls + position
        const int j = row / Ls, pos = row % Ls;
        kv[l * layer_chunks + ((long long)slots[j] * Ls_cap + pos) * row_chunks + c] = stage_kv[l * stage_layer_chunks + r];
    }
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < (long long)Bi * Ls_cap; idx += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(idx / Ls_cap), pos = (int)(idx % Ls_cap);
        keytok[(long long)slots[j] * Ls_cap + pos] = pos < Ls ? src32[(long long)j * Ls + pos] : pad;
    }
}
template <typename ActT>
void launch_admit_kv(const int* adm_slots, int Bi, int Ls, int Ls_cap, int n_layers, int E, const ActT* stage_kv, long long stage_layer_stride,
                     ActT* kv, long long layer_stride, const int* src32, int* keytok, int pad, cudaStream_t s) {
    const int row_chunks = (int)(2 * E * sizeof(ActT) / 16);
    const long long total = (long long)n_layers * Bi * Ls * row_chunks;
    const int blocks = (int)std::min<long long>((total + 255) / 256 + 1, 8LL * kNumSMs);
    admit_kv_kernel<ActT><<<blocks, 256, 0, s>>>(adm_slots, Bi, Ls, Ls_cap, n_layers, row_chunks, reinterpret_cast<const uint4*>(stage_kv),
                                                 stage_layer_stride * (long long)sizeof(ActT) / 16, reinterpret_cast<uint4*>(kv),
                                                 layer_stride * (long long)sizeof(ActT) / 16, src32, keytok, pad);
}
template void launch_admit_kv<float>(const int*, int, int, int, int, int, const float*, long long, float*, long long, const int*, int*, int,
                                     cudaStream_t);
template void launch_admit_kv<__nv_bfloat16>(const int*, int, int, int, int, int, const __nv_bfloat16*, long long, __nv_bfloat16*, long long,
                                             const int*, int*, int, cudaStream_t);

// Accept kernel of the continuous loop: the per-query step of greedy_accept_kernel, then per batch (= run of the live
// list) retirement into that batch's output, trace rows at the batch's own iteration, its error checks and width plan.
// A batch whose width reached max_len, whose queries all finished or that hit a reference error is closed: its
// remaining queries leave the live list (all-PAD rows, `n_left`).  Entries of `sel` whose query left are marked a = -1
// so that the next iteration does not append their K/V rows into a slot that may have been handed out again.
__global__ void __launch_bounds__(1024) greedy_accept_groups_kernel(GreedyState st, CbTable cb, int stage_gen) {
    __shared__ int s_nseg, s_total;
    extern __shared__ int s_dyn[];
    const int S = st.B, D = st.D, N = st.N;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
    int* s_active = s_dyn;                // [S] live list of the iteration
    int* s_front = s_active + S;          // [S] per slot
    int* s_fin = s_front + S;             // [S] per position
    int* s_newact = s_fin + S;            // [S] live list after retirement (closed batches still in)
    int* s_grp = s_newact + S;            // [S] per position: batch
    int* s_pseg = s_grp + S;              // [S] per position: run of the live list (open batch) it belongs to
    int* s_rank = s_pseg + S;             // [S] per position: index among the live queries of its batch
    int* s_nseg_of = s_rank + S;          // [S] per position of s_newact: its run
    int* s_seg = s_nseg_of + S;           // [8][S] per run: batch, width, iteration, batch size, accepted, tokens, live, error/open
    int* s_seg_grp = s_seg, *s_seg_W = s_seg + S, *s_seg_it = s_seg + 2 * S, *s_seg_B = s_seg + 3 * S;
    int* s_seg_acc = s_seg + 4 * S, *s_seg_tok = s_seg + 5 * S, *s_seg_live = s_seg + 6 * S, *s_seg_st = s_seg + 7 * S;
    int* s_seg_new0 = s_seg + 8 * S;      // [S] first position of the run in s_newact
    int* s_nacc_all = s_seg + 9 * S;      // [warps][64]
    int* s_tok_all = s_nacc_all + n_warps * 64;   // [warps][16]
    int* s_gen = s_tok_all + n_warps * 16;        // [S][gen_ld] when stage_gen
    int* s_nacc = s_nacc_all + warp * 64;
    int* s_tokw = s_tok_all + warp * 16;
    const bool keep_pred = N <= 32 && D + 1 <= 16;
    pdl_launch_dependents();
    // loads ahead of the dependency wait: written by the previous accept or admission kernel (see greedy_accept_kernel)
    const int done = st.ctrl[CTRL_DONE];
    const int n_active = st.ctrl[CTRL_N_ACTIVE];
    const int iter = st.ctrl[CTRL_ITERS];
    const int alleq_pick = st.ctrl[CTRL_ALLEQ_PICK];
    for (int b = threadIdx.x; b < S; b += blockDim.x) {
        const int a = st.active[b];
        s_active[b] = a;
        s_front[b] = st.front[b];
        if (b < n_active) s_grp[b] = cb.slots.slot_group[a];
    }
    if (stage_gen) stage_token_matrix(st, s_gen);
    pdl_wait();
    if (done) return;
    int* G = stage_gen ? s_gen : st.gen;
    __syncthreads();
    // runs of the live list (one per open batch) and the rank of every position inside its run
    if (warp == 0) {
        int nseg = 0, cur = 0;
        for (int g0 = 0; g0 < n_active; g0 += 32) {
            const int g = g0 + lane;
            const int grp = g < n_active ? s_grp[g] : -1;
            const bool start = g < n_active && (g == 0 || s_grp[g - 1] != grp);
            const unsigned m = __ballot_sync(0xffffffffu, start);
            const unsigned below = m & ((2u << lane) - 1u);
            if (g < n_active) {
                s_pseg[g] = nseg + __popc(below) - 1;
                s_rank[g] = g - (below ? g0 + 31 - __clz(below) : cur);
            }
            if (start) s_seg_grp[nseg + __popc(below) - 1] = grp;
            if (m) cur = g0 + 31 - __clz(m);
            nseg += __popc(m);
        }
        if (lane == 0) s_nseg = nseg;
    }
    __syncthreads();
    const int nseg = s_nseg;
    for (int k = threadIdx.x; k < nseg; k += blockDim.x) {
        const CbGroup& gr = cb.groups[s_seg_grp[k]];
        s_seg_W[k] = gr.W; s_seg_it[k] = gr.iter; s_seg_B[k] = gr.B;
        s_seg_acc[k] = 0; s_seg_tok[k] = 0; s_seg_live[k] = 0; s_seg_st[k] = 0;
    }
    if (threadIdx.x == 0 && st.hist) st.hist[iter] = n_active;
    __syncthreads();
    for (int g = warp; g < n_active; g += n_warps) {
        const int b = s_active[g];
        const int f = s_front[b];
        const int k = s_pseg[g];
        const CbGroup& gr = cb.groups[s_seg_grp[k]];
        const int q = cb.slots.slot_q[b], Wn = s_seg_W[k];
        const AcceptStep r = accept_query(st, g, b, f, Wn, G + (long long)b * st.gen_ld, st.gen + (long long)b * st.gen_ld, stage_gen, keep_pred,
                                          alleq_pick, s_nacc, s_tokw, gr.out + (long long)q * st.max_len);
        if (lane == 0) {
            s_front[b] = f + r.a + 1;
            st.front[b] = f + r.a + 1;
            st.sel[g * 4 + 0] = b; st.sel[g * 4 + 1] = f; st.sel[g * 4 + 2] = r.pick; st.sel[g * 4 + 3] = r.a;
            if (gr.trace) {
                int* tr = gr.trace + ((long long)s_seg_it[k] * s_seg_B[k] + s_rank[g]) * 4;
                tr[0] = q; tr[1] = r.a; tr[2] = r.pick; tr[3] = Wn;
            }
            atomicAdd(&s_seg_acc[k], r.a);
            atomicAdd(&s_seg_tok[k], r.a + 1);
            s_fin[g] = r.fin ? 1 : 0;
            if (!r.fin) atomicAdd(&s_seg_live[k], 1);
            if (r.fin && Wn > st.max_len) s_seg_st[k] = 2;   // shape error of the reference (:158): ends this batch only
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int p = 0;
        for (int k = 0; k < nseg; ++k) { s_seg_new0[k] = p; if (!s_seg_st[k]) p += s_seg_live[k]; }
        s_total = p;
    }
    // order-preserving compaction without the finished queries and without the batches that failed
    if (warp == 0) {
        int w = 0;
        for (int g0 = 0; g0 < n_active; g0 += 32) {
            const int g = g0 + lane;
            const bool alive = g < n_active && !s_fin[g] && !s_seg_st[s_pseg[g]];
            const unsigned m = __ballot_sync(0xffffffffu, alive);
            if (alive) {
                const int pos = w + __popc(m & ((1u << lane) - 1u));
                s_newact[pos] = s_active[g];
                s_nseg_of[pos] = s_pseg[g];
            }
            w += __popc(m);
        }
    }
    __syncthreads();
    // per batch: width plan of the coming iteration or closing (one warp per run); s_seg_st becomes 0 open, 1 closed
    for (int k = warp; k < nseg; k += n_warps) {
        const int cnt = s_seg_live[k], W = s_seg_W[k];
        int err = s_seg_st[k], Wn = W;
        bool open = false;
        if (!err && cnt > 0 && W < st.max_len) {
            bool oob;
            plan_width_warp(st, s_newact + s_seg_new0[k], s_front, G, cnt, W, Wn, oob);
            if (oob) err = 1;
            open = !oob;
        }
        if (lane == 0) {
            CbGroup& gr = cb.groups[s_seg_grp[k]];
            gr.iter = s_seg_it[k] + 1;
            gr.accepted += s_seg_acc[k];
            gr.tokens += s_seg_tok[k];
            gr.W = Wn;
            gr.live = open ? cnt : 0;
            gr.error = err;
            gr.n_left = open ? 0 : cnt;
            gr.closed = open ? 0 : 1;
            s_seg_st[k] = open ? 0 : 1;
        }
    }
    __syncthreads();
    // live list of the coming iteration: the queries of the batches that stay open
    if (warp == 0) {
        const int n_new = s_total;
        int w = 0;
        for (int p0 = 0; p0 < n_new; p0 += 32) {
            const int p = p0 + lane;
            const bool keep = p < n_new && !s_seg_st[s_nseg_of[p]];
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int pos = w + __popc(m & ((1u << lane) - 1u));
                const int b = s_newact[p];
                const int fb = s_front[b];
                st.active[pos] = b;
                st.desc[pos] = make_int4(b, fb, G[(long long)b * st.gen_ld + fb], st.src_len[b]);
            }
            w += __popc(m);
        }
        if (lane == 0) {
            st.ctrl[CTRL_N_SEL] = n_active;
            st.ctrl[CTRL_N_ACTIVE] = w;
            st.ctrl[CTRL_ITERS] = iter + 1;
            st.ctrl[CTRL_DONE] = w == 0 ? 1 : 0;
        }
    }
    for (int g = threadIdx.x; g < n_active; g += blockDim.x)
        if (s_fin[g] || s_seg_st[s_pseg[g]]) st.sel[g * 4 + 3] = -1;
}
void launch_greedy_accept_groups(const GreedyState& st, const CbTable& cb, cudaStream_t s) {
    const int warps = st.B < 32 ? (st.B < 4 ? 4 : st.B) : 32;
    const size_t base_ints = (size_t)17 * st.B + (size_t)warps * 80;
    const size_t gen_ints = (size_t)st.B * st.gen_ld;
    const int stage_gen = base_ints + gen_ints <= (size_t)ACCEPT_MAX_SMEM_INTS ? 1 : 0;
    const size_t smem = (base_ints + (stage_gen ? gen_ints : 0)) * sizeof(int);
    if (smem > 48 * 1024 && ensure_dyn_smem(greedy_accept_groups_kernel, (int)(ACCEPT_MAX_SMEM_INTS * sizeof(int)))) return;   // launch fails loudly
    launch_pdl(greedy_accept_groups_kernel, dim3(1), dim3(warps * 32), smem, s, st, cb, stage_gen);
}

// ---- standard greedy decoding (standard_decoding.py:29-56): one token per row and iteration ------------------
// Runs in place of the accept kernel when the loop is used without drafts (N = 1, D = 0).  Every row stays live
// until the first step in which ALL rows predict EOS or PAD (rows that already emitted EOS keep decoding, like in
// the reference), or until the token matrix is full.
__global__ void __launch_bounds__(1024) greedy_std_step_kernel(GreedyState st) {
    pdl_launch_dependents();
    pdl_wait();
    if (st.ctrl[CTRL_DONE]) return;
    const int iter = st.ctrl[CTRL_ITERS];
    const int f = iter;                     // every row holds iter + 1 tokens
    int stop = 1;
    for (int b = threadIdx.x; b < st.B; b += blockDim.x) {
        const int tok = st.pred[b];
        st.gen[(long long)b * st.gen_ld + f + 1] = tok;
        st.front[b] = f + 1;
        st.desc[b] = make_int4(b, f + 1, tok, st.src_len ? st.src_len[b] : 0x7fffffff);
        st.sel[b * 4 + 0] = b; st.sel[b * 4 + 1] = f; st.sel[b * 4 + 2] = 0; st.sel[b * 4 + 3] = 0;
        if (tok != st.eos && tok != st.pad) stop = 0;
    }
    const int all_stop = __syncthreads_and(stop);
    const bool done = all_stop || f + 2 >= st.max_len;
    if (done) {   // export: tokens 0 .. f+1, PAD behind them (the reference's pre-filled token matrix)
        for (long long idx = threadIdx.x; idx < (long long)st.B * st.max_len; idx += blockDim.x) {
            const int b = (int)(idx / st.max_len), c = (int)(idx % st.max_len);
            st.out[idx] = c <= f + 1 ? st.gen[(long long)b * st.gen_ld + c] : st.pad;
        }
    }
    if (threadIdx.x == 0) {
        if (st.hist) st.hist[iter] = st.B;
        st.ctrl[CTRL_N_SEL] = st.B;
        st.ctrl[CTRL_ITERS] = iter + 1;
        st.ctrl[CTRL_TOKENS] += st.B;
        if (done) { st.ctrl[CTRL_DONE] = 1; st.ctrl[CTRL_N_LEFT] = 0; st.ctrl[CTRL_N_ACTIVE] = 0; }
    }
}
void launch_greedy_std_step(const GreedyState& st, cudaStream_t s) {
    launch_pdl(greedy_std_step_kernel, dim3(1), dim3(st.B < 1024 ? ((st.B + 31) / 32 * 32) : 1024), 0, s, st);
}

// Step kernel of the continuous loop without drafts, in place of greedy_std_step_kernel.  What the reference couples across
// a batch is kept per batch (CbGroup): its step count (every row of the batch holds 1 + iter tokens, so it is also the
// front of each of its slots), its stop rule and its output.  A batch's slots are one run of the live list (admission
// appends them in batch order, compaction preserves the order), and a batch leaves the list whole, when it stops.
__global__ void __launch_bounds__(1024) greedy_std_step_groups_kernel(GreedyState st, CbTable cb) {
    __shared__ int s_nseg, s_nstop;
    extern __shared__ int s_dyn[];
    const int S = st.B, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int* s_active = s_dyn;          // [S] live list of the step
    int* s_grp = s_active + S;      // [S] per position: batch
    int* s_pseg = s_grp + S;        // [S] per position: run of the live list it belongs to
    int* s_stop = s_pseg + S;       // [S] positions of the batches that stop in this step
    int* s_seg_grp = s_stop + S;    // [S] per run: batch
    int* s_seg_f = s_seg_grp + S;   // [S] per run: front before the step (the batch's step count)
    int* s_seg_go = s_seg_f + S;    // [S] per run: a row predicted neither EOS nor PAD; then: the batch stays open
    pdl_launch_dependents();
    // loads ahead of the dependency wait: written by the previous step or admission kernel (see greedy_accept_kernel)
    const int done = st.ctrl[CTRL_DONE];
    const int n_active = st.ctrl[CTRL_N_ACTIVE];
    const int iter = st.ctrl[CTRL_ITERS];
    for (int g = threadIdx.x; g < n_active; g += blockDim.x) {
        const int b = st.active[g];
        s_active[g] = b;
        s_grp[g] = cb.slots.slot_group[b];
    }
    pdl_wait();
    if (done) return;
    __syncthreads();
    // runs of the live list (one per open batch): the ballot scan of greedy_accept_groups_kernel
    if (warp == 0) {
        int nseg = 0;
        for (int g0 = 0; g0 < n_active; g0 += 32) {
            const int g = g0 + lane;
            const int grp = g < n_active ? s_grp[g] : -1;
            const bool start = g < n_active && (g == 0 || s_grp[g - 1] != grp);
            const unsigned m = __ballot_sync(0xffffffffu, start);
            const int k = nseg + __popc(m & ((2u << lane) - 1u)) - 1;
            if (g < n_active) s_pseg[g] = k;
            if (start) s_seg_grp[k] = grp;
            nseg += __popc(m);
        }
        if (lane == 0) s_nseg = nseg;
    }
    __syncthreads();
    const int nseg = s_nseg;
    for (int k = threadIdx.x; k < nseg; k += blockDim.x) { s_seg_f[k] = cb.groups[s_seg_grp[k]].iter; s_seg_go[k] = 0; }
    if (threadIdx.x == 0 && st.hist) st.hist[iter] = n_active;
    __syncthreads();
    // token append (pred is indexed by live position); the K/V row of the step's input token goes to cache position f
    for (int g = threadIdx.x; g < n_active; g += blockDim.x) {
        const int b = s_active[g], k = s_pseg[g], f = s_seg_f[k];
        const int tok = st.pred[g];
        st.gen[(long long)b * st.gen_ld + f + 1] = tok;
        st.front[b] = f + 1;
        reinterpret_cast<int4*>(st.sel)[g] = make_int4(b, f, 0, 0);
        if (tok != st.eos && tok != st.pad) s_seg_go[k] = 1;
    }
    __syncthreads();
    // per batch: the stop rule of generate() (every row predicted EOS or PAD in this step, or the rows are full)
    for (int k = threadIdx.x; k < nseg; k += blockDim.x) {
        const int f = s_seg_f[k];
        const bool open = s_seg_go[k] && f + 2 < st.max_len;
        CbGroup& gr = cb.groups[s_seg_grp[k]];
        gr.iter = f + 1;
        gr.tokens += gr.B;
        gr.live = open ? gr.B : 0;
        gr.closed = open ? 0 : 1;
        s_seg_go[k] = open ? 1 : 0;
    }
    __syncthreads();
    // live list and descriptors of the coming step without the stopped batches (order preserved); positions of the stopped
    if (warp == 0) {
        int w = 0, n_stop = 0;
        for (int g0 = 0; g0 < n_active; g0 += 32) {
            const int g = g0 + lane;
            const bool keep = g < n_active && s_seg_go[s_pseg[g]];
            const bool stop = g < n_active && !keep;
            const unsigned m = __ballot_sync(0xffffffffu, keep), ms = __ballot_sync(0xffffffffu, stop);
            const unsigned lt = (1u << lane) - 1u;
            if (keep) {
                const int pos = w + __popc(m & lt);
                const int b = s_active[g];
                st.active[pos] = b;
                st.desc[pos] = make_int4(b, s_seg_f[s_pseg[g]] + 1, st.pred[g], st.src_len[b]);
            }
            if (stop) s_stop[n_stop + __popc(ms & lt)] = g;
            w += __popc(m);
            n_stop += __popc(ms);
        }
        if (lane == 0) {
            st.ctrl[CTRL_N_SEL] = n_active;
            st.ctrl[CTRL_N_ACTIVE] = w;
            st.ctrl[CTRL_ITERS] = iter + 1;
            st.ctrl[CTRL_DONE] = w == 0 ? 1 : 0;
            s_nstop = n_stop;
        }
    }
    __syncthreads();
    // stopped batches: their slots may be handed out again before the next advance kernel, which skips a < 0; each row goes
    // to the batch's output at its index in the batch, tokens 0 .. f + 1 and PAD behind them (as greedy_std_step_kernel)
    const int n_stop = s_nstop;
    for (int i = threadIdx.x; i < n_stop; i += blockDim.x) st.sel[s_stop[i] * 4 + 3] = -1;
    for (long long idx = threadIdx.x; idx < (long long)n_stop * st.max_len; idx += blockDim.x) {
        const int g = s_stop[idx / st.max_len], c = (int)(idx % st.max_len);
        const int b = s_active[g], f = s_seg_f[s_pseg[g]];
        long long* out = cb.groups[s_grp[g]].out + (long long)cb.slots.slot_q[b] * st.max_len;
        out[c] = c <= f + 1 ? st.gen[(long long)b * st.gen_ld + c] : st.pad;
    }
}
int launch_greedy_std_step_groups(const GreedyState& st, const CbTable& cb, cudaStream_t s) {
    const size_t smem = (size_t)7 * st.B * sizeof(int);
    if (ensure_dyn_smem(greedy_std_step_groups_kernel, (int)smem)) return 1;   // error recorded by ensure_dyn_smem
    TTB_CUDA_OK(launch_pdl(greedy_std_step_groups_kernel, dim3(1), dim3(st.B < 1024 ? ((st.B + 31) / 32 * 32) : 1024), smem, s, st, cb));
    return 0;
}

}  // namespace ttb
