// Kernel launchers of libttb200.  Every launcher enqueues on `stream` and never synchronises.
//
// Row counts that are only known on the device (the number of live queries shrinks while
// decoding) are passed as `RowCount{max_rows, units_dev, rows_per_unit}`: the grid is sized for
// `max_rows`, each block reads `*units_dev * rows_per_unit` and exits early beyond it.
#pragma once
#include "common.cuh"

namespace ttb {

struct RowCount {
    int max_rows;            // host-side upper bound (grid sizing)
    const int* units_dev;    // nullptr -> all max_rows rows are live
    int rows_per_unit;
    __host__ __device__ RowCount(int m = 0, const int* u = nullptr, int r = 1) : max_rows(m), units_dev(u), rows_per_unit(r) {}
    __device__ __forceinline__ int live() const { return units_dev ? (*units_dev) * rows_per_unit : max_rows; }
};

// ---- elementwise.cu ----------------------------------------------------------------------
void launch_i64_to_i32(const long long* in, int* out, long long n, cudaStream_t s);
void launch_i32_to_i64(const int* in, long long* out, long long n, cudaStream_t s);
void launch_mask_to_tokens(const unsigned char* mask, int* out, long long n, int pad_id, cudaStream_t s);
// out[b] = 1 + index of the last token of row b that differs from pad_id (0 for an all-pad row)
void launch_row_lengths(const int* tok, int B, int L, int pad_id, int* out, cudaStream_t s);
// x[t] = table[tok[t]] + pe[(t % L) + 1]; also writes the low-precision copy when xh != nullptr
template <typename ActT>
void launch_embed_seq(const int* tok, int T, int L, const float* table, const float* pe, int E,
                      float* x, ActT* xh, cudaStream_t s);
// out = LN(resid + y) * g + b ; optional second LN (final norm of the stack) applied on top
template <typename ActT>
void launch_add_layernorm(const float* resid, const float* y, const float* g, const float* b,
                          const float* g2, const float* b2, float* out, ActT* outh,
                          RowCount rows, int E, cudaStream_t s);
void launch_argmax_rows(const float* logits, int ld, int V, int* out, RowCount rows, cudaStream_t s);

// ---- gemm_simt.cu : C[M,N] = A[M,K] * W[N,K]^T + bias (fp32 FMA, exact-precision path) -------
template <typename OutT>
void launch_gemm_f32(const float* A, int lda, const float* W, const float* bias, OutT* C, int ldc,
                     RowCount rows, int N, int K, bool relu, cudaStream_t s);

// ---- gemm_tcgen05.cu : same contract, bf16 operands, fp32 accumulation in TMEM (tcgen05.mma) ----
// A is [M,K] bf16 row-major (lda elements), W is [N,K] bf16 row-major; both are TMA-loaded.
template <typename OutT>
int launch_gemm_bf16_tc(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias,
                        OutT* C, int ldc, RowCount rows, int N, int K, bool relu, cudaStream_t s);

// Fused sub-layer tail for embedding_dim 256 (bf16 path):  x <- LN2?(LN1(x + A W^T + bias)), x fp32 updated in
// place, xh = bf16 copy.  W is [256, K] bf16; g2/b2 = nullptr without the second LayerNorm.  Optional chained
// projection of the result (K == 256 only): q2 = xh W2^T + bias2 with W2 [256, 256] bf16 (the cross-attention query).
int launch_gemm_resid_ln(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias, float* x, __nv_bfloat16* xh,
                         const float* g1, const float* b1, const float* g2, const float* b2, RowCount rows, int K, cudaStream_t s,
                         const __nv_bfloat16* W2 = nullptr, const float* bias2 = nullptr, __nv_bfloat16* q2 = nullptr);

// Vocabulary projection fused with arg-max (greedy loop, bf16 path): pred[row] = argmax_v(A[row] . W[v] + bias[v]).
// Returns -1 when the shape does not fit the kernel (K % 64, V <= 512, shared memory) so the caller can fall back.
int launch_classifier_argmax(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias, int* pred, RowCount rows,
                             int V, int K, cudaStream_t s);

// Vocabulary projection fused with the statistics of the speculative beam search (bf16 path, n_best <= 16): per row the soft-max
// maximum / sum, the n_best largest logits (descending, ties: lower id) and their ids, the nucleus-truncated support size
// and the logit of token row_tok[row] -- everything beam_choose / beam_expand read; the logits never leave tensor memory.
// Returns -1 when the shape does not fit (caller: logits GEMM + launch_beam_stats).
int launch_classifier_stats(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias, RowCount rows, int V, int Kdim, int n_best,
                            const int* row_tok, float* tokv, float* lmax, float* lsum, int* nkeep, float* topv, int* topi, cudaStream_t s);

// Fused feed-forward sub-layer for embedding_dim 256 (bf16 path):
//   x <- LN2?(LN1(x + relu(xh W1^T + b1) W2^T + b2)), x fp32 and its bf16 copy xh both updated in place.
// Chained form (att, Wo given; only with the CTA-pair kernel, see ffn_pair_available): the same launch first computes the
// preceding sub-layer tail x <- LN0(x + att Wo^T + bias_o) (the cross-attention out-projection), i.e. xh is not read.
int launch_ffn_fused(__nv_bfloat16* xh, const __nv_bfloat16* W1, const float* bias1, const __nv_bfloat16* W2, const float* bias2,
                     float* x, const float* g1, const float* b1, const float* g2, const float* b2, RowCount rows, int F, cudaStream_t s,
                     const __nv_bfloat16* att = nullptr, const __nv_bfloat16* Wo = nullptr, const float* bias_o = nullptr,
                     const float* g0 = nullptr, const float* b0 = nullptr);
bool ffn_pair_available(int max_rows);   // the cta_group::2 feed-forward kernel can run all its clusters co-resident

// ---- attention.cu ---------------------------------------------------------------------------
// Generic masked attention over "groups".  Queries of group g are tokens g*Lq .. g*Lq+Lq-1 of
// `q`; its keys/values are rows kv_row0 .. kv_row0+Lk-1 with kv_row0 = (kvmap ? kvmap[g] : g) *
// kv_group_stride.  Key j is masked when key_tok[(kvmap?kvmap[g]:g)*key_tok_stride + j] == pad_id,
// and, when `causal`, when j > i.
template <typename ActT>
void launch_attention(const ActT* q, int q_ld, const ActT* k, const ActT* v, int kv_ld,
                      ActT* out, int out_ld, int n_groups_max, const int* n_groups_dev,
                      int Lq, int Lk, long long kv_group_stride, const int* kvmap,
                      const int* key_tok, int key_tok_stride, int pad_id, bool causal,
                      int heads, int head_dim, cudaStream_t s, const int* lk_dev = nullptr);

// Speculative self-attention: group g = live query slot; b = active[g]; f = front[b].
// Queries: rows (g*N + n)*(D+1) + i of `qkv` (q | k | v packed, row stride qkv_ld).
// Keys: cache positions 0..f-1 of query b (masked where gen[b][j] == pad) followed by the new
// keys i' <= i of the same draft row (i' = 0 is masked when gen[b][f] == pad).
template <typename ActT>
void launch_spec_self_attention(const ActT* qkv, int qkv_ld, const ActT* kcache, const ActT* vcache,
                                long long cache_query_stride, int cache_ld, ActT* out, int out_ld,
                                int B_max, const int* n_active_dev, const int* active, const int* front,
                                const int* gen, int gen_ld, int pad_id, int N, int D,
                                int heads, int head_dim, int max_cache_len, cudaStream_t s);

// ---- attention_mma.cu : tensor-core (mma.sync bf16) versions of the two entry points above ----------
void launch_attention_mma(const __nv_bfloat16* q, int q_ld, const __nv_bfloat16* k, const __nv_bfloat16* v, int kv_ld,
                          __nv_bfloat16* out, int out_ld, int n_groups_max, const int* n_groups_dev,
                          int Lq, int Lk, long long kv_group_stride, const int* kvmap,
                          const int* key_tok, int key_tok_stride, int pad_id, bool causal,
                          int heads, int head_dim, cudaStream_t s, const int* lk_dev = nullptr, const int* lk_group = nullptr,
                          const int4* desc = nullptr);
void launch_spec_self_attention_mma(const __nv_bfloat16* qkv, int qkv_ld, const __nv_bfloat16* kcache, const __nv_bfloat16* vcache,
                                    long long cache_query_stride, int cache_ld, __nv_bfloat16* out, int out_ld,
                                    int B_max, const int* n_active_dev, const int* active, const int* front,
                                    const int* gen, int gen_ld, int pad_id, int N, int D,
                                    int heads, int head_dim, cudaStream_t s, const int4* desc = nullptr, bool group_row_len = false);
// group_row_len (needs desc): group g's draft rows are desc[g].w <= D + 1 positions long (the rest of each row of the call is
// ignored and not written), and its outputs are the bits a call with D + 1 = desc[g].w gives

// ---- drafting.cu ------------------------------------------------------------------------------
// Mirrors utils/drafting.py::make_drafts on device; src is (B, L) int32 with row stride src_ld (the
// caller skips the BOS column by passing src + 1, L - 1).  out is (B, N, Deff) int32.
void launch_make_drafts(const int* src, int src_ld, int B, int L, int Deff, int N, int eos, int pad, int replace,
                        int* out, cudaStream_t s);

// ---- greedy.cu -------------------------------------------------------------------------------
struct GreedyState {
    int B, N, D, max_len, gen_ld, pad, bos, eos, Ls;
    int* gen;          // [B][gen_ld] generated tokens (row b of the reference's token matrix)
    int* front;        // [B] index of the last generated token
    int* active;       // [B] compact list of live query ids (order preserved, like boolean masking)
    int* ctrl;         // [CTRL_COUNT]
    const int* drafts; // [B][N][D]
    int* pred;         // [B*N*(D+1)] argmax predictions of the current iteration
    long long* out;    // [B][max_len] finished predictions (int64 like the reference)
    int* sel;          // [B][4] per pre-retirement slot: {query id, old front, draft index, n_accepted}
    int* trace;        // optional [max_len][B][4] = {query id, n_accepted, draft index, width}
    int tie_break;     // 0 = torch-CPU topk(1) emulation, 1 = lowest index
    int* hist;         // [max_len + 2] live queries at the start of every iteration
    int4* desc;        // [B] per live slot of the COMING iteration: {query id, front, token at front, source length};
                       // written by the init / accept kernels so that the kernels of an iteration need one load
                       // instead of the chain active[g] -> front[b] -> gen[b][front]
    const int* src_len;  // [B] source length per query (cross-attention key bound), may be nullptr
};
void launch_greedy_init(const GreedyState& st, cudaStream_t s);
// First kernel of an iteration: appends the K/V rows of the tokens accepted in the previous iteration (chosen
// draft recorded in st.sel) to the self-attention cache of every layer, and embeds the (D+1) step tokens of
// every live draft row.
template <typename ActT>
void launch_greedy_advance(const GreedyState& st, const float* table, const float* pe, int E, float* x, ActT* xh,
                           const ActT* qkv_all, long long qkv_layer_stride, int n_layers, int qkv_ld, ActT* kcache, ActT* vcache,
                           long long cache_layer_stride, long long cache_query_stride, int cache_ld, cudaStream_t s);
// picks the best draft per live query, appends tokens, retires finished queries, plans next width
void launch_greedy_accept(const GreedyState& st, cudaStream_t s);
// standard greedy decoding (no drafts: N = 1, D = 0): appends the predicted token of every row, stop test
void launch_greedy_std_step(const GreedyState& st, cudaStream_t s);

// ---- continuous batching, common to the three loops: several batches share the query slots of one loop ----------
// Slot table of a continuous loop, written by the loop's admission kernel.
struct SlotTable {
    int* slot_group;   // [slots] batch of the query in the slot, -1 = free (the greedy loop does not reset it: its free
                       // slots are the ones outside the live list)
    int* slot_q;       // [slots] index of that query in its batch
    int* adm_slots;    // [max batch size] slots given to the batch admitted last
};
// cross-attention K/V rows [layer][Bi * Ls][2E] and source tokens [Bi][Ls] of the batch admitted last -> its slots adm_slots
// (rows [0, Ls) of slot b at b * Ls_cap; key tokens PAD behind Ls); greedy.cu
template <typename ActT>
void launch_admit_kv(const int* adm_slots, int Bi, int Ls, int Ls_cap, int n_layers, int E, const ActT* stage_kv, long long stage_layer_stride,
                     ActT* kv, long long layer_stride, const int* src32, int* keytok, int pad, cudaStream_t s);

// Continuous batching of the speculative loop (GreedyState::B = number of slots; every per-query array is per slot).
// One record per batch: what the reference couples across the queries of a batch (width, stop, errors) plus its counters.
// The standard greedy loop uses the same record without width and errors (W, accepted, error and n_left stay 0 or unused).
struct CbGroup {
    long long* out;    // [B][max_len] the batch's predictions
    int* trace;        // optional [max_len + 1][B][4], rows indexed by the batch's own iteration and live position
    int B, W;          // batch size; token-matrix width of the batch's coming iteration
    int iter, live;    // decoder iterations the batch took part in; its live queries
    int accepted, tokens, error, n_left, closed;   // counters; error 0 / 1 (splice index) / 2 (shape); unfinished queries
    int reserved;
};
struct CbTable {
    SlotTable slots;
    CbGroup* groups;   // [n_batches]
};
// admission of batch `grp` between two iterations (drafts_in [Bi][N][D], srclen_in [Bi] computed for the batch alone); 0 or an
// error code
int launch_greedy_admit(const GreedyState& st, const CbTable& cb, int grp, int Bi, const int* drafts_in, const int* srclen_in, long long* out,
                        int* trace, int Ls_cap, cudaStream_t s);
// accept kernel of the continuous loop: per-query step of launch_greedy_accept, per-batch retirement / width plan / closing
void launch_greedy_accept_groups(const GreedyState& st, const CbTable& cb, cudaStream_t s);
// step kernel of the continuous loop without drafts (N = 1, D = 0): token append of launch_greedy_std_step with the step
// count, stop rule and output of each batch; stopped batches leave the live list whole; 0 or an error code
int launch_greedy_std_step_groups(const GreedyState& st, const CbTable& cb, cudaStream_t s);

// ---- beam.cu --------------------------------------------------------------------------------------
struct BeamState {
    int B, K, N, dl0, V, pad, bos, eos, ldw, tie_break;
    int max_len, w0;                      // length budget of the loop; width of the token matrix in the first iteration
    int* cand_cur; int* cand_next;        // [B*K][ldw] hypotheses (query-major), ping-pong
    float* logp_cur; float* logp_next;    // [B*K]
    const int* drafts;                    // [B][N][dl0]
    int* c_slot0; int* c_fin; int* c_rowbase; int* c_nacc; int* c_pick; int* acc_stat; int* ctrl;
    // per live attention group (written by beam_prepare): {candidate, front, token at front, -} for the self-attention
    // over the candidate caches and {query, -, -, source length} for the cross-attention: one 16-byte load per CTA instead
    // of the chain live list -> front -> token, and everything the attention kernels may read ahead of their dependency wait
    int4* desc_self; int4* desc_cross; const int* src_len;
    int* host_ctrl;   // pinned host mirror of ctrl (device-accessible): BC_COUNT words + a sequence word written last
    float* topv; int* topi; int* nkeep; float* lmax; float* lsum;      // per (row, position) statistics
    // token whose logit the accepted-path sums need at (row, position) = the row's next draft token (-1 behind the last
    // one), written by the embedding kernel; its logit, written by the statistics kernel
    int* row_tok; float* tokv;
    int* trace_nacc; int* trace_pick;     // optional [iter][B*K][N] / [iter][B*K]
    // live candidates as attention groups, cache bookkeeping of the new candidates
    int* live_cand; int* live_query;      // [live candidates] candidate index / query index
    int* c_front;                         // [B*K] cached positions of a candidate = first free slot - 1
    int* n_parent; int* n_keep; int* n_row;   // [B*K] new candidate: parent (-1: finished parent), accepted draft tokens, decoder row
    // smart_drafts_mode (speculative_decoding.py:600-845): `drafts` is the window library [B][n_lib][dl0] whose first
    // token is the key; a candidate tries the windows that start with its last token
    int smart, n_lib;
    int* tok_cnt; int* tok_list;          // [B][V] number of windows per first token (1..N), [B][V][N] their library indices
    int* c_cnt; int* c_last;              // [B*K] rows (drafts) of a candidate, its last token
    int* row_draft;                       // [rows] library index of the row's draft
};
void launch_beam_build_lib(const BeamState& st, cudaStream_t s);
void launch_beam_init(const BeamState& st, cudaStream_t s);
void launch_beam_prepare(const BeamState& st, int C, int beam, int dl, cudaStream_t s);
// embeds (last token, draft tokens) of every live (candidate, draft) row at positions front .. front+dl
template <typename ActT>
void launch_beam_embed_cached(const BeamState& st, int beam, int max_rows, int dl, const float* table, const float* pe, int E,
                              float* x, ActT* xh, cudaStream_t s);
// new candidate c' <- cache of its parent [0, front) + K/V of positions front .. front + n_keep of the chosen draft row
template <typename ActT>
void launch_beam_cache_update(const BeamState& st, int dl, const ActT* qkv_all, long long qkv_layer_stride, int n_layers, int qkv_ld,
                              int E, const ActT* kc_cur, const ActT* vc_cur, ActT* kc_next, ActT* vc_next, long long cache_layer_stride,
                              long long cache_cand_stride, cudaStream_t s);
void launch_beam_stats(const BeamState& st, const float* logits, int max_rows, int dl, cudaStream_t s);
void launch_beam_choose(const BeamState& st, int C, int beam, int dl, cudaStream_t s);
void launch_beam_expand(const BeamState& st, int beam, int dl, cudaStream_t s);
void launch_beam_export(const int* cand, int ldw, int R, int W, long long* out, cudaStream_t s);

// Continuous batching of the speculative beam search (BeamState::B = number of query slots; slot b owns candidates
// b K .. b K + K - 1).  One record per batch: what the reference couples across the queries of a batch plus its counters.
struct BcGroup {
    long long* out;                       // [B][K][W] the batch's hypotheses, rewritten at its width every iteration
    int* trace_nacc; int* trace_pick;     // optional, indexed by the batch's own iteration and candidate numbering
    int B, W, dl, iter;                   // batch size; width and draft length of its coming iteration; iterations taken part in
    int lmax;                             // smart drafts: most drafts of one candidate in the current iteration
    int accepted, produced, error, closed;   // counters; error 0 / 3 / 4 as BC_ERROR; 1 once the batch has stopped
    int all_fin, min_pad, acc, cnt;       // accumulators of the iteration in flight
};
struct BcTable {
    SlotTable slots;
    BcGroup* groups;   // [n_batches]
    int n_groups;      // batches admitted so far
    int* dl_min;       // [iterations] smallest draft length among the batches of every iteration
};
// admission of batch `grp` between two iterations: drafts_in [Bi][N][dl0] (smart: [Bi][lib_in][dl0] window library with
// tok_cnt_in [Bi][V], tok_list_in [Bi][V][N]), srclen_in [Bi], all computed for the batch alone; 0 or an error code
int launch_beam_admit(const BeamState& st, const BcTable& cb, int grp, int Bi, const int* drafts_in, int lib_in, const int* tok_cnt_in,
                      const int* tok_list_in, const int* srclen_in, long long* out, int* trace_nacc, int* trace_pick, int dl_first, cudaStream_t s);
// group-aware prepare / choose / expand; `dl` = draft length of the decoder call (the largest of the open batches)
void launch_beam_prepare_groups(const BeamState& st, const BcTable& cb, cudaStream_t s);
void launch_beam_choose_groups(const BeamState& st, const BcTable& cb, int dl, cudaStream_t s);
void launch_beam_expand_groups(const BeamState& st, const BcTable& cb, int dl, cudaStream_t s);
// ---- std_beam.cu : standard beam search (standard_decoding.py:90-174) -------------------------------------------
struct StdBeamState {
    int B, K, V, pad, bos, eos, ldw;
    int max_len;                          // continuous loop: a batch stops after max_len - 1 steps
    int* y_cur; int* y_next;              // [B*K][ldw] hypotheses (query-major), ping-pong
    float* score_cur; float* score_next;  // [B*K]
    int* fin; int* cand_row;              // [B*K] contains EOS / live-row index, -1 (finished) or -2 (absent)
    int* row_cand; int* row_query;        // [live rows]
    float* total;                         // [B*K][V] score + log-softmax
    int* ctrl;                            // [0] live rows, [1] hypotheses with EOS after the selection
    // KV cache: one new token per live hypothesis and step
    int* c_front;                         // [B*K] cached positions of a hypothesis (= W - 1 of its batch)
    int* parent;                          // [B*K] hypothesis of the previous step a new hypothesis continues, -1: none
    int4* desc_self; int4* desc_cross;    // per live row: {hypothesis, front, token at front, -} / {query, -, -, source length}
    const int* src_len;
    unsigned long long* host_ctrl;        // continuous loop: pinned mapped ring of four words the closing CTA posts into
};
void launch_sbeam_init(const StdBeamState& st, cudaStream_t s);
void launch_sbeam_prepare(const StdBeamState& st, int C, int beam, int W, cudaStream_t s);
void launch_sbeam_scores(const StdBeamState& st, int C, const float* logits, cudaStream_t s);
int launch_sbeam_select(const StdBeamState& st, int beam, int W, cudaStream_t s);
// shared memory of the selection of a query with `beam` hypotheses fits the kernel
bool sbeam_select_fits(int beam, int V);
// embedding of the last token (position front = W - 1 of desc_self) of every live hypothesis
template <typename ActT>
void launch_sbeam_embed_last(const StdBeamState& st, int max_rows, const float* table, const float* pe, int E, float* x, ActT* xh,
                             cudaStream_t s);
// cache of a new hypothesis = cache of its parent [0, W - 1) + K/V of the parent's row of this step (position W - 1, W of
// the parent's batch)
template <typename ActT>
void launch_sbeam_cache_update(const StdBeamState& st, const ActT* qkv_all, long long qkv_layer_stride, int n_layers, int qkv_ld, int E,
                               const ActT* kc_cur, const ActT* vc_cur, ActT* kc_next, ActT* vc_next, long long cache_layer_stride,
                               long long cache_cand_stride, cudaStream_t s);

// Continuous batching of the standard beam search (StdBeamState::B = number of query slots; slot q owns hypotheses
// q K .. q K + K - 1).  One record per batch: what the reference couples across the queries of a batch.
struct SbGroup {
    long long* out;      // [B][K][W + 1] the batch's hypotheses, rewritten at its width every step
    int B, W, beam;      // batch size; hypothesis width and hypotheses per query of its coming step
    int steps;           // steps taken part in (model calls)
    int n_eos, closed;   // hypotheses with EOS after the selection of the step in flight; 1 once the batch has stopped
};
struct SbTable {
    SlotTable slots;
    SbGroup* groups;     // [n_batches]
    int n_groups;        // batches admitted so far
};
// control words of the continuous loop behind the ones of generate()
constexpr int SBC_TICKET = 4, SBC_USED = 5, SBC_SEQ = 6, SBC_ADM_ERR = 7;
// admission of batch `grp` (Bi queries, srclen_in [Bi]) into the first Bi free slots, between two steps; 0 or an error code
int launch_sbeam_admit(const StdBeamState& st, const SbTable& cb, int grp, int Bi, const int* srclen_in, long long* out, cudaStream_t s);
// group-aware prepare and select; the select kernel's last CTA closes the step of every open batch and posts the word
// sequence (24 bits) | slots in use (16) | live rows of the next step (24)
void launch_sbeam_prepare_groups(const StdBeamState& st, const SbTable& cb, cudaStream_t s);
int launch_sbeam_select_groups(const StdBeamState& st, const SbTable& cb, int max_beam, cudaStream_t s);

// ---- sampling.cu : sampling decoding (the greedy loop with S sample slots per source, slot r = b * S + s) ---------------
// Per live position of the coming step, beside GreedyState::desc: the source of the slot (cross-attention K/V group of the
// fp32 kernels) and the cross-attention descriptor {source, -, -, source length} of the tensor-core kernels.
struct SampleLoop {
    int S;
    int* kvsrc;        // [B * S]
    int4* xdesc;       // [B * S]
};
// What a draw reads per live row g: slot and front from desc[g] (column t = front + 1), the source key keys[slot / S].
struct SampleArgs {
    const int4* desc;
    const unsigned long long* keys;
    int S;
    float temperature;
    int top_k;         // 0: whole vocabulary
    int* pred;         // [rows] drawn token
};
// keys[b] = FNV-1a-64(seed bytes, non-PAD tokens of src32[b]) (philox.cuh)
void launch_sample_keys(const int* src32, int B, int Ls, int pad, unsigned long long seed, unsigned long long* keys, cudaStream_t s);
void launch_sample_init(const GreedyState& st, const SampleLoop& sl, cudaStream_t s);
// in place of launch_greedy_std_step: token append, retirement of ended slots into st.out [B * S][max_len], compaction
void launch_sample_step(const GreedyState& st, const SampleLoop& sl, cudaStream_t s);
// draw over fp32 logits [rows][ld], any top_k
void launch_sample_rows(const float* logits, int ld, int V, RowCount rows, const SampleArgs& a, cudaStream_t s);
// Vocabulary projection fused with the draw (bf16 path): the classifier_argmax_kernel design with a Gumbel-max epilogue.
// Returns -1 where launch_classifier_argmax would, and for top_k > 8 (caller: logits GEMM + launch_sample_rows).
int launch_classifier_sample(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias, RowCount rows, int V, int K,
                             const SampleArgs& a, cudaStream_t s);

// ---- scoring.cu : teacher-forced scoring of given targets (G candidates, Lt columns each, int32 tokens tgt [G][Lt]) -----
// kvmap[g] = g / K (candidate -> source), row_tok[g * Lt + t] = tgt[g][t + 1] (-1 in the last column)
void launch_score_prepare(const int* tgt, int G, int Lt, int K, int* kvmap, int* row_tok, cudaStream_t s);
// per row of fp32 logits: logit of token row_tok[row] (0 when -1), soft-max maximum and sum of exp(logit - maximum)
void launch_logprob_stats(const float* logits, int ld, int V, const int* row_tok, int rows, float* tokv, float* lmax, float* lsum,
                          cudaStream_t s);
// per candidate: scored columns n (EOS / PAD rule), sum of tokv - lmax - log(lsum) over rows g * Lt + 0 .. n - 1, optional
// per-column values token_logp_out [G][Lt - 1] (0 at unscored columns)
void launch_score_reduce(const int* tgt, int G, int Lt, int pad, int eos, const float* tokv, const float* lmax, const float* lsum,
                         float* logp_out, int* ntok_out, float* token_logp_out, cudaStream_t s);

}  // namespace ttb
