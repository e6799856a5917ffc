/* libttb200 — C ABI of the B200-native translation-transformer inference hot path.
 *
 * Every entry point replaces one Python-level interface of Academich/translation-transformer
 * (the reference is pure Python/PyTorch; the file:line given with each function is the call a
 * reference maintainer would re-point, see INTEGRATION.md for the ctypes binding).
 *
 * Conventions
 *   - plain pointers and sizes only; no framework types.  `*_dev` pointers are device pointers of
 *     the engine's CUDA device, `stream` is a `cudaStream_t` passed as `void*` (NULL = default).
 *   - token ids are int64 at the boundary (torch.LongTensor in the reference).
 *   - every function returns 0 on success; otherwise `ttb_last_error()` describes the failure.
 *   - return code 10..19 = the reference itself would have raised at this point
 *     (TTB_ERR_REF_*), the Python wrappers re-raise the same exception type.
 *   - there is no CPU implementation behind this ABI: without a CUDA device every call fails.
 */
#ifndef TTB200_H
#define TTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TTB_ABI_VERSION 8

#define TTB_PRECISION_FP32 0 /* fp32 FMA GEMMs, exact-parity path (1e-5 logits)            */
#define TTB_PRECISION_BF16 1 /* tcgen05 bf16 GEMMs, fp32 accumulate (1e-2 logits)          */

#define TTB_ERR_REF_INDEX 10 /* reference: scatter index out of bounds (speculative_decoding.py:111) */
#define TTB_ERR_REF_SHAPE 11 /* reference: finished row wider than max_len (speculative_decoding.py:158) */
#define TTB_ERR_REF_ASSERT 12 /* reference: assert in topk_in_each_group (speculative_decoding.py:195) */

typedef struct ttb_engine ttb_engine;

/* Architecture of VanillaTransformer (src/model/modules.py:12-37). */
typedef struct {
    int32_t src_vocab_size, tgt_vocab_size;
    int32_t embedding_dim, feedforward_dim;
    int32_t num_encoder_layers, num_decoder_layers, num_heads;
    int32_t src_pad_token_idx, tgt_pad_token_idx;
    int32_t precision;      /* TTB_PRECISION_* */
    int32_t max_positions;  /* rows of the positional table minus one (the reference uses 5000) */
} ttb_model_desc;

/* Statistics of one generate() call (model_calls_num etc. of the reference generators). */
typedef struct {
    int32_t model_calls;      /* decoder invocations (speculative_decoding.py:121, :496, :742) */
    int32_t accepted_tokens;  /* draft tokens accepted                                         */
    int32_t produced_tokens;  /* accepted + bonus tokens                                       */
    int32_t unfinished;       /* queries still alive when the loop stopped                     */
    int32_t error;            /* 0, TTB_ERR_REF_INDEX or TTB_ERR_REF_SHAPE                     */
    int32_t gpu_launches;     /* kernels launched by this call                                 */
    float   gpu_ms;           /* device time of the call measured with CUDA events             */
    float   reserved;
} ttb_generate_stats;

int ttb_abi_version(void);
const char* ttb_last_error(void);
/* 0 if a usable sm_100 device is present */
int ttb_device_check(int device);

/* ---- engine lifecycle: replaces VanillaTransformer.__init__ + load_state_dict (modules.py:10-83) */
int ttb_engine_create(const ttb_model_desc* desc, int device, ttb_engine** out);
void ttb_engine_destroy(ttb_engine* e);
/* `name` is a key of VanillaTransformer.state_dict() (optionally prefixed "model.") or
 * "positional_encoding.pe"; `data` may be a host or a device pointer to `numel` floats. */
int ttb_engine_set_param(ttb_engine* e, const char* name, const float* data, int64_t numel);
int ttb_engine_finalize(ttb_engine* e);

/* ---- utils/drafting.py:5 make_drafts(src, draft_len, n_drafts, min_draft_len, max_draft_len,
 *      eos_token_idx, pad_token_idx, replace_token_idx) -> (B, N, D) int64
 * src_dev is (B, L) int64 with row stride src_ld.  Returns D (clamped draft length) in *d_out. */
int ttb_make_drafts(const int64_t* src_dev, int64_t src_ld, int32_t B, int32_t L, int32_t draft_len,
                    int32_t n_drafts, int32_t min_draft_len, int32_t max_draft_len, int32_t eos,
                    int32_t pad, int32_t replace, int64_t* out_dev, int32_t* d_out, void* stream);

/* ---- modules.py:108 encode_src(src, src_pad_mask) -> memory (B, Ls, E) fp32
 * src_pad_mask_dev may be NULL (then src == src_pad_token_idx, as every caller does). */
int ttb_encode_src(ttb_engine* e, const int64_t* src_dev, const uint8_t* src_pad_mask_dev, int32_t B,
                   int32_t Ls, float* memory_out_dev, void* stream);

/* ---- modules.py:117 decode_tgt(tgt, memory, memory_pad_mask) -> logits (B, Lt, V) fp32 */
int ttb_decode_tgt(ttb_engine* e, const int64_t* tgt_dev, int32_t B, int32_t Lt, const float* memory_dev,
                   const uint8_t* memory_pad_mask_dev, int32_t Ls, float* logits_out_dev, void* stream);

/* ---- speculative_decoding.py:39 TranslationInferenceGreedySpeculative.generate(src)
 * Whole decoding loop on the device (encoder, drafts, KV-cached decoder steps, verification,
 * retirement).  out_dev is (B, max_len) int64 (the reference returns it with a singleton middle
 * dimension).  trace_dev is optional: (max_len, B, 4) int32 = {query, n_accepted, draft, width}
 * per iteration and live slot.  tie_break: 0 = torch-CPU topk(1) order, 1 = lowest index. */
int ttb_greedy_speculative_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls,
                                    int32_t max_len, int32_t draft_len, int32_t n_drafts, int32_t pad_token,
                                    int32_t bos_token, int32_t eos_token, int32_t replace_token,
                                    int32_t tie_break, int64_t* out_dev, int32_t* trace_dev,
                                    ttb_generate_stats* stats, void* stream);

/* ---- continuous batching of speculative_decoding.py:39 generate(): n_batches independent batches share `slots`
 * query slots of ONE device loop.  Batch i is admitted (in list order) as soon as `batch_sizes[i]` slots are free;
 * its queries keep the width / stop / error rules of their own batch, so out_devs[i], trace_devs[i] and stats[i]
 * are exactly what ttb_greedy_speculative_generate returns for that batch alone.  A reference failure of one batch
 * (stats[i].error = TTB_ERR_REF_*) ends that batch only; the call returns 0 unless something else failed.
 * src_devs[i] is (batch_sizes[i], src_lens[i]) int64, out_devs[i] (batch_sizes[i], max_len) int64, trace_devs[i]
 * (max_len + 1, batch_sizes[i], 4) int32 like trace_dev above (query ids are indices within the batch).
 * slots >= max(batch_sizes).  trace_devs may be NULL, or hold NULL entries.  total (may be NULL): launches / ms of the
 * call, model_calls = decoder iterations of the shared loop.  The loop runs the default attention kernels (not the
 * opt-in tcgen05 attention).  ttb_engine_get_history afterwards gives the live slots of every iteration. */
int ttb_greedy_speculative_generate_batches(ttb_engine* e, int32_t n_batches, const int64_t* const* src_devs,
                                            const int32_t* batch_sizes, const int32_t* src_lens, int32_t slots, int32_t max_len,
                                            int32_t draft_len, int32_t n_drafts, int32_t pad_token, int32_t bos_token,
                                            int32_t eos_token, int32_t replace_token, int32_t tie_break, int64_t* const* out_devs,
                                            int32_t* const* trace_devs, ttb_generate_stats* stats, ttb_generate_stats* total,
                                            void* stream);

/* ---- standard_decoding.py:29 TranslationInferenceGreedy.generate(src)
 * Plain greedy decoding, one token per row and step, on the same KV-cached device loop (no drafts).  Like the
 * reference, rows keep decoding after their EOS until every row predicts EOS or PAD in the same step.
 * out_dev is (B, max_len) int64, PAD behind the last generated column. */
int ttb_greedy_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, int32_t max_len, int32_t pad_token,
                        int32_t bos_token, int32_t eos_token, int64_t* out_dev, ttb_generate_stats* stats, void* stream);

/* ---- continuous batching of standard_decoding.py:29 generate(): n_batches independent batches share `slots` query slots
 * of ONE device loop.  Batch i is admitted (whole, in list order) between two steps as soon as `batch_sizes[i]` slots are
 * free; it keeps the step count and stop rule of its own batch (every row predicted EOS or PAD in the same step, or the
 * rows are full) and frees its slots when it stops, so out_devs[i] and stats[i] are exactly what ttb_greedy_generate
 * returns for that batch alone (launches and time belong to the call, in `total`).  src_devs[i] is (batch_sizes[i],
 * src_lens[i]) int64, out_devs[i] (batch_sizes[i], max_len) int64.  max(batch_sizes) <= slots <= 2048.  Arguments
 * ttb_greedy_generate rejects are rejected with the same error before any device work.  total (may be NULL): launches /
 * ms of the call, model_calls = steps of the shared loop.  ttb_engine_get_history afterwards gives the query slots in use
 * at every step. */
int ttb_greedy_generate_batches(ttb_engine* e, int32_t n_batches, const int64_t* const* src_devs, const int32_t* batch_sizes,
                                const int32_t* src_lens, int32_t slots, int32_t max_len, int32_t pad_token, int32_t bos_token,
                                int32_t eos_token, int64_t* const* out_devs, ttb_generate_stats* stats, ttb_generate_stats* total,
                                void* stream);

/* ---- standard_decoding.py:90 TranslationInferenceBeamSearch.generate(src)
 * Standard beam search: one decoder call per generated column on the hypotheses without EOS; scores are
 * log(softmax(logits)) sums, finished hypotheses continue with PAD (artificial logits), the beam_size best of the
 * beam x vocabulary continuations survive (sorted).  out_dev must hold B * beam_size * max_len int64; the
 * hypotheses are written densely as (B, beam_size, *out_width). */
int ttb_beam_search_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, int32_t max_len, int32_t beam_size,
                             int32_t pad_token, int32_t bos_token, int32_t eos_token, int64_t* out_dev, int32_t* out_width,
                             ttb_generate_stats* stats, void* stream);

/* ---- continuous batching of standard_decoding.py:90 generate(): n_batches independent batches share `slots` query slots
 * of ONE device loop, each slot holding beam_size hypotheses.  Batch i is admitted (whole, in list order) between two steps
 * as soon as `batch_sizes[i]` slots are free; it keeps the width, first step and stop rule of its own batch and frees its
 * slots when it stops, so out_devs[i], out_widths[i] and stats[i].model_calls are exactly what ttb_beam_search_generate
 * returns for that batch alone (the other fields of stats[i] are 0: launches and time belong to the call, in `total`).
 * src_devs[i] is (batch_sizes[i], src_lens[i]) int64; out_devs[i] holds batch_sizes[i] * beam_size *
 * max_len int64 and receives (batch_sizes[i], beam_size, out_widths[i]) densely.  slots >= max(batch_sizes).  Arguments
 * ttb_beam_search_generate rejects are rejected with the same error before any device work.  total (may be NULL):
 * launches / ms of the call, model_calls = steps of the shared loop.  ttb_engine_get_history afterwards gives the query
 * slots in use at every step. */
int ttb_beam_search_generate_batches(ttb_engine* e, int32_t n_batches, const int64_t* const* src_devs, const int32_t* batch_sizes,
                                     const int32_t* src_lens, int32_t slots, int32_t max_len, int32_t beam_size, int32_t pad_token,
                                     int32_t bos_token, int32_t eos_token, int64_t* const* out_devs, int32_t* out_widths,
                                     ttb_generate_stats* stats, ttb_generate_stats* total, void* stream);

/* ---- speculative_decoding.py:422 TranslationInferenceBeamSearchSpeculative.generate(src)
 * smart_drafts_mode = 0: "try all the drafts" (:428-598), every candidate tries the n_drafts source windows;
 * smart_drafts_mode = 1: :600-845, a candidate tries the windows of a (Ls - 5)-window library whose first token equals
 * its last token (at most n_drafts of them).  out_dev must hold B * n_best * (max_len + clamp(draft_len,5,200) + 4)
 * int64; the hypotheses are written densely as (B, n_best, *out_width).  Optional traces: trace_nacc_dev
 * (max_len, B*n_best, n_drafts) accepted length of every draft (-1 behind a candidate's last draft), trace_pick_dev
 * (max_len, B*n_best) chosen draft, per iteration. */
int ttb_beam_speculative_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, int32_t max_len,
                                  int32_t n_best, int32_t draft_len, int32_t n_drafts, int32_t smart_drafts_mode, int32_t pad_token,
                                  int32_t bos_token, int32_t eos_token, int32_t c_token, int32_t tie_break, int64_t* out_dev,
                                  int32_t* out_width, int32_t* trace_nacc_dev, int32_t* trace_pick_dev, ttb_generate_stats* stats,
                                  void* stream);

/* ---- continuous batching of speculative_decoding.py:422 generate(): n_batches independent batches share `slots` query
 * slots of ONE device loop, each slot holding n_best candidate rows.  Batch i is admitted (in list order) between two
 * iterations as soon as `batch_sizes[i]` slots are free; its queries keep the width / draft length / stop / error rules of
 * their own batch, so out_devs[i], out_widths[i], the traces and stats[i] are exactly what ttb_beam_speculative_generate
 * returns for that batch alone.  A reference failure of one batch (stats[i].error = TTB_ERR_REF_*) ends that batch only;
 * the call returns 0 unless something else failed.  src_devs[i] is (batch_sizes[i], src_lens[i]) int64, out_devs[i] holds
 * batch_sizes[i] * n_best * (max_len + clamp(draft_len,5,200) + 4) int64 and receives (batch_sizes[i], n_best,
 * out_widths[i]) densely; trace_nacc_devs[i] / trace_pick_devs[i] are laid out as in ttb_beam_speculative_generate with
 * B = batch_sizes[i] (the arrays may be NULL or hold NULL entries).  slots >= max(batch_sizes).  total (may be NULL):
 * launches / ms of the call, model_calls = decoder iterations of the shared loop.  ttb_engine_get_history afterwards
 * gives the query slots in use at every iteration. */
int ttb_beam_speculative_generate_batches(ttb_engine* e, int32_t n_batches, const int64_t* const* src_devs,
                                          const int32_t* batch_sizes, const int32_t* src_lens, int32_t slots, int32_t max_len,
                                          int32_t n_best, int32_t draft_len, int32_t n_drafts, int32_t smart_drafts_mode,
                                          int32_t pad_token, int32_t bos_token, int32_t eos_token, int32_t c_token, int32_t tie_break,
                                          int64_t* const* out_devs, int32_t* out_widths, int32_t* const* trace_nacc_devs,
                                          int32_t* const* trace_pick_devs, ttb_generate_stats* stats, ttb_generate_stats* total,
                                          void* stream);

/* ---- sampling decoding (no reference counterpart; DESIGN.md section 15).  src_dev (B, Ls) int64; out_dev (B, n_samples,
 * max_len) int64.  Sample s of source b starts from bos_token and appends one token per step drawn by the Gumbel-max rule:
 * argmax_v (logit_v / temperature + g_v) over the top_k largest logits (top_k = 0: the whole vocabulary; ties at the
 * boundary and between equal z go to the lower token id), g_v = -log(-log(u)) with u from Philox4x32-10 at counter
 * (column, s, v >> 2, 0) and key = FNV-1a-64(seed bytes, non-PAD tokens of src[b]).  A row ends at its first drawn
 * eos_token or pad_token (kept) or when it holds max_len tokens; PAD behind.  The samples of a source depend on its tokens,
 * the seed and the settings only (identical sources with one seed get identical samples).  Rejected before any device
 * work: B * n_samples > 2048, n_samples < 1, a temperature that is not finite and > 0, top_k outside [0, V],
 * max_len < 2, pad_token == eos_token, lengths above the positional table.  stats: model_calls = decoder steps,
 * produced_tokens = drawn tokens, unfinished = rows that reached max_len without EOS or PAD. */
int ttb_sample_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, int32_t max_len, int32_t n_samples, float temperature,
                        int32_t top_k, uint64_t seed, int32_t pad_token, int32_t bos_token, int32_t eos_token, int64_t* out_dev,
                        ttb_generate_stats* stats, void* stream);

/* ---- teacher-forced scoring of given targets (no reference counterpart; DESIGN.md §14).  src_dev (B, Ls) int64,
 * tgt_dev (B, K, Lt) int64 with column 0 = start token; candidate (b,k) is tgt[b,k,1:] up to and including its first
 * eos_token or up to its first pad_token.  logp_out_dev (B*K) f32 sums, ntok_out_dev (B*K) int32 scored positions,
 * token_logp_out_dev (B*K*(Lt-1)) f32 or NULL.  Encoder and cross-attention K/V once per source.  Whole sources are
 * processed in chunks of at most 32768 decoder rows; K * Lt > 32768 is rejected.  Token ids must lie in the vocabularies
 * and no source row may be all padding.  The call returns once the results are written. */
int ttb_score_targets(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, const int64_t* tgt_dev, int32_t K,
                      int32_t Lt, int32_t pad_token, int32_t eos_token, float* logp_out_dev, int32_t* ntok_out_dev,
                      float* token_logp_out_dev, void* stream);

/* ---- instrumentation (bench.py): per-kernel-class CUDA-event timing on the launching stream.
 * class_mask bit i enables class i (names via ttb_kernel_class_name); totals accumulate over
 * generate() calls until the next ttb_engine_set_profiling. */
int ttb_kernel_class_count(void);
const char* ttb_kernel_class_name(int32_t id);
int ttb_engine_set_profiling(ttb_engine* e, uint32_t class_mask);
int ttb_engine_get_profile(ttb_engine* e, int32_t n_classes, double* ms_out, int64_t* launches_out);
/* live queries at the start of every decoder iteration of the last generate() (continuous loops: query slots in use);
 * returns their number */
int ttb_engine_get_history(ttb_engine* e, int32_t* live_queries_out, int32_t capacity);
/* last ttb_beam_speculative_generate_batches: per decoder iteration, the draft length the call ran at and the smallest
 * draft length of the batches in it (smaller when a batch near max_len shares the call); returns the iteration count */
int ttb_engine_get_draft_history(ttb_engine* e, int32_t* call_dl_out, int32_t* min_dl_out, int32_t capacity);

/* Standalone GEMM entry used by the kernel unit tests and the roofline microbenchmark:
 * C[M,N] = A[M,K] * W[N,K]^T + bias (+ReLU).  precision selects the kernel; A/W are fp32 for
 * TTB_PRECISION_FP32 and bf16 (uint16 storage) for TTB_PRECISION_BF16; C is fp32. */
int ttb_gemm(int32_t precision, const void* A_dev, const void* W_dev, const float* bias_dev, float* C_dev,
             int32_t M, int32_t N, int32_t K, int32_t relu, void* stream);

/* Same with a bf16 result (the form the decoder uses for the QKV / cross K-V projections: wide K = 256 projections run
 * on the CTA-pair kernel). */
int ttb_gemm_bf16_out(const void* A_dev, const void* W_dev, const float* bias_dev, void* C_dev, int32_t M, int32_t N, int32_t K,
                      int32_t relu, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TTB200_H */
