// Host side of libttb200: weight store, workspace, forward orchestration and the C ABI
// (include/ttb200.h).  One engine = one model on one GPU; calls on an engine are not re-entrant.
#include "kernels.cuh"
#include "../../include/ttb200.h"

#include <sched.h>
#include <cmath>
#include <cstdlib>
#include <atomic>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

namespace ttb {

static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

void launch_f32_to_bf16(const float* in, __nv_bfloat16* out, long long n, cudaStream_t s);

int ensure_dyn_smem(const void* kernel, int bytes) {
    if (bytes <= 48 * 1024) return 0;
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, int> granted;
    int dev = 0;
    TTB_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    int& have = granted[{dev, kernel}];
    if (bytes <= have) return 0;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) {
        set_last_error(std::string("cudaFuncSetAttribute(MaxDynamicSharedMemorySize, ") + std::to_string(bytes) + ") failed on device " +
                       std::to_string(dev) + ": " + cudaGetErrorString(e));
        return 1;
    }
    have = bytes;
    return 0;
}

static inline void cpu_relax() {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#elif defined(__aarch64__)
    asm volatile("yield" ::: "memory");
#endif
}

// A/B switch: true when the environment variable `name` is set to 1
static bool env_flag(const char* name) { const char* v = getenv(name); return v && v[0] == '1'; }

bool pdl_enabled() { static const bool on = !env_flag("TTB_NO_PDL"); return on; }


struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        TTB_CUDA_OK(cudaMalloc(&p, want));
        cap = want;
        return 0;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Layout of several buffers in one allocation: take() returns the offset of the next 256-byte aligned region
struct Arena {
    size_t bytes = 0;
    size_t take(size_t n) { const size_t o = bytes; bytes += (n + 255) / 256 * 256; return o; }
};

struct Param {
    int64_t numel = 0;
    float* dev = nullptr;
    __nv_bfloat16* devh = nullptr;  // bf16 copy (GEMM weights, precision = bf16)
    bool is_gemm_weight = false;
    bool set = false;
};

struct Lin {
    const float* w = nullptr;
    const float* b = nullptr;
    const __nv_bfloat16* wh = nullptr;
    int N = 0, K = 0;
    Lin rows(int r0, int n) const {
        Lin l = *this;
        l.w = w + (long long)r0 * K;
        l.wh = wh ? wh + (long long)r0 * K : nullptr;
        l.b = b ? b + r0 : nullptr;
        l.N = n;
        return l;
    }
};

struct Norm { const float* g = nullptr; const float* b = nullptr; };

// Kernel classes for the optional per-class CUDA-event timing (ttb_engine_set_profiling).
enum KC : int {
    KC_EMBED = 0, KC_GEMM_QKV, KC_SELF_ATTN, KC_GEMM_SELF_OUT, KC_LAYERNORM, KC_GEMM_CROSS_Q, KC_CROSS_ATTN,
    KC_GEMM_CROSS_OUT, KC_GEMM_FFN1, KC_GEMM_FFN2, KC_GEMM_CLASSIFIER, KC_ARGMAX, KC_ACCEPT, KC_CACHE_APPEND,
    KC_ENCODER, KC_MISC, KC_COUNT
};
static const char* kKcNames[KC_COUNT] = {
    "embed", "gemm_qkv", "self_attn", "gemm_self_out", "add_layernorm", "gemm_cross_q", "cross_attn",
    "gemm_cross_out", "gemm_ffn1", "gemm_ffn2", "gemm_classifier", "argmax", "accept", "cache_append",
    "encoder", "misc"};

struct Prof {
    uint32_t mask = 0;
    std::vector<cudaEvent_t> pool;
    size_t used = 0;
    struct Rec { int kc; size_t e0, e1; };
    std::vector<Rec> recs;
    double ms[KC_COUNT] = {};
    long long n[KC_COUNT] = {};
    int override_kc = -1;  // when >= 0 every launch is attributed to this class (encoder)
    cudaEvent_t get() {
        if (used == pool.size()) {
            cudaEvent_t ev;
            cudaEventCreate(&ev);
            pool.push_back(ev);
        }
        return pool[used++];
    }
};

struct EncLayer { Lin in_proj, out_proj, ff1, ff2; Norm n1, n2; };
struct DecLayer { Lin self_in, self_out, cross_in, cross_out, ff1, ff2; Norm n1, n2, n3; };

}  // namespace ttb

using namespace ttb;

struct ttb_engine {
    ttb_model_desc d{};
    int device = 0;
    bool finalized = false;
    std::map<std::string, Param> params;
    std::vector<EncLayer> enc;
    std::vector<DecLayer> dec;
    Norm enc_norm, dec_norm;
    Lin classifier;
    const float* src_emb = nullptr;
    const float* tgt_emb = nullptr;
    const float* pe = nullptr;

    // forward workspace (typed by the precision's activation type at use)
    DevBuf x, xh, y, qkv, att, q2, hid, logits, tok32, keytok32, pred;
    // encoder products / decoding state
    DevBuf src32, srclen, desc, memory, memh, crosskv, kcache, vcache, kcache2, vcache2, drafts, gen, front, active, ctrl, sel, out64;
    int* h_ctrl = nullptr;  // pinned snapshots of ctrl for lagged polling
    cudaEvent_t poll_ev[4]{};
    cudaEvent_t t0{}, t1{};
    long long launches = 0;
    Prof prof;
    // decoding loop: private stream + one captured CUDA graph per (shape, buffers) configuration
    cudaStream_t stream = nullptr;
    cudaEvent_t join_ev{};
    static constexpr int kBuckets = 10;
    cudaGraphExec_t graph_exec[kBuckets][2] = {};   // greedy iteration graphs per live-query bucket (grids sized for the bucket) x {long, short}
    long long graph_key[17] = {};
    long long graph_launches = 0;
    DevBuf beam;                 // arena of the beam-search state
    DevBuf hist;                 // per-iteration live-query count of the last generate()
    DevBuf cb;                   // continuous batching: slot / batch tables and the staging buffers of an admitted batch
    DevBuf cb_work;              // continuous batching: encoder workspace of an admitted batch (the loop's own must stay intact)
    DevBuf score;                // ttb_score_targets: candidate -> source map and per-row statistics of one chunk
    DevBuf smp;                  // ttb_sample_generate: per-source keys, per-live-row source and cross-attention descriptor
    std::vector<int> h_hist;
    std::vector<int> h_dl, h_dl_min;   // continuous beam-search loop: draft length of every decoder call, smallest of its batches

    int E() const { return d.embedding_dim; }
    int HD() const { return d.embedding_dim / d.num_heads; }

    // Fingerprint of this engine's workspace (address and capacity of every buffer): part of the key of the captured
    // graph, so a buffer that moved invalidates the graph of THIS engine only (several engines decode concurrently from
    // different host threads, translation_transformer_b200/pipeline.py)
    long long alloc_signature() const {
        const DevBuf* bufs[] = {&x, &xh, &y, &qkv, &att, &q2, &hid, &logits, &tok32, &keytok32, &pred, &src32, &srclen, &desc, &memory, &memh,
                                &crosskv, &kcache, &vcache, &kcache2, &vcache2, &drafts, &gen, &front, &active, &ctrl, &sel, &out64, &beam, &hist, &cb, &cb_work, &smp};
        unsigned long long h = 1469598103934665603ull;
        for (const DevBuf* b : bufs) {
            h = (h ^ (unsigned long long)reinterpret_cast<uintptr_t>(b->p)) * 1099511628211ull;
            h = (h ^ (unsigned long long)b->cap) * 1099511628211ull;
        }
        return (long long)(h >> 1);
    }
};

namespace ttb {

static int add_param(ttb_engine* e, const std::string& name, int64_t numel, bool gemm_w) {
    Param p;
    p.numel = numel;
    p.is_gemm_weight = gemm_w;
    TTB_CUDA_OK(cudaMalloc(&p.dev, (size_t)numel * sizeof(float)));
    e->params[name] = p;
    return 0;
}

static int register_params(ttb_engine* e) {
    const ttb_model_desc& d = e->d;
    const int64_t E = d.embedding_dim, F = d.feedforward_dim;
    int rc = 0;
    rc |= add_param(e, "src_token_featurizer.embedding.weight", (int64_t)d.src_vocab_size * E, false);
    rc |= add_param(e, "tgt_token_featurizer.embedding.weight", (int64_t)d.tgt_vocab_size * E, false);
    rc |= add_param(e, "positional_encoding.pe", (int64_t)(d.max_positions + 1) * E, false);
    auto attn = [&](const std::string& p) {
        rc |= add_param(e, p + ".in_proj_weight", 3 * E * E, true);
        rc |= add_param(e, p + ".in_proj_bias", 3 * E, false);
        rc |= add_param(e, p + ".out_proj.weight", E * E, true);
        rc |= add_param(e, p + ".out_proj.bias", E, false);
    };
    auto ffn = [&](const std::string& p, int norms) {
        rc |= add_param(e, p + ".linear1.weight", F * E, true);
        rc |= add_param(e, p + ".linear1.bias", F, false);
        rc |= add_param(e, p + ".linear2.weight", E * F, true);
        rc |= add_param(e, p + ".linear2.bias", E, false);
        for (int j = 1; j <= norms; ++j) {
            rc |= add_param(e, p + ".norm" + std::to_string(j) + ".weight", E, false);
            rc |= add_param(e, p + ".norm" + std::to_string(j) + ".bias", E, false);
        }
    };
    for (int i = 0; i < d.num_encoder_layers; ++i) {
        std::string p = "transformer.encoder.layers." + std::to_string(i);
        attn(p + ".self_attn");
        ffn(p, 2);
    }
    rc |= add_param(e, "transformer.encoder.norm.weight", E, false);
    rc |= add_param(e, "transformer.encoder.norm.bias", E, false);
    for (int i = 0; i < d.num_decoder_layers; ++i) {
        std::string p = "transformer.decoder.layers." + std::to_string(i);
        attn(p + ".self_attn");
        attn(p + ".multihead_attn");
        ffn(p, 3);
    }
    rc |= add_param(e, "transformer.decoder.norm.weight", E, false);
    rc |= add_param(e, "transformer.decoder.norm.bias", E, false);
    rc |= add_param(e, "next_token_classifier.weight", (int64_t)d.tgt_vocab_size * E, true);
    rc |= add_param(e, "next_token_classifier.bias", d.tgt_vocab_size, false);
    return rc;
}

static Lin make_lin(ttb_engine* e, const std::string& w, const std::string& b, int N, int K) {
    Lin l;
    l.w = e->params[w].dev;
    l.wh = e->params[w].devh;
    l.b = e->params[b].dev;
    l.N = N;
    l.K = K;
    return l;
}
static Norm make_norm(ttb_engine* e, const std::string& p) {
    Norm n;
    n.g = e->params[p + ".weight"].dev;
    n.b = e->params[p + ".bias"].dev;
    return n;
}

// RAII scope around one kernel launch: counts it and, when the class is being profiled, brackets it
// with CUDA events on the launching stream.
struct Scope {
    ttb_engine* e;
    cudaStream_t s;
    int kc;
    bool on;
    size_t e0 = 0;
    Scope(ttb_engine* e_, int kc_, cudaStream_t s_) : e(e_), s(s_), kc(e_->prof.override_kc >= 0 ? e_->prof.override_kc : kc_) {
        e->launches++;
        on = (e->prof.mask >> kc) & 1u;
        if (on) {
            e0 = e->prof.used;
            cudaEventRecord(e->prof.get(), s);
        }
    }
    ~Scope() {
        if (on) {
            size_t e1 = e->prof.used;
            cudaEventRecord(e->prof.get(), s);
            e->prof.recs.push_back({kc, e0, e1});
        }
    }
};
static void prof_collect(ttb_engine* e) {  // call after the stream has been synchronised
    for (auto& r : e->prof.recs) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e->prof.pool[r.e0], e->prof.pool[r.e1]) == cudaSuccess) {
            e->prof.ms[r.kc] += ms;
            e->prof.n[r.kc] += 1;
        }
    }
    e->prof.recs.clear();
    e->prof.used = 0;
}

// ---- typed forward helpers ---------------------------------------------------------------------
template <typename ActT> struct Prec;
template <> struct Prec<float> { static constexpr bool lowp = false; };
template <> struct Prec<__nv_bfloat16> { static constexpr bool lowp = true; };

template <typename OutT>
static int linear(ttb_engine* e, int kc, const float* A, int lda, const Lin& L, OutT* C, int ldc, RowCount rows, bool relu, cudaStream_t s) {
    Scope sc(e, kc, s);
    launch_gemm_f32<OutT>(A, lda, L.w, L.b, C, ldc, rows, L.N, L.K, relu, s);
    return 0;
}
template <typename OutT>
static int linear(ttb_engine* e, int kc, const __nv_bfloat16* A, int lda, const Lin& L, OutT* C, int ldc, RowCount rows, bool relu, cudaStream_t s) {
    Scope sc(e, kc, s);
    return launch_gemm_bf16_tc<OutT>(A, lda, L.wh, L.b, C, ldc, rows, L.N, L.K, relu, s);
}

// Sub-layer tail  x <- LN2?(LN1(x + A W^T + b)):  one fused tcgen05 kernel on the bf16 path with E = 256,
// GEMM (fp32 out) + add_layernorm otherwise.  TTB_NO_FUSED_LN=1 forces the unfused kernels (A/B comparisons).
static bool fused_ln_enabled() { static const bool on = !env_flag("TTB_NO_FUSED_LN"); return on; }
static int linear_resid_ln(ttb_engine* e, int kc, const float* A, int lda, const Lin& L, const Norm& n1, const Norm* n2,
                           float* x, float* /*xh*/, float* y, float* dst, float* dsth, RowCount rows, cudaStream_t s,
                           const Lin* = nullptr, float* = nullptr, bool* chained = nullptr) {
    if (chained) *chained = false;
    if (linear<float>(e, kc, A, lda, L, y, L.N, rows, false, s)) return 1;
    Scope sc(e, KC_LAYERNORM, s);
    launch_add_layernorm<float>(x, y, n1.g, n1.b, n2 ? n2->g : nullptr, n2 ? n2->b : nullptr, dst, dsth, rows, L.N, s);
    return 0;
}
// `chain` (optional): a projection of the normalised result that the same kernel computes on the way out
// (the cross-attention query); *chained tells the caller whether it was taken.
static bool chain_enabled() { static const bool on = !env_flag("TTB_NO_CHAIN"); return on; }
static int linear_resid_ln(ttb_engine* e, int kc, const __nv_bfloat16* A, int lda, const Lin& L, const Norm& n1, const Norm* n2,
                           float* x, __nv_bfloat16* xh, float* y, float* dst, __nv_bfloat16* dsth, RowCount rows, cudaStream_t s,
                           const Lin* chain = nullptr, __nv_bfloat16* q2 = nullptr, bool* chained = nullptr) {
    if (chained) *chained = false;
    if (L.N == 256 && dst == x && dsth == xh && fused_ln_enabled()) {
        Scope sc(e, kc, s);
        const bool do_chain = chain && q2 && L.K == 256 && chain->N == 256 && chain->K == 256 && chain_enabled();
        if (chained) *chained = do_chain;
        return launch_gemm_resid_ln(A, lda, L.wh, L.b, x, xh, n1.g, n1.b, n2 ? n2->g : nullptr, n2 ? n2->b : nullptr, rows, L.K, s,
                                    do_chain ? chain->wh : nullptr, do_chain ? chain->b : nullptr, do_chain ? q2 : nullptr);
    }
    if (linear<float>(e, kc, A, lda, L, y, L.N, rows, false, s)) return 1;
    Scope sc(e, KC_LAYERNORM, s);
    launch_add_layernorm<__nv_bfloat16>(x, y, n1.g, n1.b, n2 ? n2->g : nullptr, n2 ? n2->b : nullptr, dst, dsth, rows, L.N, s);
    return 0;
}

// Feed-forward sub-layer  x <- LN2?(LN1(x + relu(x W1^T + b1) W2^T + b2)):  one fused kernel (hidden activations stay
// on the SM) on the bf16 path with E = 256, FFN1 GEMM + (FFN2 GEMM + LN) otherwise.  TTB_NO_FUSED_FFN=1 disables it.
static bool fused_ffn_enabled() { static const bool on = !env_flag("TTB_NO_FUSED_FFN"); return on; }
static int ffn_block(ttb_engine* e, int kc1, int kc2, const Lin& L1, const Lin& L2, const Norm& n1, const Norm* n2, float* x, float* xh,
                     float* hid, float* y, float* dst, float* dsth, RowCount rows, cudaStream_t s) {
    if (linear<float>(e, kc1, x, L1.K, L1, hid, L1.N, rows, true, s)) return 1;
    return linear_resid_ln(e, kc2, hid, L1.N, L2, n1, n2, x, xh, y, dst, dsth, rows, s);
}
static int ffn_block(ttb_engine* e, int kc1, int kc2, const Lin& L1, const Lin& L2, const Norm& n1, const Norm* n2, float* x,
                     __nv_bfloat16* xh, __nv_bfloat16* hid, float* y, float* dst, __nv_bfloat16* dsth, RowCount rows, cudaStream_t s) {
    if (L2.N == 256 && L1.K == 256 && L1.N % 256 == 0 && L1.N <= 4096 && dst == x && dsth == xh && fused_ffn_enabled() && fused_ln_enabled()) {
        Scope sc(e, kc1, s);
        return launch_ffn_fused(xh, L1.wh, L1.b, L2.wh, L2.b, x, n1.g, n1.b, n2 ? n2->g : nullptr, n2 ? n2->b : nullptr, rows, L1.N, s);
    }
    if (linear<__nv_bfloat16>(e, kc1, xh, L1.K, L1, hid, L1.N, rows, true, s)) return 1;
    return linear_resid_ln(e, kc2, hid, L1.N, L2, n1, n2, x, xh, y, dst, dsth, rows, s);
}

// Out-projection + LayerNorm of the preceding sub-layer chained into the fused feed-forward launch (bf16, E = 256, CTA-pair
// kernel available).  Returns 0 when taken, -1 when not applicable (caller launches the two kernels), > 0 on error.
static int ffn_block_chained(ttb_engine*, int, const float*, const Lin&, const Norm&, const Lin&, const Lin&, const Norm&, const Norm*, float*, float*,
                             RowCount, cudaStream_t) {
    return -1;
}
static int ffn_block_chained(ttb_engine* e, int kc, const __nv_bfloat16* att, const Lin& Lo, const Norm& n0, const Lin& L1, const Lin& L2,
                             const Norm& n1, const Norm* n2, float* x, __nv_bfloat16* xh, RowCount rows, cudaStream_t s) {
    if (!(Lo.N == 256 && Lo.K == 256 && L2.N == 256 && L1.K == 256 && L1.N % 256 == 0 && L1.N <= 4096 && fused_ffn_enabled() && fused_ln_enabled() &&
          chain_enabled() && ffn_pair_available(rows.max_rows)))
        return -1;
    static const bool off = env_flag("TTB_NO_FFN_CHAIN");
    if (off) return -1;
    Scope sc(e, kc, s);
    return launch_ffn_fused(xh, L1.wh, L1.b, L2.wh, L2.b, x, n1.g, n1.b, n2 ? n2->g : nullptr, n2 ? n2->b : nullptr, rows, L1.N, s, att, Lo.wh, Lo.b,
                            n0.g, n0.b) ? 1 : 0;
}

// Attention dispatch: fp32 path -> SIMT kernels (exact), bf16 path -> tensor-core kernels
// (TTB_ATTN_SIMT=1 forces the SIMT kernels for A/B comparisons).
static bool attn_simt_forced() { static const bool on = env_flag("TTB_ATTN_SIMT"); return on; }
static void attn(const float* q, int q_ld, const float* k, const float* v, int kv_ld, float* out, int out_ld, int ng, const int* ng_dev,
                 int Lq, int Lk, long long kvs, const int* kvmap, const int* key_tok, int kts, int pad, bool causal, int H, int HD, cudaStream_t s,
                 const int* lk_dev = nullptr, const int* = nullptr, const int4* = nullptr) {
    launch_attention<float>(q, q_ld, k, v, kv_ld, out, out_ld, ng, ng_dev, Lq, Lk, kvs, kvmap, key_tok, kts, pad, causal, H, HD, s, lk_dev);
}
static void attn(const __nv_bfloat16* q, int q_ld, const __nv_bfloat16* k, const __nv_bfloat16* v, int kv_ld, __nv_bfloat16* out, int out_ld,
                 int ng, const int* ng_dev, int Lq, int Lk, long long kvs, const int* kvmap, const int* key_tok, int kts, int pad,
                 bool causal, int H, int HD, cudaStream_t s, const int* lk_dev = nullptr, const int* lk_group = nullptr,
                 const int4* desc = nullptr) {
    if (attn_simt_forced())
        launch_attention<__nv_bfloat16>(q, q_ld, k, v, kv_ld, out, out_ld, ng, ng_dev, Lq, Lk, kvs, kvmap, key_tok, kts, pad, causal, H, HD, s, lk_dev);
    else
        launch_attention_mma(q, q_ld, k, v, kv_ld, out, out_ld, ng, ng_dev, Lq, Lk, kvs, kvmap, key_tok, kts, pad, causal, H, HD, s, lk_dev, lk_group, desc);
}
static void spec_attn(const float* qkv, int ld, const float* kc, const float* vc, long long cqs, int cld, float* out, int old, int B,
                      const int* na, const int* active, const int* front, const int* gen, int gen_ld, int pad, int N, int D, int H,
                      int HD, int P, cudaStream_t s, const int4* = nullptr, bool = false) {
    launch_spec_self_attention<float>(qkv, ld, kc, vc, cqs, cld, out, old, B, na, active, front, gen, gen_ld, pad, N, D, H, HD, P, s);
}
static void spec_attn(const __nv_bfloat16* qkv, int ld, const __nv_bfloat16* kc, const __nv_bfloat16* vc, long long cqs, int cld,
                      __nv_bfloat16* out, int old, int B, const int* na, const int* active, const int* front, const int* gen,
                      int gen_ld, int pad, int N, int D, int H, int HD, int P, cudaStream_t s, const int4* desc = nullptr, bool group_row_len = false) {
    if (attn_simt_forced())
        launch_spec_self_attention<__nv_bfloat16>(qkv, ld, kc, vc, cqs, cld, out, old, B, na, active, front, gen, gen_ld, pad, N, D, H, HD, P, s);
    else
        launch_spec_self_attention_mma(qkv, ld, kc, vc, cqs, cld, out, old, B, na, active, front, gen, gen_ld, pad, N, D, H, HD, s, desc, group_row_len);
}

// GEMM A-operand view of the residual stream: fp32 path reads x itself, bf16 path its bf16 copy
template <typename ActT> static const ActT* a_view(const float* x, const ActT* xh);
template <> const float* a_view<float>(const float* x, const float*) { return x; }
template <> const __nv_bfloat16* a_view<__nv_bfloat16>(const float*, const __nv_bfloat16* xh) { return xh; }

template <typename ActT>
static int ensure_work(ttb_engine* e, long long T, int qkv_layers) {
    const long long E = e->E(), F = e->d.feedforward_dim, V = e->d.tgt_vocab_size;
    int rc = 0;
    rc |= e->x.ensure(T * E * sizeof(float));
    if (Prec<ActT>::lowp) rc |= e->xh.ensure(T * E * sizeof(ActT));
    rc |= e->y.ensure(T * E * sizeof(float));
    rc |= e->qkv.ensure(T * 3 * E * sizeof(ActT) * qkv_layers);
    rc |= e->att.ensure(T * E * sizeof(ActT));
    rc |= e->q2.ensure(T * E * sizeof(ActT));
    rc |= e->hid.ensure(T * F * sizeof(ActT));
    rc |= e->logits.ensure(T * V * sizeof(float));
    rc |= e->tok32.ensure(T * sizeof(int));
    rc |= e->pred.ensure(T * sizeof(int));
    return rc;
}

// Workspace of the encoder stack (rows = tokens): the engine's forward workspace unless the caller brings its own.
template <typename ActT> struct EncWork { float* x; ActT* xh; float* y; ActT* qkv; ActT* att; ActT* hid; };
template <typename ActT>
static size_t enc_work_bytes(const ttb_engine* e, long long T) {
    const long long E = e->E(), F = e->d.feedforward_dim;
    const long long elems[6] = {T * E * 4, Prec<ActT>::lowp ? T * E * (long long)sizeof(ActT) : 0, T * E * 4, T * 3 * E * (long long)sizeof(ActT),
                                T * E * (long long)sizeof(ActT), T * F * (long long)sizeof(ActT)};
    Arena a;
    for (long long b : elems) a.take((size_t)b);
    return a.bytes;
}
template <typename ActT>
static EncWork<ActT> enc_work_carve(const ttb_engine* e, long long T, void* base) {
    const long long E = e->E(), F = e->d.feedforward_dim;
    Arena a;
    auto take = [&](long long bytes) { return static_cast<char*>(base) + a.take((size_t)bytes); };
    EncWork<ActT> w;
    w.x = reinterpret_cast<float*>(take(T * E * 4));
    w.xh = Prec<ActT>::lowp ? reinterpret_cast<ActT*>(take(T * E * sizeof(ActT))) : nullptr;
    w.y = reinterpret_cast<float*>(take(T * E * 4));
    w.qkv = reinterpret_cast<ActT*>(take(T * 3 * E * sizeof(ActT)));
    w.att = reinterpret_cast<ActT*>(take(T * E * sizeof(ActT)));
    w.hid = reinterpret_cast<ActT*>(take(T * F * sizeof(ActT)));
    return w;
}

// Encoder stack on tokens src32 (B, Ls); writes memory (fp32) and, on the bf16 path, memh.
template <typename ActT>
static int encode_impl(ttb_engine* e, const int* src32, const int* key_tok, int B, int Ls, float* mem_out, ActT* memh_out, cudaStream_t s,
                       const EncWork<ActT>* work = nullptr) {
    const int E = e->E(), T = B * Ls, H = e->d.num_heads, HD = e->HD();
    if (!work && ensure_work<ActT>(e, T, 1)) return 1;
    float* x = work ? work->x : e->x.as<float>();
    ActT* xh = work ? work->xh : (Prec<ActT>::lowp ? e->xh.as<ActT>() : nullptr);
    float* y = work ? work->y : e->y.as<float>();
    ActT* qkv = work ? work->qkv : e->qkv.as<ActT>();
    ActT* att = work ? work->att : e->att.as<ActT>();
    ActT* hid = work ? work->hid : e->hid.as<ActT>();
    RowCount rows(T);
    e->prof.override_kc = KC_ENCODER;
    struct Reset { ttb_engine* e; ~Reset() { e->prof.override_kc = -1; } } reset{e};
    { Scope sc(e, KC_ENCODER, s); launch_embed_seq<ActT>(src32, T, Ls, e->src_emb, e->pe, E, x, xh, s); }
    const int n_layers = (int)e->enc.size();
    for (int l = 0; l < n_layers; ++l) {
        const EncLayer& L = e->enc[l];
        const bool last = l + 1 == n_layers;
        if (linear<ActT>(e, KC_ENCODER, a_view<ActT>(x, xh), E, L.in_proj, qkv, 3 * E, rows, false, s)) return 1;
        {
            Scope sc(e, KC_ENCODER, s);
            attn(qkv, 3 * E, qkv + E, qkv + 2 * E, 3 * E, att, E, B, nullptr, Ls, Ls, Ls, nullptr,
                                   key_tok, Ls, e->d.src_pad_token_idx, false, H, HD, s);
        }
        if (linear_resid_ln(e, KC_ENCODER, att, E, L.out_proj, L.n1, nullptr, x, xh, y, x, xh, rows, s)) return 1;
        float* dst = last ? mem_out : x;
        ActT* dsth = last ? memh_out : xh;
        if (ffn_block(e, KC_ENCODER, KC_ENCODER, L.ff1, L.ff2, L.n2, last ? &e->enc_norm : nullptr, x, xh, hid, y, dst, dsth, rows, s)) return 1;
    }
    return 0;
}

// Cross-attention K/V of every decoder layer from the encoder memory: crosskv[l] = (B*Ls, 2E)
template <typename ActT>
static int cross_kv_impl(ttb_engine* e, const float* mem, const ActT* memh, int rows_n, ActT* crosskv, cudaStream_t s,
                         long long layer_stride = 0) {
    const int E = e->E();
    RowCount rows(rows_n);
    if (layer_stride == 0) layer_stride = (long long)rows_n * 2 * E;
    for (size_t l = 0; l < e->dec.size(); ++l) {
        Lin kv = e->dec[l].cross_in.rows(E, 2 * E);
        if (linear<ActT>(e, KC_ENCODER, a_view<ActT>(mem, memh), E, kv, crosskv + (long long)l * layer_stride, 2 * E, rows, false, s)) return 1;
    }
    return 0;
}

// Decoder layers on the token matrix in e->x / e->xh (`rows` live rows).  `self_attn` / `cross_attn`
// enqueue the layer's attention kernels given the freshly projected q/k/v of that layer.
template <typename ActT, typename SelfAttn, typename CrossAttn>
static int decoder_stack(ttb_engine* e, RowCount rows, int qkv_layers, long long qkv_layer_stride,
                         SelfAttn self_attn, CrossAttn cross_attn, cudaStream_t s) {
    const int E = e->E();
    float* x = e->x.as<float>();
    ActT* xh = Prec<ActT>::lowp ? e->xh.as<ActT>() : nullptr;
    float* y = e->y.as<float>();
    ActT* att = e->att.as<ActT>();
    ActT* q2 = e->q2.as<ActT>();
    ActT* hid = e->hid.as<ActT>();
    const int n_layers = (int)e->dec.size();
    for (int l = 0; l < n_layers; ++l) {
        const DecLayer& L = e->dec[l];
        const bool last = l + 1 == n_layers;
        ActT* qkv = e->qkv.as<ActT>() + (qkv_layers > 1 ? (long long)l * qkv_layer_stride : 0);
        if (linear<ActT>(e, KC_GEMM_QKV, a_view<ActT>(x, xh), E, L.self_in, qkv, 3 * E, rows, false, s)) return 1;
        { Scope sc(e, KC_SELF_ATTN, s); self_attn(l, qkv, att); }
        const Lin cross_q = L.cross_in.rows(0, E);
        bool chained = false;
        if (linear_resid_ln(e, KC_GEMM_SELF_OUT, att, E, L.self_out, L.n1, nullptr, x, xh, y, x, xh, rows, s, &cross_q, q2, &chained)) return 1;
        if (!chained && linear<ActT>(e, KC_GEMM_CROSS_Q, a_view<ActT>(x, xh), E, cross_q, q2, E, rows, false, s)) return 1;
        { Scope sc(e, KC_CROSS_ATTN, s); cross_attn(l, q2, att); }
        // cross-attention out-projection + LayerNorm2 + feed-forward block + LayerNorm3 in one launch where the CTA-pair
        // feed-forward kernel runs, two launches otherwise
        int fused = ffn_block_chained(e, KC_GEMM_FFN1, att, L.cross_out, L.n2, L.ff1, L.ff2, L.n3, last ? &e->dec_norm : nullptr, x, xh, rows, s);
        if (fused > 0) return 1;
        if (fused == 0) continue;
        if (linear_resid_ln(e, KC_GEMM_CROSS_OUT, att, E, L.cross_out, L.n2, nullptr, x, xh, y, x, xh, rows, s)) return 1;
        if (ffn_block(e, KC_GEMM_FFN1, KC_GEMM_FFN2, L.ff1, L.ff2, L.n3, last ? &e->dec_norm : nullptr, x, xh, hid, y, x, xh, rows, s)) return 1;
    }
    return 0;
}

template <typename ActT>
static int encode_api(ttb_engine* e, const int64_t* src_dev, const uint8_t* mask_dev, int B, int Ls, float* mem_out, cudaStream_t s) {
    const long long T = (long long)B * Ls;
    if (e->src32.ensure(T * sizeof(int))) return 1;
    int* src32 = e->src32.as<int>();
    { Scope sc(e, KC_MISC, s); launch_i64_to_i32(reinterpret_cast<const long long*>(src_dev), src32, T, s); }
    const int* key_src = src32;
    if (mask_dev) {  // explicit mask: express it as a token-like array for the attention kernels
        if (e->keytok32.ensure(T * sizeof(int))) return 1;
        Scope sc(e, KC_MISC, s);
        launch_mask_to_tokens(mask_dev, e->keytok32.as<int>(), T, e->d.src_pad_token_idx, s);
        key_src = e->keytok32.as<int>();
    }
    if (Prec<ActT>::lowp && e->memh.ensure(T * e->E() * sizeof(ActT))) return 1;
    int rc = encode_impl<ActT>(e, src32, key_src, B, Ls, mem_out, Prec<ActT>::lowp ? e->memh.as<ActT>() : nullptr, s);
    if (rc) return rc;
    TTB_CUDA_OK(cudaGetLastError());
    return 0;
}

template <typename ActT>
static int decode_api(ttb_engine* e, const int64_t* tgt_dev, int B, int Lt, const float* memory_dev,
                      const uint8_t* mem_mask_dev, int Ls, float* logits_out, cudaStream_t s) {
    const int E = e->E(), H = e->d.num_heads, HD = e->HD(), V = e->d.tgt_vocab_size;
    const long long T = (long long)B * Lt, TS = (long long)B * Ls;
    if (ensure_work<ActT>(e, T, 1)) return 1;
    if (e->keytok32.ensure(TS * sizeof(int))) return 1;
    if (e->crosskv.ensure(TS * 2 * E * sizeof(ActT) * e->dec.size())) return 1;
    int* tgt32 = e->tok32.as<int>();
    int* memtok = e->keytok32.as<int>();
    { Scope sc(e, KC_MISC, s); launch_i64_to_i32(reinterpret_cast<const long long*>(tgt_dev), tgt32, T, s); }
    { Scope sc(e, KC_MISC, s); launch_mask_to_tokens(mem_mask_dev, memtok, TS, e->d.src_pad_token_idx, s); }
    const ActT* memh = nullptr;
    if (Prec<ActT>::lowp) {
        if (e->memh.ensure(TS * E * sizeof(ActT))) return 1;
        Scope sc(e, KC_MISC, s);
        launch_f32_to_bf16(memory_dev, reinterpret_cast<__nv_bfloat16*>(e->memh.p), TS * E, s);
        memh = e->memh.as<ActT>();
    }
    ActT* crosskv = e->crosskv.as<ActT>();
    if (cross_kv_impl<ActT>(e, memory_dev, memh, (int)TS, crosskv, s)) return 1;
    float* x = e->x.as<float>();
    ActT* xh = Prec<ActT>::lowp ? e->xh.as<ActT>() : nullptr;
    { Scope sc(e, KC_EMBED, s); launch_embed_seq<ActT>(tgt32, (int)T, Lt, e->tgt_emb, e->pe, E, x, xh, s); }
    RowCount rows((int)T);
    auto self_attn = [&](int, ActT* qkv, ActT* att) {
        attn(qkv, 3 * E, qkv + E, qkv + 2 * E, 3 * E, att, E, B, nullptr, Lt, Lt, Lt, nullptr,
                               tgt32, Lt, e->d.tgt_pad_token_idx, true, H, HD, s);
    };
    auto cross_attn = [&](int l, ActT* q2, ActT* att) {
        const ActT* kv = crosskv + (long long)l * TS * 2 * E;
        attn(q2, E, kv, kv + E, 2 * E, att, E, B, nullptr, Lt, Ls, Ls, nullptr,
                               memtok, Ls, e->d.src_pad_token_idx, false, H, HD, s);
    };
    if (decoder_stack<ActT>(e, rows, 1, 0, self_attn, cross_attn, s)) return 1;
    if (linear<float>(e, KC_GEMM_CLASSIFIER, a_view<ActT>(x, xh), E, e->classifier, logits_out, V, rows, false, s)) return 1;
    TTB_CUDA_OK(cudaGetLastError());
    return 0;
}

// Encoder and cross-attention K/V of one batch of (B, Ls) int64 sources: tokens into e->src32, per-query source lengths
// into `srclen` (the cross-attention kernels skip the padding behind them), the K/V of decoder layer l at
// kv + l * kv_layer_stride.  `work`: the encoder's workspace, nullptr for the engine's forward workspace.
template <typename ActT>
static int encode_batch(ttb_engine* e, const int64_t* src, int B, int Ls, int* srclen, ActT* kv, long long kv_layer_stride, cudaStream_t s,
                        const EncWork<ActT>* work = nullptr) {
    const long long TS = (long long)B * Ls;
    int* src32 = e->src32.as<int>();
    float* mem = e->memory.as<float>();
    ActT* memh = Prec<ActT>::lowp ? e->memh.as<ActT>() : nullptr;
    { Scope sc(e, KC_MISC, s); launch_i64_to_i32(reinterpret_cast<const long long*>(src), src32, TS, s); }
    { Scope sc(e, KC_MISC, s); launch_row_lengths(src32, B, Ls, e->d.src_pad_token_idx, srclen, s); }
    if (encode_impl<ActT>(e, src32, src32, B, Ls, mem, memh, s, work)) return 1;
    return cross_kv_impl<ActT>(e, mem, memh, (int)TS, kv, s, kv_layer_stride);
}

// Buffers of a decoding loop that depend on the source length are sized for a rounded-up capacity: batches of different
// length must not reallocate (cudaFree synchronises the whole device, i.e. every other engine decoding on this GPU as well)
// nor invalidate the captured graph.
static int ls_capacity(int Ls) { return std::max(256, (Ls + 63) / 64 * 64); }

// Buffers of encode_batch: the encoder products of TS_enc source tokens, source lengths of B queries, and the
// cross-attention K/V of TS_kv source tokens in every decoder layer.
template <typename ActT>
static int ensure_encoder(ttb_engine* e, long long TS_enc, int B, long long TS_kv) {
    const int E = e->E();
    if (e->src32.ensure(TS_enc * sizeof(int)) || e->memory.ensure(TS_enc * E * sizeof(float)) || e->srclen.ensure((size_t)B * sizeof(int))) return 1;
    if (Prec<ActT>::lowp && e->memh.ensure(TS_enc * E * sizeof(ActT))) return 1;
    return e->crosskv.ensure(TS_kv * 2 * E * sizeof(ActT) * e->dec.size());
}

// Vocabulary projection of the decoder rows and the per-row reduction a loop reads.  bf16 path with `use_fused`:
// fused_launch(xh), a tcgen05 kernel that keeps the logits in tensor memory (0 taken, < 0 refused, > 0 error).  Otherwise,
// or when it refuses, the logits GEMM into `logits` and fallback(logits).
template <typename ActT, typename Fused, typename Fallback>
static int classifier_head(ttb_engine* e, RowCount rows, bool use_fused, Fused fused_launch, Fallback fallback, float* logits, cudaStream_t s) {
    if constexpr (Prec<ActT>::lowp) {
        if (use_fused) {
            Scope sc(e, KC_GEMM_CLASSIFIER, s);
            const int rc = fused_launch(e->xh.as<ActT>());
            if (rc >= 0) return rc > 0 ? 1 : 0;
            e->launches--;   // refused: nothing was launched
        }
    }
    const ActT* a = a_view<ActT>(e->x.as<float>(), Prec<ActT>::lowp ? e->xh.as<ActT>() : nullptr);
    if (linear<float>(e, KC_GEMM_CLASSIFIER, a, e->E(), e->classifier, logits, e->d.tgt_vocab_size, rows, false, s)) return 1;
    Scope sc(e, KC_ARGMAX, s);
    fallback(logits);
    return 0;
}

// The decoding loops run on the engine's own stream (graph capture is not allowed on the legacy default stream), ordered
// after the caller's stream and drained before they return.
static int join_caller_stream(ttb_engine* e, cudaStream_t user_stream) {
    TTB_CUDA_OK(cudaEventRecord(e->join_ev, user_stream));
    TTB_CUDA_OK(cudaStreamWaitEvent(e->stream, e->join_ev, 0));
    return 0;
}
// End of a decoding loop: drains the engine's stream and collects the kernel-class timings; ms = time since e->t0.
static int finish_loop(ttb_engine* e, float& ms) {
    TTB_CUDA_OK(cudaEventRecord(e->t1, e->stream));
    TTB_CUDA_OK(cudaStreamSynchronize(e->stream));
    TTB_CUDA_OK(cudaGetLastError());
    prof_collect(e);
    ms = 0.f;
    cudaEventElapsedTime(&ms, e->t0, e->t1);
    return 0;
}

// ---- continuous batching, common to the three loops (DESIGN.md section 10) --------------------------------------------
// The batches that share the query slots of one loop (ttb_*_generate_batches).
struct BatchList {
    int n;                              // batches, admitted in list order
    const int64_t* const* src;          // [n] (B_i, Ls_i) int64 sources
    const int32_t* bs;                  // [n] B_i
    const int32_t* ls;                  // [n] Ls_i
    int64_t* const* out;                // [n] outputs, laid out as the loop's generate() writes them
    ttb_generate_stats* stats;          // [n]
    int32_t* out_width;                 // [n] width of each batch's hypotheses (beam searches), or NULL
    int32_t* const* trace;              // [n] optional greedy traces, or NULL
    int32_t* const* trace_nacc;         // [n] optional speculative beam-search traces, or NULL
    int32_t* const* trace_pick;
};

// Slot tables of a continuous loop and staging of the batch being admitted, in e->cb; the admitted batch's encoder
// workspace in e->cb_work (never the loop's x / qkv: the next iteration's first kernel still reads qkv).  Admission of
// batch i: encode(i), the loop's own staging and admission kernel (which takes the free slots), then scatter(i).
template <typename ActT>
struct Staging {
    const BatchList* cb;
    int B_stage = 0;             // largest batch; the encoder of an admitted batch runs on the largest batch shape
    long long TS_stage = 0;
    int slots = 0, Ls_cap = 0;
    int* srclen = nullptr;       // [B_stage] source lengths of the batch being admitted
    ActT* kv = nullptr;          // [layers][TS_stage][2E] its cross-attention K/V
    EncWork<ActT> work{};
    long long sig0 = 0;          // e->alloc_signature() once the loop is sized: nothing is allocated after it

    explicit Staging(const BatchList* cb_) : cb(cb_) {
        for (int i = 0; cb && i < cb->n; ++i) {
            B_stage = std::max(B_stage, (int)cb->bs[i]);
            TS_stage = std::max(TS_stage, (long long)cb->bs[i] * cb->ls[i]);
        }
    }
    // Sizes and carves e->cb for B slots: the slot tables and t.groups first, at offsets that depend on the slot count only
    // (the greedy loop's captured graphs bake them; the slot count is part of the graph key), then the common staging and
    // the loop's `extra` regions {&pointer, bytes}.  Also sizes cb_work and the slot-major key tokens.
    template <typename Table>
    int alloc(ttb_engine* e, Table& t, int B, int Ls_cap_, std::initializer_list<std::pair<int**, size_t>> extra) {
        using G = std::remove_pointer_t<decltype(t.groups)>;
        const int E = e->E();
        TTB_CHECK((2 * E * sizeof(ActT)) % 16 == 0, "continuous batching needs 16-byte cross-attention K/V rows");
        slots = B;
        Ls_cap = Ls_cap_;
        Arena a;
        const size_t o_sg = a.take((size_t)B * 4), o_sq = a.take((size_t)B * 4), o_as = a.take((size_t)B * 4), o_gr = a.take((size_t)cb->n * sizeof(G));
        const size_t o_sl = a.take((size_t)B_stage * 4), o_kv = a.take(e->dec.size() * TS_stage * 2 * E * sizeof(ActT));
        std::vector<size_t> o_extra;
        for (const auto& x : extra) o_extra.push_back(a.take(x.second));
        if (e->cb.ensure(a.bytes) || e->cb_work.ensure(enc_work_bytes<ActT>(e, TS_stage)) || e->keytok32.ensure((size_t)B * Ls_cap * sizeof(int))) return 1;
        char* base = e->cb.as<char>();
        t.slots = SlotTable{(int*)(base + o_sg), (int*)(base + o_sq), (int*)(base + o_as)};
        t.groups = (G*)(base + o_gr);
        srclen = (int*)(base + o_sl);
        kv = (ActT*)(base + o_kv);
        size_t k = 0;
        for (const auto& x : extra) *x.first = (int*)(base + o_extra[k++]);
        work = enc_work_carve<ActT>(e, TS_stage, e->cb_work.p);
        return 0;
    }
    // encoder, source lengths and cross K/V of batch i, for the batch alone; its int32 tokens stay in e->src32
    int encode(ttb_engine* e, int i, cudaStream_t s) {
        return encode_batch<ActT>(e, cb->src[i], cb->bs[i], cb->ls[i], srclen, kv, TS_stage * 2 * e->E(), s, &work);
    }
    // after the admission kernel: the staged K/V and key tokens of batch i -> its slots (slot-major, Ls_cap rows per slot)
    int scatter(ttb_engine* e, const SlotTable& t, int i, cudaStream_t s) {
        const int E = e->E();
        {
            Scope sc(e, KC_MISC, s);
            launch_admit_kv<ActT>(t.adm_slots, cb->bs[i], cb->ls[i], Ls_cap, (int)e->dec.size(), E, kv, TS_stage * 2 * E, e->crosskv.as<ActT>(),
                                  (long long)slots * Ls_cap * 2 * E, e->src32.as<int>(), e->keytok32.as<int>(), e->d.src_pad_token_idx, s);
        }
        TTB_CUDA_OK(cudaGetLastError());
        TTB_CHECK(e->alloc_signature() == sig0, "a workspace buffer moved while a continuous decoding loop was running");
        return 0;
    }
    // Admits the next batches, whole and in list order, while `free_slots` suffice; admit(i) is the loop's admission of
    // batch i.  Adds the queries admitted to *n_admitted.
    int next = 0;
    template <typename Admit>
    int admit_fitting(int free_slots, int* n_admitted, Admit admit) {
        while (next < cb->n && free_slots - *n_admitted >= cb->bs[next]) {
            if (int rc = admit(next)) return rc;
            *n_admitted += cb->bs[next++];
        }
        return 0;
    }
};

// Per-batch records of a continuous loop that has drained: every batch must have been admitted whole and closed.
template <typename G>
static int read_groups(const BatchList* cb, const G* dev, std::vector<G>& groups) {
    groups.resize((size_t)cb->n);
    TTB_CUDA_OK(cudaMemcpy(groups.data(), dev, groups.size() * sizeof(G), cudaMemcpyDeviceToHost));
    for (int i = 0; i < cb->n; ++i)
        TTB_CHECK(groups[(size_t)i].closed == 1 && groups[(size_t)i].B == cb->bs[i], "continuous decoding loop ended before every batch was finished");
    return 0;
}

// Sampling decoding (ttb_sample_generate, DESIGN.md section 15): S sample slots per source, drawn with temperature T from
// the top_k largest logits (0: all) under the per-source keys of `seed`.  The defaults stand for one slot per query.
struct SampleCfg {
    int S = 1;
    float temperature = 1.f;
    int top_k = 0;
    unsigned long long seed = 0;
};

// The decodings greedy_api runs: speculative greedy decoding; the standard greedy decoding, the same KV-cached loop with one
// row per query and no draft tokens (standard_decoding.py); sampling, the standard loop with a draw in place of the arg-max.
enum class GreedyMode : int { speculative = 0, standard = 1, sampling = 2 };

// With `cb` the loop is the continuous one: B is the number of query slots, Ls the longest source of all batches, and the
// batches of `cb` are admitted into free slots between two graph launches.  Sampling: B is the number of sample slots
// (sources x smp.S), slot b * S + s is sample s of source b.
template <typename ActT>
static int greedy_api(ttb_engine* e, const int64_t* src_dev, int B, int Ls, int max_len, int draft_len, int N,
                      int pad, int bos, int eos, int replace, int tie_break, int64_t* out_dev, int32_t* trace_dev,
                      ttb_generate_stats* stats, cudaStream_t user_stream, GreedyMode mode, const BatchList* cb = nullptr,
                      const SampleCfg& smp = SampleCfg{}) {
    const int E = e->E(), H = e->d.num_heads, HD = e->HD(), V = e->d.tgt_vocab_size;
    const int n_dec = (int)e->dec.size();
    cudaStream_t s = e->stream;
    if (int rc = join_caller_stream(e, user_stream)) return rc;
    const bool standard = mode != GreedyMode::speculative, sampling = mode == GreedyMode::sampling;
    // speculative: make_drafts(min_draft_len=1, max_draft_len=max_len)
    const int D = standard ? 0 : std::min(std::max(1, draft_len), max_len);
    if (standard) N = 1;
    const int Ls_cap = ls_capacity(Ls);
    // sampling: the encoder and the cross-attention K/V run once per source, shared by its S slots
    const int S = smp.S, B_src = B / S;
    const long long TS_cap = (long long)B_src * Ls_cap;
    const int per_q = N * (D + 1);
    const long long T = (long long)B * per_q;
    const int gen_ld = max_len + D + 2;
    const int P = gen_ld;  // cache positions per query
    const long long launches0 = e->launches;
    const bool cont = cb != nullptr;
    // continuous loop: every batch takes part in at most max_len + 1 iterations; the host stays at most (LAG + 1) graph
    // launches ahead of the control words it reads, i.e. a few no-op iterations per admission
    const long long max_iters = cont ? (long long)cb->n * (max_len + 1) + (long long)(cb->n + 1) * 3 * 16 : max_len + 1;
    Staging<ActT> sg(cb);

    // encoder + cross-attention K/V (computed once per query, not once per draft row and iteration)
    if (ensure_encoder<ActT>(e, cont ? sg.TS_stage : TS_cap, B, TS_cap)) return 1;
    const size_t cache_bytes = (size_t)n_dec * B * P * E * sizeof(ActT);
    if (e->kcache.ensure(cache_bytes) || e->vcache.ensure(cache_bytes)) return 1;
    if (e->drafts.ensure((size_t)B * N * D * sizeof(int)) || e->gen.ensure((size_t)B * gen_ld * sizeof(int))) return 1;
    if (e->front.ensure(B * sizeof(int)) || e->active.ensure(B * sizeof(int)) || e->ctrl.ensure(CTRL_COUNT * sizeof(int))) return 1;
    if (e->sel.ensure((size_t)B * 4 * sizeof(int)) || e->out64.ensure((size_t)B * max_len * sizeof(long long))) return 1;
    if (e->desc.ensure((size_t)B * sizeof(int4))) return 1;
    if (e->hist.ensure((size_t)(max_iters + 1) * sizeof(int))) return 1;
    if (ensure_work<ActT>(e, cont ? T : std::max(T, TS_cap), n_dec)) return 1;
    SampleLoop sl{S, nullptr, nullptr};
    unsigned long long* smp_keys = nullptr;
    if (sampling) {
        if (e->smp.ensure((size_t)B_src * 8 + (size_t)B * 20 + 256)) return 1;
        smp_keys = e->smp.as<unsigned long long>();
        sl.xdesc = reinterpret_cast<int4*>(e->smp.as<char>() + ((size_t)B_src * 8 + 15) / 16 * 16);
        sl.kvsrc = reinterpret_cast<int*>(sl.xdesc + B);
    }
    // the fused / fallback classifier (arg-max or draw) is chosen per call and is part of the graph key, so that one process
    // can compare both
    const bool use_fused = Prec<ActT>::lowp && !env_flag("TTB_NO_FUSED_ARGMAX");
    // continuous loop: slot / batch tables, staging of an admitted batch (drafts as well)
    CbTable cbt{};
    int* stage_drafts = nullptr;
    if (cont) {
        TTB_CHECK(B <= 2048, "continuous batching supports at most 2048 slots");
        if (int rc = sg.alloc(e, cbt, B, Ls_cap, {{&stage_drafts, (size_t)sg.B_stage * N * D * sizeof(int)}})) return rc;
    }
    // nothing is allocated from here on: the captured graphs bake these addresses
    sg.sig0 = e->alloc_signature();

    TTB_CUDA_OK(cudaEventRecord(e->t0, s));
    int* src32 = e->src32.as<int>();
    ActT* crosskv = e->crosskv.as<ActT>();
    GreedyState st{};
    st.B = B; st.N = N; st.D = D; st.max_len = max_len; st.gen_ld = gen_ld; st.pad = pad; st.bos = bos; st.eos = eos; st.Ls = Ls;
    st.gen = e->gen.as<int>(); st.front = e->front.as<int>(); st.active = e->active.as<int>(); st.ctrl = e->ctrl.as<int>();
    st.drafts = e->drafts.as<int>(); st.pred = e->pred.as<int>(); st.out = cont ? nullptr : e->out64.as<long long>();
    st.sel = e->sel.as<int>(); st.trace = cont ? nullptr : trace_dev; st.tie_break = tie_break; st.hist = e->hist.as<int>();
    st.desc = e->desc.as<int4>(); st.src_len = e->srclen.as<int>();
    // admission of batch i (continuous loop): encoder, cross K/V and drafts of the batch alone, as below for one batch,
    // then the kernels that move it into free slots
    auto admit = [&](int i) -> int {
        const int Bi = cb->bs[i], Li = cb->ls[i];
        if (int rc = sg.encode(e, i, s)) return rc;
        if (!standard) { Scope sc(e, KC_MISC, s); launch_make_drafts(src32 + 1, Li, Bi, Li - 1, D, N, eos, pad, replace, stage_drafts, s); }
        {
            Scope sc(e, KC_MISC, s);
            if (int rc = launch_greedy_admit(st, cbt, i, Bi, stage_drafts, sg.srclen, reinterpret_cast<long long*>(cb->out[i]),
                                             cb->trace ? cb->trace[i] : nullptr, Ls_cap, s))
                return rc;
        }
        return sg.scatter(e, cbt.slots, i, s);
    };
    if (cont) {
        TTB_CUDA_OK(cudaMemsetAsync(st.ctrl, 0, CTRL_COUNT * sizeof(int), s));
    } else {
        if (encode_batch<ActT>(e, src_dev, B_src, Ls, e->srclen.as<int>(), crosskv, TS_cap * 2 * E, s)) return 1;
        // drafts from the source without its BOS column (speculative_decoding.py:64-73)
        if (!standard) { Scope sc(e, KC_MISC, s); launch_make_drafts(src32 + 1, Ls, B, Ls - 1, D, N, eos, pad, replace, e->drafts.as<int>(), s); }
        if (sampling) {
            { Scope sc(e, KC_MISC, s); launch_sample_keys(src32, B_src, Ls, e->d.src_pad_token_idx, smp.seed, smp_keys, s); }
            { Scope sc(e, KC_MISC, s); launch_sample_init(st, sl, s); }
        } else {
            Scope sc(e, KC_MISC, s);
            launch_greedy_init(st, s);
        }
    }

    float* x = e->x.as<float>();
    ActT* xh = Prec<ActT>::lowp ? e->xh.as<ActT>() : nullptr;
    ActT* kc = e->kcache.as<ActT>();
    ActT* vc = e->vcache.as<ActT>();
    const long long cache_q_stride = (long long)P * E, cache_l_stride = (long long)B * P * E;
    const long long qkv_l_stride = T * 3 * E;
    const int* n_active = st.ctrl + CTRL_N_ACTIVE;
    // Grids of an iteration are sized for `Bq` queries: the whole batch, or -- once the host has seen queries retire -- one of
    // a few smaller buckets (live-query count only shrinks, so the count the host read last is an upper bound for every
    // iteration it launches afterwards).  CTAs beyond the live range exit at once either way, but each of them still has to
    // find an SM with ~200 KB of shared memory free just to do so, which serialises the kernels of the OTHER batches in
    // flight behind it; with batches that thin out (trained-like weights) most CTAs of a full-size grid are such no-ops.
    int Bq = B;

    auto self_attn = [&](int l, ActT* qkv, ActT* att) {
        spec_attn(qkv, 3 * E, kc + l * cache_l_stride, vc + l * cache_l_stride, cache_q_stride, E,
                                         att, E, Bq, n_active, st.active, st.front, st.gen, gen_ld, e->d.tgt_pad_token_idx,
                                         N, D, H, HD, P, s, st.desc);
    };
    // cross-attention K/V rows and key tokens: per query, for sampling those of the slot's source (generate()), or slot-major
    // with Ls_cap (= CTRL_LS) rows per slot (continuous loop)
    const int kv_ls = cont ? Ls_cap : Ls;
    const int* kv_map = sampling ? sl.kvsrc : st.active;
    const int* key_tok = cont ? e->keytok32.as<int>() : src32;
    const int4* cross_desc = sampling ? sl.xdesc : st.desc;
    auto cross_attn = [&](int l, ActT* q2, ActT* att) {
        const ActT* kv = crosskv + (long long)l * TS_cap * 2 * E;
        attn(q2, E, kv, kv + E, 2 * E, att, E, Bq, n_active, per_q, kv_ls, kv_ls, kv_map, key_tok, kv_ls, e->d.src_pad_token_idx, false, H,
             HD, s, st.ctrl + CTRL_LS, e->srclen.as<int>(), cross_desc);
    };

    auto enqueue_iteration = [&]() -> int {
        RowCount rows(Bq * per_q, n_active, per_q);
        {   // KV-cache append of the previous iteration's accepted tokens + embedding of this iteration's step tokens
            Scope sc(e, KC_EMBED, s);
            GreedyState stq = st;
            stq.B = Bq;               // grid sizing only: the kernel indexes the live slots, all below the bucket
            launch_greedy_advance<ActT>(stq, e->tgt_emb, e->pe, E, x, xh, e->qkv.as<ActT>(), qkv_l_stride, n_dec, 3 * E, kc, vc,
                                        cache_l_stride, cache_q_stride, E, s);
        }
        if (decoder_stack<ActT>(e, rows, n_dec, qkv_l_stride, self_attn, cross_attn, s)) return 1;
        if (sampling) {
            const SampleArgs sa{st.desc, smp_keys, S, smp.temperature, smp.top_k, st.pred};
            auto fused = [&](const auto* a) { return launch_classifier_sample(a, E, e->classifier.wh, e->classifier.b, rows, V, E, sa, s); };
            auto fallback = [&](const float* lg) { launch_sample_rows(lg, V, V, rows, sa, s); };
            if (classifier_head<ActT>(e, rows, use_fused, fused, fallback, e->logits.as<float>(), s)) return 1;
            Scope sc(e, KC_ACCEPT, s);
            launch_sample_step(st, sl, s);
            return 0;
        }
        auto fused = [&](const auto* a) { return launch_classifier_argmax(a, E, e->classifier.wh, e->classifier.b, st.pred, rows, V, E, s); };
        auto fallback = [&](const float* lg) { launch_argmax_rows(lg, V, V, st.pred, rows, s); };
        if (classifier_head<ActT>(e, rows, use_fused, fused, fallback, e->logits.as<float>(), s)) return 1;
        Scope sc(e, KC_ACCEPT, s);
        if (standard && cont) return launch_greedy_std_step_groups(st, cbt, s) ? 1 : 0;
        if (standard) launch_greedy_std_step(st, s);
        else if (cont) launch_greedy_accept_groups(st, cbt, s);
        else launch_greedy_accept(st, s);
        return 0;
    };

    // One decoding iteration is a fixed kernel sequence on fixed buffers (all sizes that change while
    // decoding live in device memory), so it is captured once into a CUDA graph and replayed.
    static const bool no_graph = env_flag("TTB_NO_GRAPH");
    bool traced = trace_dev != nullptr;
    if (cont && cb->trace)
        for (int i = 0; i < cb->n; ++i) traced |= cb->trace[i] != nullptr;
    const bool use_graph = !no_graph && !traced && e->prof.mask == 0;
    // Several iterations per graph: back-to-back graph launches of one stream leave the GPU idle for ~12 us (launch latency
    // plus the control-word copy in between), a graph edge costs ~2 us.  Iterations behind the end of the loop are no-ops
    // (every kernel reads a live count of zero), so a longer graph only adds a few of those per batch.
    static const int graph_iters = [] { const char* v = getenv("TTB_GRAPH_ITERS"); const int k = v ? atoi(v) : 4; return k < 1 ? 1 : (k > 16 ? 16 : k); }();
    const int K_it = use_graph ? graph_iters : 1;
    // buckets of live queries a graph is captured for (largest first; lazily, the first time the host picks one)
    int bucket_q[ttb_engine::kBuckets];
    int n_buckets = 0;
    {
        static const bool no_buckets = env_flag("TTB_NO_BUCKETS");
        int cand[ttb_engine::kBuckets];
        for (int i = 0; i < 8; ++i) cand[i] = (B * (8 - i) + 7) / 8;      // B, 7B/8, ... B/8
        cand[8] = (B + 15) / 16;
        cand[9] = 1;
        for (int i = 0; i < ttb_engine::kBuckets; ++i) {
            // generate() of the standard greedy decoding keeps every row to the end; its continuous loop sheds stopped batches
            // and sampling retires every slot on its own
            if (i > 0 && (no_buckets || (mode == GreedyMode::standard && !cont))) break;
            if (n_buckets == 0 || (cand[i] >= 1 && cand[i] < bucket_q[n_buckets - 1])) bucket_q[n_buckets++] = cand[i];
        }
    }
    if (use_graph) {
        // everything a call may change that the captured kernels take by value (the sampling keys are in device memory)
        uint32_t t_bits = 0;
        memcpy(&t_bits, &smp.temperature, 4);
        const long long key[17] = {B, N, D, (long long)mode + (cont ? 4 : 0), max_len, pad, bos, eos, tie_break,
                                   e->alloc_signature(), (long long)sizeof(ActT) + 16 * K_it, replace, cont ? Ls_cap : 0, S,
                                   (long long)t_bits, smp.top_k, use_fused ? 1 : 0};
        if (memcmp(key, e->graph_key, sizeof(key)) != 0) {
            for (auto& gb : e->graph_exec) for (auto& g : gb) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
            memcpy(e->graph_key, key, sizeof(key));
        }
    }
    // Once queries retire the graphs get SHORT (half the iterations): the host then follows the shrinking live count more
    // closely (smaller buckets sooner) and fewer no-op iterations run behind the end of the batch; while the whole batch is
    // alive (always, with random-init weights) the long graph saves the ~12 us boundary between launches.
    const int K_short = std::max(1, K_it / 2);
    auto graph_for = [&](int bi, int sh) -> int {      // capture on first use
        if (e->graph_exec[bi][sh]) return 0;
        const long long l0 = e->launches;
        cudaGraph_t graph = nullptr;
        Bq = bucket_q[bi];
        const int n_it = sh ? K_short : K_it;
        TTB_CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed));
        int rc = 0;
        for (int k = 0; k < n_it && !rc; ++k) rc = enqueue_iteration();
        cudaError_t ce = cudaStreamEndCapture(s, &graph);
        if (rc || ce != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            if (!rc) set_last_error(std::string("CUDA graph capture failed: ") + cudaGetErrorString(ce));
            return 1;
        }
        TTB_CUDA_OK(cudaGraphInstantiate(&e->graph_exec[bi][sh], graph, 0));
        cudaGraphDestroy(graph);
        e->graph_launches = (e->launches - l0) / n_it;   // per iteration
        e->launches = l0;  // capturing did not launch anything
        return 0;
    };

    // Lagged polling: the host looks at the control words of iteration (it - LAG) while iterations up
    // to `it` are already queued, so the GPU never waits for it.
    constexpr int RING = 4;
    const int LAG = K_it > 1 ? 1 : 2;   // launches (of K_it iterations each) the host stays ahead of the control words it reads
    // `bound` is an upper bound of the live queries of every iteration enqueued from now on: the count of the newest control
    // words read plus every query admitted after the launch they belong to (the device only retires queries).  It picks the
    // bucket -- a bucket below the true live count would drop queries.  Continuous loop: B - bound is a lower bound of the
    // free slots, a batch is admitted at a graph boundary once they suffice.  One batch: nothing is admitted, the loop ends
    // when the device has raised CTRL_DONE, and a live count of 0 read without it counts as 1.
    long long admitted = 0, adm_at[RING] = {};
    long long iters_enq = 0;
    int bound = cont ? 0 : B, it = 0;
    while (true) {
        if (cont) {
            int n = 0;
            if (sg.admit_fitting(B - bound, &n, admit)) return 1;
            bound += n;
            admitted += n;
        }
        if (bound == 0) break;   // done, or (continuous) nothing live and nothing pending: every batch fits the slots
        if (iters_enq >= max_iters) {
            TTB_CHECK(!cont, "continuous decoding loop did not terminate within max_len + 1 iterations per batch");
            break;
        }
        int bi = 0;
        while (bi + 1 < n_buckets && bucket_q[bi + 1] >= bound) ++bi;
        Bq = bucket_q[bi];
        if (use_graph) {
            const int sh = (bound < B && K_short < K_it) ? 1 : 0;
            if (graph_for(bi, sh)) return 1;
            TTB_CUDA_OK(cudaGraphLaunch(e->graph_exec[bi][sh], s));
            e->launches += e->graph_launches * (sh ? K_short : K_it);
            iters_enq += sh ? K_short : K_it;
        } else if (enqueue_iteration()) {
            return 1;
        } else {
            ++iters_enq;
        }
        TTB_CUDA_OK(cudaMemcpyAsync(e->h_ctrl + (it % RING) * CTRL_COUNT, st.ctrl, CTRL_COUNT * sizeof(int), cudaMemcpyDeviceToHost, s));
        TTB_CUDA_OK(cudaEventRecord(e->poll_ev[it % RING], s));
        adm_at[it % RING] = admitted;
        if (it >= LAG) {
            const int j = (it - LAG) % RING;
            TTB_CUDA_OK(cudaEventSynchronize(e->poll_ev[j]));
            const int* cj = e->h_ctrl + j * CTRL_COUNT;
            TTB_CHECK(cj[CTRL_ERROR] != 3, "continuous batching admitted a batch without enough free slots");
            const int live = cj[CTRL_DONE] ? 0 : (cont ? cj[CTRL_N_ACTIVE] : std::max(1, cj[CTRL_N_ACTIVE]));
            bound = std::min(bound, live + (int)(admitted - adm_at[j]));
        }
        ++it;
    }
    if (!cont) TTB_CUDA_OK(cudaMemcpyAsync(out_dev, st.out, (size_t)B * max_len * sizeof(long long), cudaMemcpyDeviceToDevice, s));
    TTB_CUDA_OK(cudaMemcpyAsync(e->h_ctrl, st.ctrl, CTRL_COUNT * sizeof(int), cudaMemcpyDeviceToHost, s));
    float ms = 0.f;
    if (int rc = finish_loop(e, ms)) return rc;
    const int* c = e->h_ctrl;
    std::vector<CbGroup> groups;
    if (cont) {
        TTB_CHECK(c[CTRL_ERROR] != 3, "continuous batching admitted a batch without enough free slots");
        TTB_CHECK(c[CTRL_DONE] == 1 && c[CTRL_N_ACTIVE] == 0, "continuous decoding loop ended with live queries");
        if (int rc = read_groups(cb, cbt.groups, groups)) return rc;
    } else {
        TTB_CHECK(c[CTRL_DONE] == 1, "greedy decoding loop did not terminate within max_len + 1 iterations");
    }
    e->h_hist.assign((size_t)c[CTRL_ITERS], 0);
    if (c[CTRL_ITERS] > 0)
        TTB_CUDA_OK(cudaMemcpy(e->h_hist.data(), st.hist, (size_t)c[CTRL_ITERS] * sizeof(int), cudaMemcpyDeviceToHost));
    auto ref_error = [](int err) { return err == 1 ? TTB_ERR_REF_INDEX : (err == 2 ? TTB_ERR_REF_SHAPE : 0); };
    if (cont) {   // per-batch records
        ttb_generate_stats sum{};
        for (int i = 0; i < cb->n; ++i) {
            const CbGroup& g = groups[(size_t)i];
            ttb_generate_stats& o = cb->stats[i];
            o = ttb_generate_stats{};
            o.model_calls = g.iter;
            o.accepted_tokens = g.accepted;
            o.produced_tokens = g.tokens;
            o.unfinished = g.n_left;
            o.error = ref_error(g.error);
            sum.accepted_tokens += g.accepted;
            sum.produced_tokens += g.tokens;
            sum.unfinished += g.n_left;
        }
        if (stats) {
            sum.model_calls = c[CTRL_ITERS];
            sum.gpu_launches = (int32_t)(e->launches - launches0);
            sum.gpu_ms = ms;
            *stats = sum;
        }
        return 0;
    }
    if (stats) {
        stats->model_calls = c[CTRL_ITERS];
        stats->accepted_tokens = c[CTRL_ACCEPTED];
        stats->produced_tokens = c[CTRL_TOKENS];
        stats->unfinished = c[CTRL_N_LEFT];
        stats->error = ref_error(c[CTRL_ERROR]);
        stats->gpu_launches = (int32_t)(e->launches - launches0);
        stats->gpu_ms = ms;
    }
    if (c[CTRL_ERROR] == 1) {
        set_last_error("index out of bounds while splicing drafts into the token matrix (reference scatter, speculative_decoding.py:111)");
        return TTB_ERR_REF_INDEX;
    }
    if (c[CTRL_ERROR] == 2) {
        set_last_error("shape mismatch: a finished row is wider than max_len (reference speculative_decoding.py:158)");
        return TTB_ERR_REF_SHAPE;
    }
    return 0;
}


// Waits for the word the closing CTA of iteration (step) `seq` of a beam-search loop posts into the pinned mapped ring at
// h_ctrl + 16 (four 64-bit words, sequence number in the top 24 bits).  *arrived = false when the stream drained without it
// (the mapping is unavailable); `pure_spin`: never give the core away between polls.
static int wait_posted_word(ttb_engine* e, cudaStream_t s, int seq, unsigned long long* out, bool* arrived, bool pure_spin) {
    volatile unsigned long long* word = reinterpret_cast<volatile unsigned long long*>(e->h_ctrl + 16) + (seq & 3);
    auto match = [&](unsigned long long w) { return (unsigned)((w >> 40) & 0xffffff) == (unsigned)(seq & 0xffffff); };
    *arrived = true;
    for (long spin = 0;; ++spin) {
        *out = *word;
        if (match(*out)) return 0;
        // the word normally arrives within a few microseconds of the last launch call; past that (long iterations,
        // several engines per GPU and ranks per box sharing the cores) the thread gives its core away between polls
        if (spin < 256 || pure_spin) cpu_relax(); else sched_yield();
        if ((spin & 0x3FFF) == 0x3FFF) {
            const cudaError_t q = cudaStreamQuery(s);
            if (q == cudaSuccess) {   // stream drained: the word is there, or the mapping is unavailable
                *out = *word;
                *arrived = match(*out);
                return 0;
            }
            if (q != cudaErrorNotReady) TTB_CUDA_OK(q);
        }
    }
}

// Device pointer of that ring, cleared, or nullptr when the mapping is unavailable.
static void* map_posted_ring(ttb_engine* e) {
    void* dp = nullptr;
    for (int i = 16; i < 24; ++i) e->h_ctrl[i] = 0;
    const bool mapped = cudaHostGetDevicePointer(&dp, e->h_ctrl + 16, 0) == cudaSuccess;
    (void)cudaGetLastError();
    return mapped ? dp : nullptr;
}

// ---- speculative beam search (speculative_decoding.py:428-598), host loop + device kernels ---------------
// The per-iteration shapes (token-matrix width, draft length, live rows) depend on the hypotheses, so the
// host reads a handful of control words back once per iteration; tokens, scores and logits never leave
// the device.  With `cb` the loop is the continuous one: B is the number of query slots, Ls the longest source of all
// batches, and the batches of `cb` are admitted into free slots between two iterations.
template <typename ActT>
static int beam_api(ttb_engine* e, const int64_t* src_dev, int B, int Ls, int max_len, int K, int draft_len, int N,
                    int pad, int bos, int eos, int c_token, int tie_break, int64_t* out_dev, int32_t* out_width,
                    int32_t* trace_nacc, int32_t* trace_pick, ttb_generate_stats* stats, cudaStream_t user_stream, bool smart,
                    const BatchList* cb = nullptr) {
    const int E = e->E(), H = e->d.num_heads, HD = e->HD(), V = e->d.tgt_vocab_size;
    const int n_dec = (int)e->dec.size();
    cudaStream_t s = e->stream;
    if (int rc = join_caller_stream(e, user_stream)) return rc;
    const long long launches0 = e->launches;
    const int D0 = std::min(std::max(5, draft_len), 200);       // speculative_decoding.py:278-284
    // smart_drafts_mode (:600-615): library of Ls - 5 windows of draft_len + 1 tokens (BOS column included), first token = key
    const int D_lib = std::min(std::max(5, D0 + 1), 200);
    const int n_lib = Ls - 5;
    if (smart) TTB_CHECK(n_lib > 0, "The number of drafts must be greater than 0");
    const int Ls_cap = ls_capacity(Ls);
    const long long TS_cap = (long long)B * Ls_cap;
    const int Cmax = B * K, Rmax = Cmax * N;
    const int ldw = max_len + D0 + 4;
    // only the dl+1 scored positions of every (candidate, draft) row go through the decoder, the prefix of a candidate is
    // served from its self-attention cache, which follows the hypotheses through the re-parenting of every step
    const bool cont = cb != nullptr;
    Staging<ActT> sg(cb);
    const long long Tc = (long long)Rmax * (D0 + 1);
    // bf16 path: the statistics the search reads come from the fused classifier (TTB_NO_FUSED_STATS=1: GEMM + beam_stats)
    const bool use_fused = Prec<ActT>::lowp && !env_flag("TTB_NO_FUSED_STATS");

    if (ensure_encoder<ActT>(e, cont ? sg.TS_stage : TS_cap, B, TS_cap)) return 1;
    if (e->drafts.ensure(smart ? (size_t)B * std::max(n_lib, Ls_cap) * D_lib * sizeof(int) : (size_t)B * N * D0 * sizeof(int))) return 1;
    if (ensure_work<ActT>(e, cont ? Tc : std::max(Tc, TS_cap), n_dec)) return 1;
    const long long cache_c_stride = (long long)ldw * E, cache_l_stride = (long long)Cmax * ldw * E;
    const size_t cbytes = (size_t)n_dec * cache_l_stride * sizeof(ActT);
    if (e->kcache.ensure(cbytes) || e->vcache.ensure(cbytes) || e->kcache2.ensure(cbytes) || e->vcache2.ensure(cbytes)) return 1;
    DevBuf& bb = e->beam;
    // one arena for the small beam buffers
    Arena a;
    const size_t o_cand0 = a.take((size_t)Cmax * ldw * 4), o_cand1 = a.take((size_t)Cmax * ldw * 4);
    const size_t o_lp0 = a.take(Cmax * 4), o_lp1 = a.take(Cmax * 4);
    const size_t o_slot = a.take(Cmax * 4), o_fin = a.take(Cmax * 4), o_base = a.take(Cmax * 4), o_nacc = a.take((size_t)Cmax * N * 4);
    const size_t o_pick = a.take(Cmax * 4), o_acc = a.take(Cmax * 4), o_ctrl = a.take(32 * 4);   // control words + loop-control accumulators
    const size_t n_rp = (size_t)Rmax * (D0 + 1);
    const size_t o_topv = a.take(n_rp * K * 4), o_topi = a.take(n_rp * K * 4), o_keep = a.take(n_rp * 4), o_max = a.take(n_rp * 4), o_sum = a.take(n_rp * 4);
    const size_t o_lg = a.take(n_rp * V * 4), o_rt = a.take(n_rp * 4), o_tv = a.take(n_rp * 4);
    const size_t o_lc = a.take(Rmax * 4), o_lq = a.take(Rmax * 4), o_cf = a.take(Cmax * 4), o_np = a.take(Cmax * 4), o_nk = a.take(Cmax * 4), o_nr = a.take(Cmax * 4);
    const size_t o_tc = a.take(smart ? (size_t)B * V * 4 : 4), o_tl = a.take(smart ? (size_t)B * V * N * 4 : 4), o_cc = a.take(Cmax * 4),
                 o_cl = a.take(Cmax * 4), o_rd = a.take(Rmax * 4), o_ds = a.take(Rmax * 16), o_dc = a.take(Rmax * 16);
    if (bb.ensure(a.bytes)) return 1;
    char* base = bb.as<char>();
    // continuous loop: slot / batch tables, staging of an admitted batch (drafts or window library as well), smallest draft
    // length of every iteration
    BcTable cbt{};
    int *stage_drafts = nullptr, *stage_tokcnt = nullptr, *stage_toklist = nullptr;
    if (cont) {
        TTB_CHECK(B <= 2048 && (long long)B * K < 65536, "continuous batching supports at most 2048 slots and 65535 candidates");
        const size_t B_stage = (size_t)sg.B_stage;
        if (int rc = sg.alloc(e, cbt, B, Ls_cap, {{&stage_drafts, (smart ? (size_t)std::max(n_lib, 1) * D_lib : (size_t)N * D0) * B_stage * 4},
                                                   {&stage_tokcnt, smart ? B_stage * V * 4 : 4},
                                                   {&stage_toklist, smart ? B_stage * V * N * 4 : 4},
                                                   {&cbt.dl_min, ((size_t)cb->n * (max_len + 1) + 1) * sizeof(int)}}))
            return rc;
    }
    // nothing is allocated from here on (cudaFree would synchronise the device)
    sg.sig0 = e->alloc_signature();

    TTB_CUDA_OK(cudaEventRecord(e->t0, s));
    int* src32 = e->src32.as<int>();
    ActT* crosskv = e->crosskv.as<ActT>();
    const long long ckv_l_stride = TS_cap * 2 * E;
    // cross-attention key tokens and K/V rows: per query (generate()) or slot-major with Ls_cap rows per slot (continuous loop)
    const int kv_ls = cont ? Ls_cap : Ls;
    const int* key_tok = cont ? e->keytok32.as<int>() : src32;
    if (!cont) {
        if (encode_batch<ActT>(e, src_dev, B, Ls, e->srclen.as<int>(), crosskv, ckv_l_stride, s)) return 1;
        if (smart) { Scope sc(e, KC_MISC, s); launch_make_drafts(src32, Ls, B, Ls, D_lib, n_lib, eos, pad, c_token, e->drafts.as<int>(), s); }
        else { Scope sc(e, KC_MISC, s); launch_make_drafts(src32 + 1, Ls, B, Ls - 1, D0, N, eos, pad, c_token, e->drafts.as<int>(), s); }
    }

    BeamState st{};
    st.B = B; st.K = K; st.N = N; st.dl0 = smart ? D_lib : D0; st.V = V; st.smart = smart ? 1 : 0; st.n_lib = n_lib; st.pad = pad; st.bos = bos; st.eos = eos; st.ldw = ldw; st.tie_break = tie_break;
    st.max_len = max_len;
    {   // width of the token matrix in the first iteration (the loop below applies the same rule)
        const int dl_first = std::min(max_len - 2, smart ? D_lib - 1 : D0);
        st.w0 = 1 + std::max(dl_first + 1, 0);
    }
    st.cand_cur = (int*)(base + o_cand0); st.cand_next = (int*)(base + o_cand1);
    st.logp_cur = (float*)(base + o_lp0); st.logp_next = (float*)(base + o_lp1);
    st.drafts = e->drafts.as<int>();
    st.c_slot0 = (int*)(base + o_slot); st.c_fin = (int*)(base + o_fin); st.c_rowbase = (int*)(base + o_base);
    st.c_nacc = (int*)(base + o_nacc); st.c_pick = (int*)(base + o_pick); st.acc_stat = (int*)(base + o_acc); st.ctrl = (int*)(base + o_ctrl);
    st.topv = (float*)(base + o_topv); st.topi = (int*)(base + o_topi); st.nkeep = (int*)(base + o_keep);
    st.lmax = (float*)(base + o_max); st.lsum = (float*)(base + o_sum);
    st.trace_nacc = trace_nacc; st.trace_pick = trace_pick;
    st.host_ctrl = static_cast<int*>(map_posted_ring(e));   // the expand kernel posts into it
    st.row_tok = (int*)(base + o_rt); st.tokv = (float*)(base + o_tv);
    st.live_cand = (int*)(base + o_lc); st.live_query = (int*)(base + o_lq); st.c_front = (int*)(base + o_cf);
    st.n_parent = (int*)(base + o_np); st.n_keep = (int*)(base + o_nk); st.n_row = (int*)(base + o_nr);
    st.tok_cnt = (int*)(base + o_tc); st.tok_list = (int*)(base + o_tl); st.c_cnt = (int*)(base + o_cc); st.c_last = (int*)(base + o_cl);
    st.row_draft = (int*)(base + o_rd);
    st.desc_self = (int4*)(base + o_ds); st.desc_cross = (int4*)(base + o_dc); st.src_len = e->srclen.as<int>();
    ActT* kc_cur = e->kcache.as<ActT>();
    ActT* vc_cur = e->vcache.as<ActT>();
    ActT* kc_next = e->kcache2.as<ActT>();
    ActT* vc_next = e->vcache2.as<ActT>();
    const int* n_live_cands = st.ctrl + BC_NLIVE_CANDS;
    float* logits = (float*)(base + o_lg);
    if (cont) {
        TTB_CHECK(st.host_ctrl, "continuous batching needs mapped pinned host memory for its control word");
        TTB_CUDA_OK(cudaMemsetAsync(st.ctrl, 0, 32 * sizeof(int), s));
        TTB_CUDA_OK(cudaMemsetAsync(cbt.slots.slot_group, 0xff, (size_t)B * sizeof(int), s));   // every slot free
        TTB_CUDA_OK(cudaMemsetAsync(st.n_parent, 0xff, (size_t)Cmax * sizeof(int), s));
        TTB_CUDA_OK(cudaMemsetAsync(cbt.groups, 0, (size_t)cb->n * sizeof(BcGroup), s));
    } else {
        { Scope sc(e, KC_MISC, s); launch_beam_init(st, s); }
        if (smart) { Scope sc(e, KC_MISC, s); launch_beam_build_lib(st, s); }
    }

    float* x = e->x.as<float>();
    ActT* xh = Prec<ActT>::lowp ? e->xh.as<ActT>() : nullptr;
    const int* n_live = st.ctrl + BC_NLIVE_ROWS;
    int W = 1, empty_cols = 0, filled = 1, budget = max_len - filled - 1, dl = smart ? D_lib - 1 : D0, C = B, beam = 1, iters = 0;
    const int dl_steady = dl;   // full draft length: an iteration at it may be enqueued ahead (host loop below)
    int* hc = e->h_ctrl;
    hc[BC_ERROR] = 0;
    // the two hypothesis / score / cache buffer sets: iteration i (0-based) reads set i & 1 and writes the other one
    int* const cand_set[2] = {st.cand_cur, st.cand_next};
    float* const logp_set[2] = {st.logp_cur, st.logp_next};
    ActT* const kc_set[2] = {kc_cur, kc_next};
    ActT* const vc_set[2] = {vc_cur, vc_next};

    // One iteration = a fixed kernel sequence whose arguments depend on (C, beam, dl) and on the ping-pong parity of the
    // hypothesis / cache buffers only: the width of the token matrix and the iteration number live in device memory
    // (beam.cu: BCX_W, BCX_ITER), and the device applies the stop rule itself (BCX_DONE), so the steady state (C = B K,
    // full draft length) can be enqueued AHEAD of the host reading the outcome of the iteration before it.
    // `Cb`: upper bound of the candidates that are still unfinished in this iteration (exact when the host has read the word
    // of the iteration before, C otherwise): the decoder-side grids are sized for Cb * N rows instead of C * N, so that the
    // no-op CTAs of finished candidates do not queue for SMs that the other batches in flight are using (§4c of DESIGN.md)
    auto enqueue_iteration = [&](int it, int C, int beam, int dl, int Cb) -> int {
        const int parity = it & 1;
        st.cand_cur = cand_set[parity]; st.cand_next = cand_set[parity ^ 1];
        st.logp_cur = logp_set[parity]; st.logp_next = logp_set[parity ^ 1];
        kc_cur = kc_set[parity]; kc_next = kc_set[parity ^ 1];
        vc_cur = vc_set[parity]; vc_next = vc_set[parity ^ 1];
        const int R = (smart && !cont ? C : std::min(C, std::max(1, Cb))) * N;
        if (cont) { Scope sc(e, KC_MISC, s); launch_beam_prepare_groups(st, cbt, s); }
        else { Scope sc(e, KC_MISC, s); launch_beam_prepare(st, C, beam, dl, s); }
        RowCount rows(R * (dl + 1), n_live, dl + 1);
        { Scope sc(e, KC_EMBED, s); launch_beam_embed_cached<ActT>(st, beam, R, dl, e->tgt_emb, e->pe, E, x, xh, s); }
        // attention groups: the N rows of a live candidate share its cache prefix; in smart mode candidates own a
        // different number of rows, so every row is a group of its own
        const int G = smart ? R : R / N, n_per_group = smart ? 1 : N;
        auto self_attn = [&](int l, ActT* qkv, ActT* att) {
            // continuous loop: a candidate's draft rows are its batch's dl + 1 positions long (desc_self.w), whatever the
            // call's dl, so that the tensor-core kernel lays out its keys as generate() does
            spec_attn(qkv, 3 * E, kc_cur + l * cache_l_stride, vc_cur + l * cache_l_stride, cache_c_stride, E, att, E, G, n_live_cands,
                      st.live_cand, st.c_front, st.cand_cur, ldw, e->d.tgt_pad_token_idx, n_per_group, dl, H, HD, ldw, s, st.desc_self, cont);
        };
        auto cross_attn = [&](int l, ActT* q2, ActT* att) {
            const ActT* kv = crosskv + (long long)l * ckv_l_stride;
            attn(q2, E, kv, kv + E, 2 * E, att, E, G, n_live_cands, n_per_group * (dl + 1), kv_ls, kv_ls, st.live_query, key_tok, kv_ls,
                 e->d.src_pad_token_idx, false, H, HD, s, nullptr, nullptr, st.desc_cross);
        };
        if (decoder_stack<ActT>(e, rows, n_dec, Tc * 3 * E, self_attn, cross_attn, s)) return 1;
        // every decoder row is a scored position: the statistics the search reads (logits in tensor memory when fused)
        auto fused = [&](const auto* a) {
            return launch_classifier_stats(a, E, e->classifier.wh, e->classifier.b, rows, V, E, K, st.row_tok, st.tokv, st.lmax, st.lsum,
                                           st.nkeep, st.topv, st.topi, s);
        };
        auto fallback = [&](const float* lg) { launch_beam_stats(st, lg, R, dl, s); };
        if (classifier_head<ActT>(e, rows, use_fused, fused, fallback, logits, s)) return 1;
        if (cont) { Scope sc(e, KC_ACCEPT, s); launch_beam_choose_groups(st, cbt, dl, s); }
        else { Scope sc(e, KC_ACCEPT, s); launch_beam_choose(st, C, beam, dl, s); }
        // the expand kernel also closes the iteration: its last CTA writes the control words and, last, the iteration's
        // sequence number into pinned host memory; the host reads them while the caches are still being re-parented
        if (cont) { Scope sc(e, KC_ACCEPT, s); launch_beam_expand_groups(st, cbt, dl, s); }
        else { Scope sc(e, KC_ACCEPT, s); launch_beam_expand(st, beam, dl, s); }
        {
            Scope sc(e, KC_CACHE_APPEND, s);
            launch_beam_cache_update<ActT>(st, dl, e->qkv.as<ActT>(), Tc * 3 * E, n_dec, 3 * E, E, kc_cur, vc_cur, kc_next, vc_next,
                                           cache_l_stride, cache_c_stride, s);
        }
        return 0;
    };
    // wait for the packed word the expand kernel posts for iteration `seq` (sequence | error | all finished | empty columns)
    static const bool pure_spin = env_flag("TTB_BEAM_SPIN");
    int live_next = B;      // unfinished candidates entering the next iteration, from the newest word read
    int cont_used = 0, cont_dl = 0;   // continuous loop: slots in use and largest draft length of the open batches, idem
    auto wait_word = [&](int seq) -> int {
        unsigned long long w = 0;
        bool arrived = true;
        if (int rc = wait_posted_word(e, s, seq, &w, &arrived, pure_spin)) return rc;
        if (!arrived) {   // the stream drained without the word (mapping unavailable): take a copy of the control words
            TTB_CHECK(!cont, "the control word of the continuous beam-search loop did not arrive");
            TTB_CUDA_OK(cudaMemcpy(hc, st.ctrl, BC_COUNT * sizeof(int), cudaMemcpyDeviceToHost));
            w = ((unsigned long long)(seq & 0xffffff) << 40) | ((unsigned long long)(hc[BC_ERROR] & 0xf) << 36) |
                ((unsigned long long)(hc[BC_ALL_FINISHED] & 1) << 35) | ((unsigned long long)(hc[BC_EMPTY_COLS] & 0xfff) << 23) |
                ((unsigned long long)0xffff << 7);   // live candidates unknown: full grids
        }
        if (cont) {   // sequence | slots in use | largest draft length of the open batches | unfinished candidates
            cont_used = (int)((w >> 28) & 0xfff);
            cont_dl = (int)((w >> 20) & 0xff);
            live_next = (int)((w >> 4) & 0xffff);
            return 0;
        }
        hc[BC_ERROR] = (int)((w >> 36) & 0xf);
        hc[BC_ALL_FINISHED] = (int)((w >> 35) & 1);
        hc[BC_EMPTY_COLS] = (int)((w >> 23) & 0xfff);
        live_next = (int)((w >> 7) & 0xffff);
        return 0;
    };
    // Host loop.  `iters` iterations have been read back (their outcome is known exactly: W, filled, budget, dl below are
    // the reference's values before iteration `iters`); `enq` iterations have been enqueued.  In the steady state the next
    // iteration is enqueued BEFORE the word of the current one is awaited whenever its arguments cannot depend on that
    // word: C = B K and beam = K from the second iteration on, and the draft length stays dl as long as the length budget
    // cannot drop below it (one iteration fills at most dl + 1 more columns).  If the current iteration ends the loop the
    // device has raised BCX_DONE and the iteration enqueued ahead does nothing.
    if (cont) {
        // Continuous loop.  Between two iterations the host admits the next batches (whole, in list order) while the free
        // slots of the newest word suffice, then enqueues one iteration at the largest draft length of the open batches
        // and waits for its word.  Nothing is enqueued ahead: the coming iteration's draft length and admissions depend
        // on the word.
        const int dl_first = std::min(max_len - 2, dl);   // the first iteration's draft length (budget max_len - 2)
        auto admit = [&](int i) -> int {
            const int Bi = cb->bs[i], Li = cb->ls[i], lib_i = Li - 5;
            if (int rc = sg.encode(e, i, s)) return rc;
            if (smart) {
                { Scope sc(e, KC_MISC, s); launch_make_drafts(src32, Li, Bi, Li, D_lib, lib_i, eos, pad, c_token, stage_drafts, s); }
                BeamState lib = st;   // the batch's library alone, as generate() builds it
                lib.B = Bi; lib.n_lib = lib_i; lib.drafts = stage_drafts; lib.tok_cnt = stage_tokcnt; lib.tok_list = stage_toklist;
                Scope sc(e, KC_MISC, s);
                launch_beam_build_lib(lib, s);
            } else {
                Scope sc(e, KC_MISC, s);
                launch_make_drafts(src32 + 1, Li, Bi, Li - 1, D0, N, eos, pad, c_token, stage_drafts, s);
            }
            {
                Scope sc(e, KC_MISC, s);
                if (int rc = launch_beam_admit(st, cbt, i, Bi, stage_drafts, lib_i, stage_tokcnt, stage_toklist, sg.srclen,
                                               reinterpret_cast<long long*>(cb->out[i]), cb->trace_nacc ? cb->trace_nacc[i] : nullptr,
                                               cb->trace_pick ? cb->trace_pick[i] : nullptr, dl_first, s))
                    return rc;
            }
            cbt.n_groups = i + 1;
            return sg.scatter(e, cbt.slots, i, s);
        };
        // every batch takes part in at most max_len iterations
        const long long max_iters = (long long)cb->n * (max_len + 1);
        std::vector<int> hist, hist_dl;
        int it = 0;
        live_next = 0;
        // TTB_BEAM_CB_FULL_DL=1 (read per call): every decoder call runs at the first iteration's draft length, so that
        // every batch near max_len runs with a shorter dl than the call's (a check that results do not depend on it)
        const bool force_full_dl = env_flag("TTB_BEAM_CB_FULL_DL");
        while (true) {
            int dl_it = force_full_dl ? dl_first : cont_dl;
            int n = 0;
            if (sg.admit_fitting(B - cont_used, &n, admit)) return 1;
            cont_used += n;
            live_next += n;
            if (n > 0) dl_it = std::max(dl_it, dl_first);
            if (cont_used == 0) break;   // nothing open and nothing pending (every batch fits the slots)
            TTB_CHECK(it < max_iters, "continuous beam-search loop did not terminate within max_len iterations per batch");
            hist.push_back(cont_used);
            hist_dl.push_back(dl_it);
            if (enqueue_iteration(it, B * K, K, dl_it, std::min(live_next, B * K))) return 1;
            if (wait_word(it + 1)) return 1;
            ++it;
        }
        float ms = 0.f;
        if (int rc = finish_loop(e, ms)) return rc;
        int ctrl_end[32] = {};
        TTB_CUDA_OK(cudaMemcpy(ctrl_end, st.ctrl, sizeof(ctrl_end), cudaMemcpyDeviceToHost));
        TTB_CHECK(ctrl_end[BC_COUNT + 11] == 0, "continuous batching admitted a batch without enough free slots");
        std::vector<BcGroup> groups;
        if (int rc = read_groups(cb, cbt.groups, groups)) return rc;
        e->h_hist = hist;
        e->h_dl = hist_dl;
        e->h_dl_min.assign(hist_dl.size(), 0);
        if (it > 0) TTB_CUDA_OK(cudaMemcpy(e->h_dl_min.data(), cbt.dl_min, (size_t)it * sizeof(int), cudaMemcpyDeviceToHost));
        ttb_generate_stats sum{};
        for (int i = 0; i < cb->n; ++i) {
            const BcGroup& g = groups[(size_t)i];
            ttb_generate_stats& o = cb->stats[i];
            o = ttb_generate_stats{};
            o.model_calls = g.iter;
            o.accepted_tokens = g.accepted;
            o.produced_tokens = g.produced;
            o.error = g.error == 3 ? TTB_ERR_REF_SHAPE : (g.error == 4 ? TTB_ERR_REF_ASSERT : 0);
            cb->out_width[i] = g.W;
            sum.accepted_tokens += g.accepted;
            sum.produced_tokens += g.produced;
        }
        if (stats) {
            sum.model_calls = it;
            sum.gpu_launches = (int32_t)(e->launches - launches0);
            sum.gpu_ms = ms;
            *stats = sum;
        }
        return 0;
    }
    static const bool no_ahead = env_flag("TTB_BEAM_NO_AHEAD");
    const bool ahead_ok = st.host_ctrl && !no_ahead && !trace_nacc && !trace_pick;
    int enq = 0, dl_enq = dl;
    bool ended = false;
    while (!ended) {
        if (enq == iters) {                              // nothing in flight: the coming iteration from exact knowledge
            if (!(budget >= 1 && filled <= max_len)) break;
            dl = std::min(budget, dl);
            const int grow = dl + 1 - empty_cols;
            if (grow > 0) W += grow;
            TTB_CHECK(W <= ldw, "beam search token matrix outgrew its buffer");
            if (enqueue_iteration(enq, C, beam, dl, std::min(live_next, C))) return 1;
            dl_enq = dl;
            ++enq;
        }
        // ahead of the word only while every candidate is alive (iteration 0 aside): once hypotheses finish, the exact live
        // count of the word sizes the next iteration's grids, which is worth more than the host's head start (both measured)
        if (ahead_ok && enq == iters + 1 && dl_enq == dl_steady && max_len - (filled + 2 * (dl_enq + 1)) - 1 >= dl_enq &&
            W + 2 * (dl_enq + 1) <= ldw && (iters == 0 || live_next >= B * K)) {
            // `filled` is the exact count before the iteration in flight: after it and one more at most 2 (dl + 1) columns are added
            if (enqueue_iteration(enq, B * K, K, dl_enq, B * K)) return 1;
            ++enq;
        }
        if (wait_word(iters + 1)) return 1;
        ++iters;
        if (hc[BC_ERROR]) break;
        C = B * K;
        beam = K;
        if (hc[BC_ALL_FINISHED]) break;
        empty_cols = hc[BC_EMPTY_COLS];
        filled = W - empty_cols;
        budget = max_len - filled - 1;
        if (enq > iters) {
            // the iteration enqueued ahead runs with the values the reference would use: same dl (checked above), and
            // its token matrix is this one's plus the columns the device adds with the same rule
            if (!(budget >= 1 && filled <= max_len)) { ended = true; break; }   // the device stopped as well (BCX_DONE)
            const int grow = dl + 1 - empty_cols;
            if (grow > 0) W += grow;
        }
    }
    // the hypotheses of the last iteration that really ran are in the set it wrote
    st.cand_cur = cand_set[iters & 1];
    TTB_CUDA_OK(cudaGetLastError());
    const int err = hc[BC_ERROR];
    if (!err) {
        TTB_CHECK(iters > 0, "max_len too small for the speculative beam search (the reference fails as well)");
        launch_beam_export(st.cand_cur, ldw, B * K, W, reinterpret_cast<long long*>(out_dev), s);
        e->launches++;
    }
    float ms = 0.f;
    if (int rc = finish_loop(e, ms)) return rc;
    if (out_width) *out_width = W;
    if (stats) {
        int fin_ctrl[BC_COUNT] = {};
        if (iters > 0) TTB_CUDA_OK(cudaMemcpy(fin_ctrl, st.ctrl, sizeof(fin_ctrl), cudaMemcpyDeviceToHost));
        stats->model_calls = iters;
        stats->accepted_tokens = fin_ctrl[BC_ACCEPTED];
        stats->produced_tokens = fin_ctrl[BC_PRODUCED];
        stats->unfinished = 0;
        stats->error = err;
        stats->gpu_launches = (int32_t)(e->launches - launches0);
        stats->gpu_ms = ms;
    }
    if (err == 3) {
        set_last_error("PAD predicted inside a hypothesis: draft slots are not contiguous (the reference fails on the reshape at speculative_decoding.py:524-526)");
        return TTB_ERR_REF_SHAPE;
    }
    if (err == 4) {
        set_last_error("fewer candidate continuations than n_best (reference assert in topk_in_each_group, speculative_decoding.py:195)");
        return TTB_ERR_REF_ASSERT;
    }
    return 0;
}

// ---- standard beam search (standard_decoding.py:90-174), host loop + device kernels -----------------------------
// One decoder call per generated column on the hypotheses that have not produced EOS, one new token each (the prefix of a
// hypothesis is served from its self-attention cache, which follows the hypotheses through the re-parenting of every step,
// in two ping-pong copies); tokens, scores and logits stay on the device, the host reads the control words of the stop
// test one step behind.

// With `cb` the loop is the continuous one: B is the number of query slots, Ls the longest source of all batches, and the
// batches of `cb` are admitted into free slots between two steps.
template <typename ActT>
static int std_beam_api(ttb_engine* e, const int64_t* src_dev, int B, int Ls, int max_len, int K, int pad, int bos, int eos,
                        int64_t* out_dev, int32_t* out_width, ttb_generate_stats* stats, cudaStream_t user_stream, const BatchList* cb = nullptr) {
    const int E = e->E(), H = e->d.num_heads, HD = e->HD(), V = e->d.tgt_vocab_size;
    const int n_dec = (int)e->dec.size();
    cudaStream_t s = e->stream;
    if (int rc = join_caller_stream(e, user_stream)) return rc;
    const long long launches0 = e->launches;
    const bool cont = cb != nullptr;
    const long long TS = (long long)B * Ls;
    const int Ls_cap = ls_capacity(Ls);
    const long long TS_cap = (long long)B * Ls_cap;
    const int Cmax = B * K, ldw = max_len;
    Staging<ActT> sg(cb);

    if (ensure_encoder<ActT>(e, cont ? sg.TS_stage : TS_cap, B, TS_cap)) return 1;
    if (ensure_work<ActT>(e, cont ? (long long)Cmax : std::max<long long>(Cmax, TS_cap), n_dec)) return 1;
    DevBuf& bb = e->beam;
    Arena a;
    const size_t o_y0 = a.take((size_t)Cmax * ldw * 4), o_y1 = a.take((size_t)Cmax * ldw * 4);
    const size_t o_s0 = a.take(Cmax * 4), o_s1 = a.take(Cmax * 4), o_fin = a.take(Cmax * 4), o_cr = a.take(Cmax * 4), o_rc = a.take(Cmax * 4),
                 o_rq = a.take(Cmax * 4), o_tot = a.take((size_t)Cmax * V * 4), o_ctrl = a.take(64), o_lg = a.take((size_t)Cmax * V * 4),
                 o_cf = a.take(Cmax * 4), o_par = a.take(Cmax * 4), o_ds = a.take(Cmax * 16), o_dc = a.take(Cmax * 16);
    if (bb.ensure(a.bytes)) return 1;
    const long long cache_c_stride = (long long)max_len * E, cache_l_stride = (long long)Cmax * max_len * E;
    const size_t cbytes = (size_t)n_dec * cache_l_stride * sizeof(ActT);
    if (e->kcache.ensure(cbytes) || e->vcache.ensure(cbytes) || e->kcache2.ensure(cbytes) || e->vcache2.ensure(cbytes)) return 1;
    // continuous loop: slot / batch tables, staging of an admitted batch
    SbTable cbt{};
    if (cont)
        if (int rc = sg.alloc(e, cbt, B, Ls_cap, {})) return rc;
    // nothing is allocated from here on (cudaFree would synchronise the device)
    sg.sig0 = e->alloc_signature();
    char* base = bb.as<char>();

    TTB_CUDA_OK(cudaEventRecord(e->t0, s));
    int* src32 = e->src32.as<int>();
    ActT* crosskv = e->crosskv.as<ActT>();
    if (!cont && encode_batch<ActT>(e, src_dev, B, Ls, e->srclen.as<int>(), crosskv, TS * 2 * E, s)) return 1;

    StdBeamState st{};
    st.B = B; st.K = K; st.V = V; st.pad = pad; st.bos = bos; st.eos = eos; st.ldw = ldw; st.max_len = max_len;
    st.y_cur = (int*)(base + o_y0); st.y_next = (int*)(base + o_y1);
    st.score_cur = (float*)(base + o_s0); st.score_next = (float*)(base + o_s1);
    st.fin = (int*)(base + o_fin); st.cand_row = (int*)(base + o_cr); st.row_cand = (int*)(base + o_rc); st.row_query = (int*)(base + o_rq);
    st.total = (float*)(base + o_tot); st.ctrl = (int*)(base + o_ctrl);
    float* logits = (float*)(base + o_lg);
    int* const y_set[2] = {st.y_cur, st.y_next};
    float* const score_set[2] = {st.score_cur, st.score_next};
    st.c_front = (int*)(base + o_cf); st.parent = (int*)(base + o_par);
    st.desc_self = (int4*)(base + o_ds); st.desc_cross = (int4*)(base + o_dc);
    st.src_len = e->srclen.as<int>();
    ActT *kc_cur = e->kcache.as<ActT>(), *vc_cur = e->vcache.as<ActT>(), *kc_next = e->kcache2.as<ActT>(), *vc_next = e->vcache2.as<ActT>();
    if (cont) {
        st.host_ctrl = static_cast<unsigned long long*>(map_posted_ring(e));   // the select kernel posts into it
        TTB_CHECK(st.host_ctrl, "continuous batching needs mapped pinned host memory for its control word");
        TTB_CUDA_OK(cudaMemsetAsync(st.ctrl, 0, 64, s));
        TTB_CUDA_OK(cudaMemsetAsync(cbt.slots.slot_group, 0xff, (size_t)B * sizeof(int), s));   // every slot free
        TTB_CUDA_OK(cudaMemsetAsync(cbt.groups, 0, (size_t)cb->n * sizeof(SbGroup), s));
    } else {
        Scope sc(e, KC_MISC, s);
        launch_sbeam_init(st, s);
    }

    float* x = e->x.as<float>();
    ActT* xh = Prec<ActT>::lowp ? e->xh.as<ActT>() : nullptr;
    const int* n_live = st.ctrl;
    // cross-attention K/V and key tokens: per query (generate()) or slot-major with Ls_cap rows per slot (continuous loop)
    const int kv_ls = cont ? Ls_cap : Ls;
    const int* key_tok = cont ? e->keytok32.as<int>() : src32;
    const long long ckv_l_stride = (cont ? TS_cap : TS) * 2 * E;
    const int max_beam = max_len > 2 ? K : 1;   // the first step of a query selects among V continuations, later ones among K V
    // One step: C hypotheses (grid of the per-hypothesis kernels), at most R live rows (grid of the decoder kernels), W and
    // beam of generate()'s step (the continuous kernels read them per batch)
    auto enqueue_step = [&](int C, int beam, int W, int R) -> int {
        if (cont) { Scope sc(e, KC_MISC, s); launch_sbeam_prepare_groups(st, cbt, s); }
        else { Scope sc(e, KC_MISC, s); launch_sbeam_prepare(st, C, beam, W, s); }
        RowCount rows1(R, n_live, 1);
        { Scope sc(e, KC_EMBED, s); launch_sbeam_embed_last<ActT>(st, R, e->tgt_emb, e->pe, E, x, xh, s); }
        auto self_attn = [&](int l, ActT* qkv, ActT* att) {
            spec_attn(qkv, 3 * E, kc_cur + l * cache_l_stride, vc_cur + l * cache_l_stride, cache_c_stride, E, att, E, R, n_live, st.row_cand,
                      st.c_front, st.y_cur, ldw, e->d.tgt_pad_token_idx, 1, 0, H, HD, max_len, s, st.desc_self);
        };
        auto cross_attn = [&](int l, ActT* q2, ActT* att) {
            const ActT* kv = crosskv + (long long)l * ckv_l_stride;
            attn(q2, E, kv, kv + E, 2 * E, att, E, R, n_live, 1, kv_ls, kv_ls, st.row_query, key_tok, kv_ls, e->d.src_pad_token_idx, false, H, HD, s,
                 nullptr, nullptr, st.desc_cross);
        };
        if (decoder_stack<ActT>(e, rows1, n_dec, (long long)Cmax * 3 * E, self_attn, cross_attn, s)) return 1;
        // every live row is the last position of its hypothesis: logits straight from the residual stream
        if (linear<float>(e, KC_GEMM_CLASSIFIER, a_view<ActT>(x, xh), E, e->classifier, logits, V, rows1, false, s)) return 1;
        { Scope sc(e, KC_ARGMAX, s); launch_sbeam_scores(st, C, logits, s); }
        {
            Scope sc(e, KC_ACCEPT, s);
            const int rc = cont ? launch_sbeam_select_groups(st, cbt, max_beam, s) : launch_sbeam_select(st, beam, W, s);
            TTB_CHECK(rc == 0, "beam_size * vocabulary too large for the selection kernel");
        }
        {
            Scope sc(e, KC_CACHE_APPEND, s);
            launch_sbeam_cache_update<ActT>(st, e->qkv.as<ActT>(), (long long)Cmax * 3 * E, n_dec, 3 * E, E, kc_cur, vc_cur, kc_next, vc_next,
                                            cache_l_stride, cache_c_stride, s);
        }
        std::swap(kc_cur, kc_next);
        std::swap(vc_cur, vc_next);
        return 0;
    };

    if (!cont) {
        int* hc = e->h_ctrl;
        int W = 1, beam = 1, calls = 0;
        constexpr int sb_lag = 1;   // steps the host stays ahead of the control words it reads (blocking-sync events: the wait sleeps)
        // step 0 on the BOS column (:106), then at most max_len - 2 further columns (:127)
        for (int step = 0; step < max_len - 1; ++step) {
            const int C = B * beam;
            if (int rc = enqueue_step(C, beam, W, C)) return rc;
            // the stop test runs on the device (std_beam.cu: ctrl[2]); the host reads the control words of step - 1 while
            // this step is already enqueued (a step behind the end is a no-op), so the GPU never waits for the host
            TTB_CUDA_OK(cudaMemcpyAsync(hc + 32 + (step & 3) * 8, st.ctrl, 4 * sizeof(int), cudaMemcpyDeviceToHost, s));
            TTB_CUDA_OK(cudaEventRecord(e->poll_ev[step & 3], s));
            std::swap(st.y_cur, st.y_next);
            std::swap(st.score_cur, st.score_next);
            beam = K;
            W += 1;
            if (step >= sb_lag) {
                const int j = (step - sb_lag) & 3;
                TTB_CUDA_OK(cudaEventSynchronize(e->poll_ev[j]));
                if (hc[32 + j * 8 + 2]) break;       // every hypothesis contains EOS (:169)
            }
        }
        // steps that really ran (the host may have enqueued one more, a no-op): width, call count, and the hypothesis set
        // the last real step wrote (step i reads set i & 1 and writes the other one)
        int fin[4] = {};
        TTB_CUDA_OK(cudaMemcpyAsync(fin, st.ctrl, sizeof(fin), cudaMemcpyDeviceToHost, s));
        TTB_CUDA_OK(cudaStreamSynchronize(s));
        calls = fin[3];
        W = 1 + calls;
        st.y_cur = (calls & 1) ? y_set[1] : y_set[0];
        launch_beam_export(st.y_cur, ldw, B * K, W, reinterpret_cast<long long*>(out_dev), s);
        e->launches++;
        float ms = 0.f;
        if (int rc = finish_loop(e, ms)) return rc;
        if (out_width) *out_width = W;
        if (stats) {
            stats->model_calls = calls;
            stats->accepted_tokens = 0;
            stats->produced_tokens = 0;
            stats->unfinished = 0;
            stats->error = 0;
            stats->gpu_launches = (int32_t)(e->launches - launches0);
            stats->gpu_ms = ms;
        }
        return 0;
    }

    // Continuous loop.  Between two steps the host admits the next batches (whole, in list order) while the free slots of
    // the newest word suffice, then enqueues one step with decoder grids sized for the live rows of the word and waits for
    // the word of that step (the closing CTA of the select kernel posts it while the caches are still being re-parented).
    auto admit = [&](int i) -> int {
        if (int rc = sg.encode(e, i, s)) return rc;
        {
            Scope sc(e, KC_MISC, s);
            if (int rc = launch_sbeam_admit(st, cbt, i, cb->bs[i], sg.srclen, reinterpret_cast<long long*>(cb->out[i]), s)) return rc;
        }
        cbt.n_groups = i + 1;
        return sg.scatter(e, cbt.slots, i, s);
    };
    // every batch takes part in at most max_len - 1 steps
    const long long max_steps = (long long)cb->n * (max_len + 1);
    std::vector<int> hist;
    int step = 0, used = 0, live_next = 0;
    while (true) {
        int n = 0;
        if (int rc = sg.admit_fitting(B - used, &n, admit)) return rc;
        used += n;
        live_next += n;   // one BOS hypothesis per query
        if (used == 0) break;   // nothing open and nothing pending (every batch fits the slots)
        TTB_CHECK(step < max_steps, "continuous beam-search loop did not terminate within max_len steps per batch");
        hist.push_back(used);
        st.y_cur = y_set[step & 1]; st.y_next = y_set[(step & 1) ^ 1];
        st.score_cur = score_set[step & 1]; st.score_next = score_set[(step & 1) ^ 1];
        if (int rc = enqueue_step(Cmax, K, 0, std::max(1, std::min(live_next, Cmax)))) return rc;
        unsigned long long w = 0;
        bool arrived = true;
        if (int rc = wait_posted_word(e, s, step + 1, &w, &arrived, false)) return rc;
        TTB_CHECK(arrived, "the control word of the continuous beam-search loop did not arrive");
        used = (int)((w >> 24) & 0xffff);
        live_next = (int)(w & 0xffffff);
        ++step;
    }
    float ms = 0.f;
    if (int rc = finish_loop(e, ms)) return rc;
    int ctrl_end[16] = {};
    TTB_CUDA_OK(cudaMemcpy(ctrl_end, st.ctrl, sizeof(ctrl_end), cudaMemcpyDeviceToHost));
    TTB_CHECK(ctrl_end[SBC_ADM_ERR] == 0, "continuous batching admitted a batch without enough free slots");
    std::vector<SbGroup> groups;
    if (int rc = read_groups(cb, cbt.groups, groups)) return rc;
    e->h_hist = hist;
    for (int i = 0; i < cb->n; ++i) {
        const SbGroup& g = groups[(size_t)i];
        cb->stats[i] = ttb_generate_stats{};
        cb->stats[i].model_calls = g.steps;
        cb->out_width[i] = 1 + g.steps;
    }
    if (stats) {
        *stats = ttb_generate_stats{};
        stats->model_calls = step;
        stats->gpu_launches = (int32_t)(e->launches - launches0);
        stats->gpu_ms = ms;
    }
    return 0;
}

// ---- teacher-forced scoring of given targets (DESIGN.md section 14) ------------------------------------------------------
// Decoder rows per chunk (and encoder rows: source tokens of the chunk): bounds the workspace ensure_work grows to, about
// 10 KB per row at the full architecture.
constexpr int kScoreMaxRows = 32768;

// Whole sources per chunk: the encoder and the cross-attention K/V of every decoder layer once per source, then one decoder
// pass over the K * Lt rows of its candidates (cross-attention groups mapped to their source by kvmap), the vocabulary
// projection reduced per row to (logit of the next target token, soft-max maximum, sum), and one warp per candidate that
// sums the log-probabilities of its scored columns.
template <typename ActT>
static int score_api(ttb_engine* e, const int64_t* src_dev, int B, int Ls, const int64_t* tgt_dev, int K, int Lt, int pad, int eos,
                     float* logp_out, int* ntok_out, float* token_logp_out, cudaStream_t user_stream) {
    const int E = e->E(), H = e->d.num_heads, HD = e->HD(), V = e->d.tgt_vocab_size;
    const int n_dec = (int)e->dec.size();
    cudaStream_t s = e->stream;
    if (int rc = join_caller_stream(e, user_stream)) return rc;
    const int Bc = std::max(1, std::min(B, kScoreMaxRows / std::max(K * Lt, Ls)));
    const long long T_cap = (long long)Bc * K * Lt, TS_cap = (long long)Bc * Ls;
    if (ensure_work<ActT>(e, std::max(T_cap, TS_cap), 1)) return 1;
    if (ensure_encoder<ActT>(e, TS_cap, Bc, TS_cap)) return 1;
    // kvmap [Bc K], then per row: tokv, lmax, lsum and the top-1 / support outputs of classifier_stats that nothing reads
    const size_t G_cap = (size_t)Bc * K, R = (size_t)T_cap;
    if (e->score.ensure((G_cap + 6 * R) * 4)) return 1;
    int* kvmap = e->score.as<int>();
    float* tokv = e->score.as<float>() + G_cap;
    float* lmax = tokv + R;
    float* lsum = lmax + R;
    float* topv = lsum + R;
    int* nkeep = reinterpret_cast<int*>(topv + R);
    int* topi = nkeep + R;
    int* tgt32 = e->tok32.as<int>();
    int* row_tok = e->pred.as<int>();
    int* src32 = e->src32.as<int>();
    int* srclen = e->srclen.as<int>();
    ActT* crosskv = e->crosskv.as<ActT>();
    float* x = e->x.as<float>();
    ActT* xh = Prec<ActT>::lowp ? e->xh.as<ActT>() : nullptr;
    const bool use_fused = Prec<ActT>::lowp && !env_flag("TTB_NO_FUSED_STATS");
    TTB_CUDA_OK(cudaEventRecord(e->t0, s));

    for (int b0 = 0; b0 < B; b0 += Bc) {
        const int nb = std::min(Bc, B - b0), G = nb * K;
        const long long T = (long long)G * Lt, TS = (long long)nb * Ls;
        if (encode_batch<ActT>(e, src_dev + (long long)b0 * Ls, nb, Ls, srclen, crosskv, TS * 2 * E, s)) return 1;
        { Scope sc(e, KC_MISC, s); launch_i64_to_i32(reinterpret_cast<const long long*>(tgt_dev) + (long long)b0 * K * Lt, tgt32, T, s); }
        { Scope sc(e, KC_MISC, s); launch_score_prepare(tgt32, G, Lt, K, kvmap, row_tok, s); }
        { Scope sc(e, KC_EMBED, s); launch_embed_seq<ActT>(tgt32, (int)T, Lt, e->tgt_emb, e->pe, E, x, xh, s); }
        RowCount rows((int)T);
        auto self_attn = [&](int, ActT* qkv, ActT* att) {
            attn(qkv, 3 * E, qkv + E, qkv + 2 * E, 3 * E, att, E, G, nullptr, Lt, Lt, Lt, nullptr, tgt32, Lt, e->d.tgt_pad_token_idx, true, H, HD, s);
        };
        auto cross_attn = [&](int l, ActT* q2, ActT* att) {
            const ActT* kv = crosskv + (long long)l * TS * 2 * E;
            attn(q2, E, kv, kv + E, 2 * E, att, E, G, nullptr, Lt, Ls, Ls, kvmap, src32, Ls, e->d.src_pad_token_idx, false, H, HD, s,
                 nullptr, srclen);
        };
        if (decoder_stack<ActT>(e, rows, 1, 0, self_attn, cross_attn, s)) return 1;
        auto fused = [&](const auto* a) {
            return launch_classifier_stats(a, E, e->classifier.wh, e->classifier.b, rows, V, E, 1, row_tok, tokv, lmax, lsum, nkeep, topv, topi, s);
        };
        auto fallback = [&](const float* lg) { launch_logprob_stats(lg, V, V, row_tok, (int)T, tokv, lmax, lsum, s); };
        if (classifier_head<ActT>(e, rows, use_fused, fused, fallback, e->logits.as<float>(), s)) return 1;
        {
            Scope sc(e, KC_ACCEPT, s);
            launch_score_reduce(tgt32, G, Lt, pad, eos, tokv, lmax, lsum, logp_out + (long long)b0 * K, ntok_out + (long long)b0 * K,
                                token_logp_out ? token_logp_out + (long long)b0 * K * (Lt - 1) : nullptr, s);
        }
        TTB_CUDA_OK(cudaGetLastError());
    }
    float ms = 0.f;
    return finish_loop(e, ms);
}


// Calls f(t, stream) on the engine's device, t a value of the engine's activation type: float on the fp32 path,
// __nv_bfloat16 on the bf16 path.
template <typename F>
static int with_act_type(ttb_engine* e, void* stream, F f) {
    TTB_CUDA_OK(cudaSetDevice(e->device));
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    return e->d.precision == TTB_PRECISION_FP32 ? f(float{}, s) : f(__nv_bfloat16{}, s);
}

// Argument rules of the C entry points, each in the order the reference asserts them.  The *_generate_batches entries pass
// Ls = 0: their source lengths are checked batch by batch.
static int check_draft_tokens(int n_drafts, int pad, int eos, int replace) {   // drafting.py:38-42
    TTB_CHECK(n_drafts > 0, "The number of drafts must be greater than 0");
    TTB_CHECK(pad != replace, "The pad token and the replace token must be different");
    TTB_CHECK(eos != replace, "The eos token and the replace token must be different");
    TTB_CHECK(eos != pad, "The eos token and the pad token must be different");
    return 0;
}
static int check_beam(const ttb_engine* e, int Ls, int max_len, int beam_size) {
    TTB_CHECK(max_len > 1 && beam_size > 0, "max_len must be greater than 1 and beam_size greater than 0");
    TTB_CHECK(beam_size <= e->d.tgt_vocab_size, "beam_size larger than the vocabulary (the reference's first topk fails as well)");
    TTB_CHECK(Ls <= e->d.max_positions && max_len + 2 <= e->d.max_positions, "sequence longer than the positional table");
    return 0;
}
static int check_beam_speculative(const ttb_engine* e, int Ls, int max_len, int n_best, int n_drafts, int pad, int eos, int c_token) {
    TTB_CHECK(n_best >= 1 && n_best <= 32, "n_best must be in [1, 32]");
    if (int rc = check_draft_tokens(n_drafts, pad, eos, c_token)) return rc;
    TTB_CHECK(Ls <= e->d.max_positions && max_len + 210 <= e->d.max_positions, "sequence longer than the positional table");
    TTB_CHECK(e->d.tgt_vocab_size <= 1024, "vocabularies above 1024 tokens are not supported by the beam statistics kernel");
    return 0;
}

// The batches of a *_generate_batches call, batch by batch: pointers, B_i > 0 and Ls_i >= min_ls, then B_i <= slots and
// Ls_i <= max_positions, that pair in the order of `table_first`; with `smart`, last, the Ls_i > 5 that the window library
// of smart drafts needs.  *Ls_max: the longest source, at least min_ls.
static int check_batch_list(const ttb_engine* e, int n, const int64_t* const* src, const int32_t* bs, const int32_t* ls, int64_t* const* out,
                            int slots, int min_ls, bool table_first, bool smart, int* Ls_max) {
    *Ls_max = min_ls;
    for (int i = 0; i < n; ++i) {
        TTB_CHECK(src[i] && out[i] && bs[i] > 0 && ls[i] >= min_ls, "bad arguments");
        if (table_first) TTB_CHECK(ls[i] <= e->d.max_positions, "sequence longer than the positional table");
        TTB_CHECK(bs[i] <= slots, "slots must be at least the largest batch size");
        if (!table_first) TTB_CHECK(ls[i] <= e->d.max_positions, "sequence longer than the positional table");
        if (smart) TTB_CHECK(ls[i] > 5, "The number of drafts must be greater than 0");
        *Ls_max = std::max(*Ls_max, (int)ls[i]);
    }
    return 0;
}
static int check_greedy(const ttb_engine* e, int Ls, int max_len) {
    TTB_CHECK(max_len > 1, "bad arguments");
    TTB_CHECK(Ls <= e->d.max_positions && max_len + 2 <= e->d.max_positions, "sequence longer than the positional table");
    return 0;
}

}  // namespace ttb

// =================================================================================================
extern "C" {

int ttb_abi_version(void) { return TTB_ABI_VERSION; }
const char* ttb_last_error(void) { return g_last_error.c_str(); }

int ttb_device_check(int device) {
    int n = 0;
    TTB_CUDA_OK(cudaGetDeviceCount(&n));
    TTB_CHECK(device >= 0 && device < n, "no such CUDA device");
    cudaDeviceProp p{};
    TTB_CUDA_OK(cudaGetDeviceProperties(&p, device));
    TTB_CHECK(p.major == 10, "libttb200 is built for sm_100a (B200) only");
    return 0;
}

int ttb_engine_create(const ttb_model_desc* desc, int device, ttb_engine** out) {
    TTB_CHECK(desc && out, "null argument");
    TTB_CHECK(desc->embedding_dim % desc->num_heads == 0, "embedding_dim must be divisible by num_heads");
    const int hd = desc->embedding_dim / desc->num_heads;
    TTB_CHECK(hd == 16 || hd == 32 || hd == 64, "head_dim must be 16, 32 or 64");
    TTB_CHECK(desc->embedding_dim % 16 == 0 && desc->feedforward_dim % 16 == 0, "embedding_dim and feedforward_dim must be multiples of 16");
    TTB_CHECK(desc->embedding_dim <= 1024, "embedding_dim above 1024 is not supported");
    if (desc->precision == TTB_PRECISION_BF16)
        TTB_CHECK(desc->embedding_dim % 64 == 0 && desc->feedforward_dim % 64 == 0, "bf16 path needs embedding_dim and feedforward_dim multiples of 64");
    if (int rc = ttb_device_check(device)) return rc;
    TTB_CUDA_OK(cudaSetDevice(device));
    ttb_engine* e = new ttb_engine();
    e->d = *desc;
    e->device = device;
    if (register_params(e)) { ttb_engine_destroy(e); return 1; }
    TTB_CUDA_OK(cudaMallocHost(&e->h_ctrl, 4 * CTRL_COUNT * sizeof(int)));
    // blocking sync: the decoding loop polls one graph (four iterations, ~1.2 ms) behind the GPU, so a sleeping host thread
    // costs nothing, and several engines per GPU x several ranks per box do not each burn a core spinning
    for (auto& ev : e->poll_ev) TTB_CUDA_OK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming | cudaEventBlockingSync));
    TTB_CUDA_OK(cudaEventCreate(&e->t0));
    TTB_CUDA_OK(cudaEventCreate(&e->t1));
    TTB_CUDA_OK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    TTB_CUDA_OK(cudaEventCreateWithFlags(&e->join_ev, cudaEventDisableTiming));
    *out = e;
    return 0;
}

void ttb_engine_destroy(ttb_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    for (auto& kv : e->params) {
        if (kv.second.dev) cudaFree(kv.second.dev);
        if (kv.second.devh) cudaFree(kv.second.devh);
    }
    DevBuf* bufs[] = {&e->x, &e->xh, &e->y, &e->qkv, &e->att, &e->q2, &e->hid, &e->logits, &e->tok32, &e->keytok32, &e->pred,
                      &e->src32, &e->memory, &e->memh, &e->crosskv, &e->kcache, &e->vcache, &e->drafts, &e->gen, &e->front,
                      &e->active, &e->ctrl, &e->sel, &e->out64, &e->hist, &e->beam, &e->srclen, &e->desc, &e->kcache2, &e->vcache2,
                      &e->cb, &e->cb_work, &e->score, &e->smp};
    for (DevBuf* b : bufs) b->release();
    if (e->h_ctrl) cudaFreeHost(e->h_ctrl);
    for (auto& ev : e->poll_ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : e->prof.pool) cudaEventDestroy(ev);
    for (auto& gb : e->graph_exec) for (auto& g : gb) if (g) cudaGraphExecDestroy(g);
    if (e->stream) cudaStreamDestroy(e->stream);
    if (e->join_ev) cudaEventDestroy(e->join_ev);
    if (e->t0) cudaEventDestroy(e->t0);
    if (e->t1) cudaEventDestroy(e->t1);
    delete e;
}

int ttb_engine_set_param(ttb_engine* e, const char* name, const float* data, int64_t numel) {
    TTB_CHECK(e && name && data, "null argument");
    std::string n(name);
    if (n.rfind("model.", 0) == 0) n = n.substr(6);
    auto it = e->params.find(n);
    TTB_CHECK(it != e->params.end(), std::string("unexpected parameter name: ") + n);
    TTB_CHECK(it->second.numel == numel, std::string("size mismatch for ") + n + ": expected " +
              std::to_string(it->second.numel) + " elements, got " + std::to_string(numel));
    TTB_CUDA_OK(cudaSetDevice(e->device));
    TTB_CUDA_OK(cudaMemcpy(it->second.dev, data, (size_t)numel * sizeof(float), cudaMemcpyDefault));
    it->second.set = true;
    e->finalized = false;
    return 0;
}

int ttb_engine_finalize(ttb_engine* e) {
    TTB_CHECK(e, "null engine");
    TTB_CUDA_OK(cudaSetDevice(e->device));
    for (auto& kv : e->params) TTB_CHECK(kv.second.set, std::string("missing parameter: ") + kv.first);
    if (e->d.precision == TTB_PRECISION_BF16) {
        for (auto& kv : e->params) {
            Param& p = kv.second;
            if (!p.is_gemm_weight) continue;
            if (!p.devh) TTB_CUDA_OK(cudaMalloc(&p.devh, (size_t)p.numel * sizeof(__nv_bfloat16)));
            launch_f32_to_bf16(p.dev, p.devh, p.numel, 0);
        }
        TTB_CUDA_OK(cudaDeviceSynchronize());
    }
    const int E = e->d.embedding_dim, F = e->d.feedforward_dim;
    e->enc.clear();
    e->dec.clear();
    for (int i = 0; i < e->d.num_encoder_layers; ++i) {
        std::string p = "transformer.encoder.layers." + std::to_string(i);
        EncLayer L;
        L.in_proj = make_lin(e, p + ".self_attn.in_proj_weight", p + ".self_attn.in_proj_bias", 3 * E, E);
        L.out_proj = make_lin(e, p + ".self_attn.out_proj.weight", p + ".self_attn.out_proj.bias", E, E);
        L.ff1 = make_lin(e, p + ".linear1.weight", p + ".linear1.bias", F, E);
        L.ff2 = make_lin(e, p + ".linear2.weight", p + ".linear2.bias", E, F);
        L.n1 = make_norm(e, p + ".norm1");
        L.n2 = make_norm(e, p + ".norm2");
        e->enc.push_back(L);
    }
    for (int i = 0; i < e->d.num_decoder_layers; ++i) {
        std::string p = "transformer.decoder.layers." + std::to_string(i);
        DecLayer L;
        L.self_in = make_lin(e, p + ".self_attn.in_proj_weight", p + ".self_attn.in_proj_bias", 3 * E, E);
        L.self_out = make_lin(e, p + ".self_attn.out_proj.weight", p + ".self_attn.out_proj.bias", E, E);
        L.cross_in = make_lin(e, p + ".multihead_attn.in_proj_weight", p + ".multihead_attn.in_proj_bias", 3 * E, E);
        L.cross_out = make_lin(e, p + ".multihead_attn.out_proj.weight", p + ".multihead_attn.out_proj.bias", E, E);
        L.ff1 = make_lin(e, p + ".linear1.weight", p + ".linear1.bias", F, E);
        L.ff2 = make_lin(e, p + ".linear2.weight", p + ".linear2.bias", E, F);
        L.n1 = make_norm(e, p + ".norm1");
        L.n2 = make_norm(e, p + ".norm2");
        L.n3 = make_norm(e, p + ".norm3");
        e->dec.push_back(L);
    }
    e->enc_norm = make_norm(e, "transformer.encoder.norm");
    e->dec_norm = make_norm(e, "transformer.decoder.norm");
    e->classifier = make_lin(e, "next_token_classifier.weight", "next_token_classifier.bias", e->d.tgt_vocab_size, E);
    e->src_emb = e->params["src_token_featurizer.embedding.weight"].dev;
    e->tgt_emb = e->params["tgt_token_featurizer.embedding.weight"].dev;
    e->pe = e->params["positional_encoding.pe"].dev;
    e->finalized = true;
    return 0;
}

int ttb_make_drafts(const int64_t* src_dev, int64_t src_ld, int32_t B, int32_t L, int32_t draft_len,
                    int32_t n_drafts, int32_t min_draft_len, int32_t max_draft_len, int32_t eos,
                    int32_t pad, int32_t replace, int64_t* out_dev, int32_t* d_out, void* stream) {
    // same argument checks, same order, as drafting.py:38-42 (the wrappers raise AssertionError)
    TTB_CHECK(n_drafts > 0, "The number of drafts must be greater than 0");
    TTB_CHECK(min_draft_len <= max_draft_len, "The minimum draft length must not be greater than the maximum draft length");
    TTB_CHECK(pad != replace, "The pad token and the replace token must be different");
    TTB_CHECK(eos != replace, "The eos token and the replace token must be different");
    TTB_CHECK(eos != pad, "The eos token and the pad token must be different");
    TTB_CHECK(src_dev && out_dev && B > 0 && L > 0, "bad source tensor");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    const int D = std::min(std::max(min_draft_len, draft_len), max_draft_len);
    if (d_out) *d_out = D;
    int *src32 = nullptr, *out32 = nullptr;
    TTB_CUDA_OK(cudaMallocAsync(&src32, (size_t)B * L * sizeof(int), s));
    TTB_CUDA_OK(cudaMallocAsync(&out32, (size_t)B * n_drafts * D * sizeof(int), s));
    if (src_ld == L) {
        launch_i64_to_i32(reinterpret_cast<const long long*>(src_dev), src32, (long long)B * L, s);
    } else {
        for (int b = 0; b < B; ++b)
            launch_i64_to_i32(reinterpret_cast<const long long*>(src_dev) + (long long)b * src_ld, src32 + (long long)b * L, L, s);
    }
    launch_make_drafts(src32, L, B, L, D, n_drafts, eos, pad, replace, out32, s);
    launch_i32_to_i64(out32, reinterpret_cast<long long*>(out_dev), (long long)B * n_drafts * D, s);
    TTB_CUDA_OK(cudaFreeAsync(src32, s));
    TTB_CUDA_OK(cudaFreeAsync(out32, s));
    TTB_CUDA_OK(cudaGetLastError());
    return 0;
}

// Every exit of a decoding loop leaves the engine's stream drained: kernels still queued there write to the caller's
// `out` / `trace` buffers, which the caller is free to release as soon as the call returns (error exits included).
static int drained(ttb_engine* e, int rc) {
    if (rc != 0 && e->stream) {
        const std::string keep = g_last_error;
        cudaStreamSynchronize(e->stream);
        (void)cudaGetLastError();
        g_last_error = keep;
    }
    return rc;
}

int ttb_encode_src(ttb_engine* e, const int64_t* src_dev, const uint8_t* src_pad_mask_dev, int32_t B,
                   int32_t Ls, float* memory_out_dev, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(src_dev && memory_out_dev && B > 0 && Ls > 0, "bad arguments");
    TTB_CHECK(Ls <= e->d.max_positions, "source longer than the positional table");
    return with_act_type(e, stream, [&](auto t, cudaStream_t s) { return encode_api<decltype(t)>(e, src_dev, src_pad_mask_dev, B, Ls, memory_out_dev, s); });
}

int ttb_decode_tgt(ttb_engine* e, const int64_t* tgt_dev, int32_t B, int32_t Lt, const float* memory_dev,
                   const uint8_t* memory_pad_mask_dev, int32_t Ls, float* logits_out_dev, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(tgt_dev && memory_dev && memory_pad_mask_dev && logits_out_dev && B > 0 && Lt > 0 && Ls > 0, "bad arguments");
    TTB_CHECK(Lt <= e->d.max_positions, "target longer than the positional table");
    return with_act_type(e, stream, [&](auto t, cudaStream_t s) { return decode_api<decltype(t)>(e, tgt_dev, B, Lt, memory_dev, memory_pad_mask_dev, Ls, logits_out_dev, s); });
}

int ttb_greedy_speculative_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls,
                                    int32_t max_len, int32_t draft_len, int32_t n_drafts, int32_t pad_token,
                                    int32_t bos_token, int32_t eos_token, int32_t replace_token,
                                    int32_t tie_break, int64_t* out_dev, int32_t* trace_dev,
                                    ttb_generate_stats* stats, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(src_dev && out_dev && B > 0 && Ls > 1 && max_len > 1, "bad arguments");
    if (int rc = check_draft_tokens(n_drafts, pad_token, eos_token, replace_token)) return rc;
    TTB_CHECK(Ls <= e->d.max_positions && max_len + draft_len + 2 <= e->d.max_positions, "sequence longer than the positional table");
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return greedy_api<decltype(t)>(e, src_dev, B, Ls, max_len, draft_len, n_drafts, pad_token, bos_token, eos_token, replace_token, tie_break,
                                       out_dev, trace_dev, stats, s, GreedyMode::speculative);
    }));
}

int ttb_greedy_speculative_generate_batches(ttb_engine* e, int32_t n_batches, const int64_t* const* src_devs, const int32_t* batch_sizes,
                                            const int32_t* src_lens, int32_t slots, int32_t max_len, int32_t draft_len, int32_t n_drafts,
                                            int32_t pad_token, int32_t bos_token, int32_t eos_token, int32_t replace_token, int32_t tie_break,
                                            int64_t* const* out_devs, int32_t* const* trace_devs, ttb_generate_stats* stats,
                                            ttb_generate_stats* total, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(n_batches >= 0 && max_len > 1 && slots > 0, "bad arguments");
    TTB_CHECK(n_batches == 0 || (src_devs && batch_sizes && src_lens && out_devs && stats), "bad arguments");
    if (int rc = check_draft_tokens(n_drafts, pad_token, eos_token, replace_token)) return rc;
    TTB_CHECK(max_len + draft_len + 2 <= e->d.max_positions, "sequence longer than the positional table");
    int Ls_max = 0;
    if (int rc = check_batch_list(e, n_batches, src_devs, batch_sizes, src_lens, out_devs, slots, 2, false, false, &Ls_max)) return rc;
    if (total) *total = ttb_generate_stats{};
    if (n_batches == 0) return 0;
    const BatchList cb{n_batches, src_devs, batch_sizes, src_lens, out_devs, stats, nullptr, trace_devs, nullptr, nullptr};
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return greedy_api<decltype(t)>(e, nullptr, slots, Ls_max, max_len, draft_len, n_drafts, pad_token, bos_token, eos_token, replace_token,
                                       tie_break, nullptr, nullptr, total, s, GreedyMode::speculative, &cb);
    }));
}

int ttb_greedy_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, int32_t max_len, int32_t pad_token,
                        int32_t bos_token, int32_t eos_token, int64_t* out_dev, ttb_generate_stats* stats, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(src_dev && out_dev && B > 0 && Ls > 0, "bad arguments");
    if (int rc = check_greedy(e, Ls, max_len)) return rc;
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return greedy_api<decltype(t)>(e, src_dev, B, Ls, max_len, 0, 1, pad_token, bos_token, eos_token, -1, 1, out_dev, nullptr, stats, s,
                                       GreedyMode::standard);
    }));
}

int ttb_greedy_generate_batches(ttb_engine* e, int32_t n_batches, const int64_t* const* src_devs, const int32_t* batch_sizes,
                                const int32_t* src_lens, int32_t slots, int32_t max_len, int32_t pad_token, int32_t bos_token,
                                int32_t eos_token, int64_t* const* out_devs, ttb_generate_stats* stats, ttb_generate_stats* total,
                                void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(n_batches >= 0 && slots > 0, "bad arguments");
    TTB_CHECK(n_batches == 0 || (src_devs && batch_sizes && src_lens && out_devs && stats), "bad arguments");
    // the rules of ttb_greedy_generate, in its order, before any device work
    for (int i = 0; i < n_batches; ++i) TTB_CHECK(src_devs[i] && out_devs[i] && batch_sizes[i] > 0 && src_lens[i] > 0, "bad arguments");
    if (int rc = check_greedy(e, 0, max_len)) return rc;
    int Ls_max = 0;
    if (int rc = check_batch_list(e, n_batches, src_devs, batch_sizes, src_lens, out_devs, slots, 1, true, false, &Ls_max)) return rc;
    TTB_CHECK(slots <= 2048, "continuous batching supports at most 2048 slots");
    if (total) *total = ttb_generate_stats{};
    if (n_batches == 0) return 0;
    const BatchList cb{n_batches, src_devs, batch_sizes, src_lens, out_devs, stats, nullptr, nullptr, nullptr, nullptr};
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return greedy_api<decltype(t)>(e, nullptr, slots, Ls_max, max_len, 0, 1, pad_token, bos_token, eos_token, -1, 1, nullptr, nullptr, total, s,
                                       GreedyMode::standard, &cb);
    }));
}

int ttb_sample_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, int32_t max_len, int32_t n_samples, float temperature,
                        int32_t top_k, uint64_t seed, int32_t pad_token, int32_t bos_token, int32_t eos_token, int64_t* out_dev,
                        ttb_generate_stats* stats, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(src_dev && out_dev && B > 0 && Ls > 0, "bad arguments");
    TTB_CHECK(n_samples >= 1, "n_samples must be at least 1");
    TTB_CHECK((long long)B * n_samples <= 2048, "B * n_samples above 2048 sample slots");
    TTB_CHECK(std::isfinite(temperature) && temperature > 0.f, "temperature must be finite and greater than 0");
    TTB_CHECK(top_k >= 0 && top_k <= e->d.tgt_vocab_size, "top_k must lie in [0, vocabulary size]");
    TTB_CHECK(max_len >= 2, "max_len must be at least 2");
    TTB_CHECK(pad_token != eos_token, "The eos token and the pad token must be different");
    TTB_CHECK(Ls <= e->d.max_positions && max_len + 2 <= e->d.max_positions, "sequence longer than the positional table");
    const SampleCfg smp{n_samples, temperature, top_k, (unsigned long long)seed};
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return greedy_api<decltype(t)>(e, src_dev, B * n_samples, Ls, max_len, 0, 1, pad_token, bos_token, eos_token, -1, 1, out_dev, nullptr,
                                       stats, s, GreedyMode::sampling, nullptr, smp);
    }));
}

int ttb_beam_search_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, int32_t max_len, int32_t beam_size,
                             int32_t pad_token, int32_t bos_token, int32_t eos_token, int64_t* out_dev, int32_t* out_width,
                             ttb_generate_stats* stats, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(src_dev && out_dev && B > 0 && Ls > 0, "bad arguments");
    if (int rc = check_beam(e, Ls, max_len, beam_size)) return rc;
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return std_beam_api<decltype(t)>(e, src_dev, B, Ls, max_len, beam_size, pad_token, bos_token, eos_token, out_dev, out_width, stats, s);
    }));
}

int ttb_beam_search_generate_batches(ttb_engine* e, int32_t n_batches, const int64_t* const* src_devs, const int32_t* batch_sizes,
                                     const int32_t* src_lens, int32_t slots, int32_t max_len, int32_t beam_size, int32_t pad_token,
                                     int32_t bos_token, int32_t eos_token, int64_t* const* out_devs, int32_t* out_widths,
                                     ttb_generate_stats* stats, ttb_generate_stats* total, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(n_batches >= 0 && slots > 0, "bad arguments");
    TTB_CHECK(n_batches == 0 || (src_devs && batch_sizes && src_lens && out_devs && out_widths && stats), "bad arguments");
    for (int i = 0; i < n_batches; ++i) TTB_CHECK(src_devs[i] && out_devs[i] && batch_sizes[i] > 0 && src_lens[i] > 0, "bad arguments");
    // the rules of ttb_beam_search_generate, in its order, before any device work
    if (int rc = check_beam(e, 0, max_len, beam_size)) return rc;
    int Ls_max = 0;
    if (int rc = check_batch_list(e, n_batches, src_devs, batch_sizes, src_lens, out_devs, slots, 1, true, false, &Ls_max)) return rc;
    // generate() fails in its first step (one hypothesis per query) or its second (beam_size of them)
    TTB_CHECK(sbeam_select_fits(1, e->d.tgt_vocab_size) && (max_len == 2 || sbeam_select_fits(beam_size, e->d.tgt_vocab_size)),
              "beam_size * vocabulary too large for the selection kernel");
    TTB_CHECK(slots <= 65535 && (long long)slots * beam_size < (1 << 24), "continuous batching supports at most 65535 slots and 2^24 - 1 hypotheses");
    if (total) *total = ttb_generate_stats{};
    if (n_batches == 0) return 0;
    const BatchList cb{n_batches, src_devs, batch_sizes, src_lens, out_devs, stats, out_widths, nullptr, nullptr, nullptr};
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return std_beam_api<decltype(t)>(e, nullptr, slots, Ls_max, max_len, beam_size, pad_token, bos_token, eos_token, nullptr, nullptr, total,
                                         s, &cb);
    }));
}

int ttb_beam_speculative_generate(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, int32_t max_len,
                                  int32_t n_best, int32_t draft_len, int32_t n_drafts, int32_t smart_drafts_mode, int32_t pad_token,
                                  int32_t bos_token, int32_t eos_token, int32_t c_token, int32_t tie_break, int64_t* out_dev,
                                  int32_t* out_width, int32_t* trace_nacc_dev, int32_t* trace_pick_dev, ttb_generate_stats* stats,
                                  void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(src_dev && out_dev && B > 0 && Ls > 1 && max_len > 2, "bad arguments");
    if (int rc = check_beam_speculative(e, Ls, max_len, n_best, n_drafts, pad_token, eos_token, c_token)) return rc;
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return beam_api<decltype(t)>(e, src_dev, B, Ls, max_len, n_best, draft_len, n_drafts, pad_token, bos_token, eos_token, c_token, tie_break,
                                     out_dev, out_width, trace_nacc_dev, trace_pick_dev, stats, s, smart_drafts_mode != 0);
    }));
}

int ttb_beam_speculative_generate_batches(ttb_engine* e, int32_t n_batches, const int64_t* const* src_devs, const int32_t* batch_sizes,
                                          const int32_t* src_lens, int32_t slots, int32_t max_len, int32_t n_best, int32_t draft_len,
                                          int32_t n_drafts, int32_t smart_drafts_mode, int32_t pad_token, int32_t bos_token, int32_t eos_token,
                                          int32_t c_token, int32_t tie_break, int64_t* const* out_devs, int32_t* out_widths,
                                          int32_t* const* trace_nacc_devs, int32_t* const* trace_pick_devs, ttb_generate_stats* stats,
                                          ttb_generate_stats* total, void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(n_batches >= 0 && max_len > 2 && slots > 0, "bad arguments");
    TTB_CHECK(n_batches == 0 || (src_devs && batch_sizes && src_lens && out_devs && out_widths && stats), "bad arguments");
    if (int rc = check_beam_speculative(e, 0, max_len, n_best, n_drafts, pad_token, eos_token, c_token)) return rc;
    int Ls_max = 0;
    if (int rc = check_batch_list(e, n_batches, src_devs, batch_sizes, src_lens, out_devs, slots, 2, false, smart_drafts_mode != 0, &Ls_max))
        return rc;
    if (total) *total = ttb_generate_stats{};
    if (n_batches == 0) return 0;
    const BatchList cb{n_batches, src_devs, batch_sizes, src_lens, out_devs, stats, out_widths, nullptr, trace_nacc_devs, trace_pick_devs};
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return beam_api<decltype(t)>(e, nullptr, slots, Ls_max, max_len, n_best, draft_len, n_drafts, pad_token, bos_token, eos_token, c_token,
                                     tie_break, nullptr, nullptr, nullptr, nullptr, total, s, smart_drafts_mode != 0, &cb);
    }));
}

int ttb_score_targets(ttb_engine* e, const int64_t* src_dev, int32_t B, int32_t Ls, const int64_t* tgt_dev, int32_t K, int32_t Lt,
                      int32_t pad_token, int32_t eos_token, float* logp_out_dev, int32_t* ntok_out_dev, float* token_logp_out_dev,
                      void* stream) {
    TTB_CHECK(e && e->finalized, "engine not finalized");
    TTB_CHECK(src_dev && tgt_dev && logp_out_dev && ntok_out_dev, "bad arguments");
    TTB_CHECK(B > 0 && K > 0 && Ls > 0 && Lt > 1, "bad arguments: B, K, Ls >= 1 and Lt >= 2");
    TTB_CHECK(Ls <= e->d.max_positions && Lt <= e->d.max_positions, "sequence longer than the positional table");
    TTB_CHECK((long long)K * Lt <= kScoreMaxRows, "K * Lt above 32768 decoder rows per source");
    TTB_CHECK(pad_token != eos_token, "The eos token and the pad token must be different");
    return drained(e, with_act_type(e, stream, [&](auto t, cudaStream_t s) {
        return score_api<decltype(t)>(e, src_dev, B, Ls, tgt_dev, K, Lt, pad_token, eos_token, logp_out_dev, ntok_out_dev, token_logp_out_dev, s);
    }));
}

int ttb_kernel_class_count(void) { return KC_COUNT; }
const char* ttb_kernel_class_name(int32_t id) { return (id >= 0 && id < KC_COUNT) ? kKcNames[id] : ""; }

int ttb_engine_set_profiling(ttb_engine* e, uint32_t class_mask) {
    TTB_CHECK(e, "null engine");
    e->prof.mask = class_mask;
    for (int i = 0; i < KC_COUNT; ++i) { e->prof.ms[i] = 0.0; e->prof.n[i] = 0; }
    return 0;
}

int ttb_engine_get_profile(ttb_engine* e, int32_t n_classes, double* ms_out, int64_t* launches_out) {
    TTB_CHECK(e && ms_out && launches_out, "null argument");
    for (int i = 0; i < n_classes && i < KC_COUNT; ++i) { ms_out[i] = e->prof.ms[i]; launches_out[i] = e->prof.n[i]; }
    return 0;
}

int ttb_engine_get_history(ttb_engine* e, int32_t* live_queries_out, int32_t capacity) {
    TTB_CHECK(e && live_queries_out, "null argument");
    const int n = (int)e->h_hist.size();
    for (int i = 0; i < n && i < capacity; ++i) live_queries_out[i] = e->h_hist[i];
    return n;
}

int ttb_engine_get_draft_history(ttb_engine* e, int32_t* call_dl_out, int32_t* min_dl_out, int32_t capacity) {
    TTB_CHECK(e && call_dl_out && min_dl_out, "null argument");
    const int n = (int)e->h_dl.size();
    for (int i = 0; i < n && i < capacity; ++i) { call_dl_out[i] = e->h_dl[i]; min_dl_out[i] = e->h_dl_min[i]; }
    return n;
}

int ttb_gemm(int32_t precision, const void* A_dev, const void* W_dev, const float* bias_dev, float* C_dev,
             int32_t M, int32_t N, int32_t K, int32_t relu, void* stream) {
    TTB_CHECK(A_dev && W_dev && C_dev && M > 0 && N > 0 && K > 0, "bad arguments");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (precision == TTB_PRECISION_FP32) {
        TTB_CHECK(K % 16 == 0, "K must be a multiple of 16");
        launch_gemm_f32<float>(static_cast<const float*>(A_dev), K, static_cast<const float*>(W_dev), bias_dev, C_dev, N,
                               RowCount(M), N, K, relu != 0, s);
    } else {
        TTB_CHECK(K % 64 == 0, "K must be a multiple of 64");
        if (int rc = launch_gemm_bf16_tc<float>(static_cast<const __nv_bfloat16*>(A_dev), K, static_cast<const __nv_bfloat16*>(W_dev),
                                                bias_dev, C_dev, N, RowCount(M), N, K, relu != 0, s))
            return rc;
    }
    TTB_CUDA_OK(cudaGetLastError());
    return 0;
}

int ttb_gemm_bf16_out(const void* A_dev, const void* W_dev, const float* bias_dev, void* C_dev, int32_t M, int32_t N, int32_t K,
                      int32_t relu, void* stream) {
    TTB_CHECK(A_dev && W_dev && C_dev && M > 0 && N > 0 && K > 0, "bad arguments");
    TTB_CHECK(K % 64 == 0, "K must be a multiple of 64");
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (int rc = launch_gemm_bf16_tc<__nv_bfloat16>(static_cast<const __nv_bfloat16*>(A_dev), K, static_cast<const __nv_bfloat16*>(W_dev), bias_dev,
                                                    static_cast<__nv_bfloat16*>(C_dev), N, RowCount(M), N, K, relu != 0, s))
        return rc;
    TTB_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
