// Tensor-core attention for the bf16 path (short sequences, head_dim 16/32/64).
//
// One CTA per (group, head, block of 256 query rows).  A warp owns 32 query rows (two m16 tiles): Q
// fragments live in registers; the K/V rows the CTA needs are staged in shared memory as bf16 (row
// pitch head_dim + 8 elements -> conflict-free ldmatrix) with cp.async — for the sequence lengths of
// this model (<= 224 shared keys, <= 288 private keys) ALL of them in one round, i.e. one global
// memory latency and one barrier per CTA instead of one per 64-key tile.  S = Q K^T and O += P V run
// on mma.sync.m16n8k16 (bf16 in, fp32 accumulate), the softmax is the usual online (flash) formulation
// in fp32 with exp2.  P is rounded to bf16 for the second product (precision contract, DESIGN.md §5).
//
// Key sources
//   phase A ("shared" keys): all queries of the group see the same keys — encoder self-attention,
//            cross-attention over the cached source memory, the accepted-prefix KV cache of
//            speculative decoding, or (causal) the whole target of decode_tgt;
//   phase B ("private" keys, speculative self-attention only): the freshly projected K/V of the
//            draft row a query belongs to, block-diagonal + causal inside the (D+1)-token row.
// Masking mirrors torch: masked keys get probability 0, a fully masked query row yields NaN.
#include "kernels.cuh"

namespace ttb {
namespace amma {

constexpr int WARPS = 8, THREADS = WARPS * 32, ROWS_PER_WARP = 32, ROWS_PER_CTA = WARPS * ROWS_PER_WARP;
constexpr int KTA = 224;  // shared keys staged per round (covers max_len + draft_len + 2 = 212 and sources <= 224)
constexpr int KTB = 288;  // private keys staged per round (256 query rows + one draft row of look-back)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x2(uint32_t& r0, uint32_t& r1, uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];\n" : "=r"(r0), "=r"(r1) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
__device__ __forceinline__ float fast_exp2(float x) {   // ex2.approx: exact 0 for -inf, 1 for 0
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void ldsm_x4(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
struct NoMask { __device__ __forceinline__ bool operator()(int, int) const { return false; } };
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
}

struct Params {
    const __nv_bfloat16* q; int q_ld;            // query rows: token (g*Lq + i), head offset h*HD
    const __nv_bfloat16* k; const __nv_bfloat16* v; int kv_ld;   // shared keys: row kvg*kv_group_stride + j
    __nv_bfloat16* out; int out_ld;
    const int* n_groups_dev;
    int Lq, Lk;                                  // Lk ignored when spec (prefix length = front[b])
    long long kv_group_stride;
    const int* kvmap;
    const int* key_tok; int key_tok_stride; int pad_id;
    int causal;
    const int* lk_dev;                           // when set: Lk = kv_group_stride = key_tok_stride = *lk_dev (graph replay)
    const int* lk_group;                         // optional [kv group]: keys behind it are padding (never unmasked)
    const int4* desc;                            // optional per-slot descriptor {kv group, front, token at front, key bound}
    float scale_log2e;
    // speculative self-attention
    int spec;
    const int* active; const int* front; const int* gen; int gen_ld;
    const __nv_bfloat16* newk; const __nv_bfloat16* newv; int new_ld;   // new K/V rows: token (g*Lq + r)
    int row_len;                                 // D + 1
};

// Staged keys: k/v rows of PITCH = HD + 8 elements ((HD+8)*2 bytes keeps 16-byte row alignment),
// bias = 0 or -inf per staged key.
template <int HD>
struct Tile {
    static constexpr int PITCH = HD + 8;
    __nv_bfloat16* k;
    __nv_bfloat16* v;
    float* bias;
};
template <int HD> constexpr int smem_bytes() { return (KTA + KTB) * (HD + 8) * 2 * 2 + (KTA + KTB) * 4; }

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

// Stage rows [row0, nk) of a K/V source into a tile (asynchronously) and zero rows [max(row0, nk), nfill).
template <int HD>
__device__ __forceinline__ void stage_rows(const Tile<HD>& t, const __nv_bfloat16* ksrc, const __nv_bfloat16* vsrc, int ld, int nk, int nfill,
                                           int row0 = 0) {
    constexpr int CH = HD / 8, PITCH = Tile<HD>::PITCH;
    for (int idx = row0 * CH + threadIdx.x; idx < nfill * CH; idx += THREADS) {
        const int j = idx / CH, c = idx % CH;
        __nv_bfloat16* kd = t.k + j * PITCH + c * 8;
        __nv_bfloat16* vd = t.v + j * PITCH + c * 8;
        if (j < nk) {
            cp_async16(kd, ksrc + (long long)j * ld + c * 8);
            cp_async16(vd, vsrc + (long long)j * ld + c * 8);
        } else {
            *reinterpret_cast<uint4*>(kd) = make_uint4(0, 0, 0, 0);
            *reinterpret_cast<uint4*>(vd) = make_uint4(0, 0, 0, 0);
        }
    }
}

// One 32-key sub-block (keys kb..kb+31 of the staged tile) for one m16 tile of queries.
//   MaskFn(row_sel, col) -> true when the (query row, key column) pair is masked; row_sel 0 = row A
//   (lane/4), 1 = row B (+8); col = 0..31 inside the sub-block.
template <int HD, typename MaskFn>
__device__ __forceinline__ void process_block(const Tile<HD>& t, int kb, const uint32_t (&qa)[HD / 16][4], float (&o)[HD / 8][4],
                                              float& mA, float& mB, float& lA, float& lB, float scale_log2e, int lane, MaskFn masked) {
    float s[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        // matrices: keys kb+nt*8..+7 x dims {0..7 | 8..15 | 16..23 | 24..31} (+32 per x4): lanes 8m..8m+7 give
        // the row addresses of matrix m, so one ldmatrix.x4 feeds two k16 steps
        const int key = kb + nt * 8 + (lane & 7);
        if constexpr (HD % 32 == 0) {
#pragma unroll
            for (int kp = 0; kp < HD / 32; ++kp) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4(b0, b1, b2, b3, smem_u32(t.k + key * Tile<HD>::PITCH + kp * 32 + (lane >> 3) * 8));
                mma16816(s[nt], qa[2 * kp], b0, b1);
                mma16816(s[nt], qa[2 * kp + 1], b2, b3);
            }
        } else {
#pragma unroll
            for (int ks = 0; ks < HD / 16; ++ks) {
                uint32_t b0, b1;
                ldsm_x2(b0, b1, smem_u32(t.k + key * Tile<HD>::PITCH + ks * 16 + ((lane >> 3) & 1) * 8));
                mma16816(s[nt], qa[ks], b0, b1);
            }
        }
    }
    const int c0 = (lane & 3) * 2;
    float mxA = -INFINITY, mxB = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int col = nt * 8 + c0 + (e & 1);
            float val = s[nt][e] * scale_log2e + t.bias[kb + col];
            if (masked(e >> 1, col)) val = -INFINITY;
            s[nt][e] = val;
            if (e < 2) mxA = fmaxf(mxA, val); else mxB = fmaxf(mxB, val);
        }
    }
    mxA = fmaxf(mxA, __shfl_xor_sync(0xffffffffu, mxA, 1));
    mxA = fmaxf(mxA, __shfl_xor_sync(0xffffffffu, mxA, 2));
    mxB = fmaxf(mxB, __shfl_xor_sync(0xffffffffu, mxB, 1));
    mxB = fmaxf(mxB, __shfl_xor_sync(0xffffffffu, mxB, 2));
    const float nA = fmaxf(mA, mxA), nB = fmaxf(mB, mxB);
    const float uA = (nA == -INFINITY) ? 0.f : nA, uB = (nB == -INFINITY) ? 0.f : nB;
    const float cA = fast_exp2(mA - uA), cB = fast_exp2(mB - uB);   // m = -inf -> 0
    mA = nA; mB = nB;
    float sumA = 0.f, sumB = 0.f;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        s[nt][0] = fast_exp2(s[nt][0] - uA); s[nt][1] = fast_exp2(s[nt][1] - uA);
        s[nt][2] = fast_exp2(s[nt][2] - uB); s[nt][3] = fast_exp2(s[nt][3] - uB);
        sumA += s[nt][0] + s[nt][1];
        sumB += s[nt][2] + s[nt][3];
    }
    lA = lA * cA + sumA;
    lB = lB * cB + sumB;
#pragma unroll
    for (int nd = 0; nd < HD / 8; ++nd) { o[nd][0] *= cA; o[nd][1] *= cA; o[nd][2] *= cB; o[nd][3] *= cB; }
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {  // two k16 steps over the 32 keys
        uint32_t pa[4];
        pa[0] = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
        pa[1] = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
        pa[2] = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[3] = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
        for (int nd = 0; nd < HD / 8; nd += 2) {
            uint32_t r0, r1, r2, r3;
            const int key = kb + kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
            const int dim = nd * 8 + (lane >> 4) * 8;
            ldsm_x4_trans(r0, r1, r2, r3, smem_u32(t.v + key * Tile<HD>::PITCH + dim));
            mma16816(o[nd], pa, r0, r1);
            mma16816(o[nd + 1], pa, r2, r3);
        }
    }
}

// GRP (speculative self-attention of the continuous beam-search loop): the draft rows of the call are p.row_len positions
// long, but group g's own draft length gives it rows of desc[g].w positions.  The kernel then works on the group's compact
// rows -- query tiles, key blocks and their columns exactly as a call with D + 1 = desc[g].w would lay them out -- and maps a
// compact row r to the call's row (r / desc[g].w) * p.row_len + r % desc[g].w for its loads and stores.  So a group's
// outputs do not depend on the draft length of the other groups in the call; the positions behind its own are not written.
// (the row mapping needs a few more registers than two CTAs per SM leave: the GRP form runs one CTA per SM without spills)
template <int HD, bool GRP>
__global__ void __launch_bounds__(THREADS, GRP ? 1 : 2)
attn_mma_kernel(Params p) {
    const int g = blockIdx.y, h = blockIdx.x;
    pdl_launch_dependents();
    // With a descriptor table (decoding loop) everything but the queries and the K/V rows appended in this very
    // iteration was written before the iteration's first kernel, which is a fully serialised launch: those reads
    // may run ahead of the programmatic dependency, i.e. the key staging overlaps the tail of the preceding GEMM.
    const bool early = p.desc != nullptr;
    if (!early) pdl_wait();
    // the three scalar fetches every CTA starts with are issued together (behind the early-exit test the compiler could
    // not hoist them: two dependent global round trips)
    int4 dsc = make_int4(0, 0, 0, 0x7fffffff);
    if (p.desc) dsc = p.desc[g];
    const int dynLk = p.lk_dev ? *p.lk_dev : 0;
    const int n_groups_live = p.n_groups_dev ? *p.n_groups_dev : 0x7fffffff;
    if (g >= n_groups_live) return;
    const int RLp = p.spec ? p.row_len : 1;                          // positions per draft row of the call
    const int RL = GRP ? dsc.w : RLp;                                // ... of this group
    const int Lq = GRP ? (p.Lq / p.row_len) * RL : p.Lq;             // query rows of this group (compact)
    auto prow = [&](int r) { return GRP ? (r / RL) * RLp + r % RL : r; };
    if (GRP && (int)blockIdx.z * ROWS_PER_CTA >= Lq) return;
    extern __shared__ __align__(16) uint8_t attn_smem[];
    constexpr int PITCH = Tile<HD>::PITCH;
    Tile<HD> tileA, tileB;
    tileA.k = reinterpret_cast<__nv_bfloat16*>(attn_smem);
    tileA.v = tileA.k + KTA * PITCH;
    tileB.k = tileA.v + KTA * PITCH;
    tileB.v = tileB.k + KTB * PITCH;
    tileA.bias = reinterpret_cast<float*>(tileB.v + KTB * PITCH);
    tileB.bias = tileA.bias + KTA;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kvg = p.desc ? dsc.x : (p.spec ? p.active[g] : (p.kvmap ? p.kvmap[g] : g));
    const int Lk_all = p.spec ? (p.desc ? dsc.y : p.front[kvg]) : (p.lk_dev ? dynLk : p.Lk);
    const int Lk = p.spec ? Lk_all : (p.desc ? min(Lk_all, dsc.w) : (p.lk_group ? min(Lk_all, p.lk_group[kvg]) : Lk_all));
    const long long kv_group_stride = p.lk_dev ? dynLk : p.kv_group_stride;
    const int key_tok_stride = p.lk_dev ? dynLk : p.key_tok_stride;
    const int* key_tok = p.spec ? p.gen + (long long)kvg * p.gen_ld : (p.key_tok ? p.key_tok + (long long)kvg * key_tok_stride : nullptr);
    const bool first_new_masked = p.spec ? ((p.desc ? dsc.z : p.gen[(long long)kvg * p.gen_ld + Lk]) == p.pad_id) : false;
    const __nv_bfloat16* kbase = p.k + (long long)kvg * kv_group_stride * p.kv_ld + h * HD;
    const __nv_bfloat16* vbase = p.v + (long long)kvg * kv_group_stride * p.kv_ld + h * HD;
    const int rA = lane >> 2, c0 = (lane & 3) * 2;

    {   // one block of ROWS_PER_CTA query rows per CTA (blockIdx.z): more, smaller CTAs balance the 148 SMs better
        const int blk0 = blockIdx.z * ROWS_PER_CTA;
        const int wrow0 = blk0 + warp * ROWS_PER_WARP;       // first query row of this warp
        const bool warp_live = wrow0 < Lq;
        const int wrow_last = min(Lq, wrow0 + ROWS_PER_WARP) - 1;

        // ---- staging (asynchronous; the Q fragments are fetched while the copies are in flight) ----
        // phase A window [j0, j0 + KTA): keys shared by the whole group
        const int kA_end = p.causal ? min(Lk, min(Lq, blk0 + ROWS_PER_CTA)) : Lk;
        // keys behind the last unmasked one (source padding) contribute exactly nothing: s_last_key bounds the scan
        __shared__ int s_last_key;
        if (threadIdx.x == 0) s_last_key = 0;
        __syncthreads();
        auto stage_A = [&](int j0, int row0) {
            const int nk = min(KTA, kA_end - j0);
            if (nk <= 0) return;
            const int nfill = (nk + 31) & ~31;
            stage_rows<HD>(tileA, kbase + (long long)j0 * p.kv_ld, vbase + (long long)j0 * p.kv_ld, p.kv_ld, nk, nfill, row0);
            int last = 0;
            for (int j = threadIdx.x; j < nfill; j += THREADS) {
                const bool ok = j < nk && !(key_tok && key_tok[j0 + j] == p.pad_id);
                tileA.bias[j] = ok ? 0.f : -INFINITY;
                if (ok) last = j0 + j + 1;
            }
            if (last) atomicMax(&s_last_key, last);
        };
        // phase B window [u0, u0 + KTB): freshly projected keys of the draft rows this CTA's queries belong to
        const int endB = p.spec ? min(Lq, blk0 + ROWS_PER_CTA) : 0;
        const int firstB = (blk0 / RL) * RL;   // start of the draft row that contains the CTA's first query
        const __nv_bfloat16* nkb = p.spec ? p.newk + (long long)g * p.Lq * p.new_ld + h * HD : nullptr;
        const __nv_bfloat16* nvb = p.spec ? p.newv + (long long)g * p.Lq * p.new_ld + h * HD : nullptr;
        // short draft rows (<= 17 tokens): the keys an m16 query tile can see span at most 32 consecutive rows, so
        // each tile runs ONE 32-key block that starts at its first draft row instead of walking aligned blocks
        const bool fastB = p.spec && RL <= 17 && endB - firstB <= KTB;
        auto stage_B = [&](int u0) {
            const int nk = min(KTB, endB - u0);
            if (nk <= 0) return;
            const int nfill = fastB ? KTB : ((nk + 31) & ~31);
            if constexpr (GRP) {   // compact key row u0 + j lives in the call's row prow(u0 + j)
                constexpr int CH = HD / 8;
                for (int idx = threadIdx.x; idx < nfill * CH; idx += THREADS) {
                    const int j = idx / CH, c = idx % CH;
                    __nv_bfloat16* kd = tileB.k + j * PITCH + c * 8;
                    __nv_bfloat16* vd = tileB.v + j * PITCH + c * 8;
                    if (j < nk) {
                        const long long r = (long long)prow(u0 + j) * p.new_ld + c * 8;
                        cp_async16(kd, nkb + r);
                        cp_async16(vd, nvb + r);
                    } else {
                        *reinterpret_cast<uint4*>(kd) = make_uint4(0, 0, 0, 0);
                        *reinterpret_cast<uint4*>(vd) = make_uint4(0, 0, 0, 0);
                    }
                }
            } else {
                stage_rows<HD>(tileB, nkb + (long long)u0 * p.new_ld, nvb + (long long)u0 * p.new_ld, p.new_ld, nk, nfill);
            }
            for (int j = threadIdx.x; j < nfill; j += THREADS) {
                const bool bad = j >= nk || (first_new_masked && ((u0 + j) % RL) == 0);
                tileB.bias[j] = bad ? -INFINITY : 0.f;
            }
        };
        int n_pre = 0;
        if (early) {
            // cache rows older than this iteration (everything for cross-attention; all but the last draft row's
            // worth of positions for the self-attention prefix) before the dependency wait
            n_pre = min(KTA, kA_end);
            if (p.spec) n_pre = max(0, n_pre - RL);
            if (n_pre > 0) stage_rows<HD>(tileA, kbase, vbase, p.kv_ld, n_pre, n_pre);
            pdl_wait();
        }
        stage_A(0, n_pre);
        if (p.spec) stage_B(firstB);

        uint32_t qa[2][HD / 16][4];
        float o[2][HD / 8][4];
        float m[2][2], l[2][2];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            m[mt][0] = m[mt][1] = -INFINITY;
            l[mt][0] = l[mt][1] = 0.f;
#pragma unroll
            for (int nd = 0; nd < HD / 8; ++nd) o[mt][nd][0] = o[mt][nd][1] = o[mt][nd][2] = o[mt][nd][3] = 0.f;
            const int rowA = wrow0 + mt * 16 + rA, rowB = rowA + 8;
            const __nv_bfloat16* qA = p.q + ((long long)g * p.Lq + prow(rowA)) * p.q_ld + h * HD;
            const __nv_bfloat16* qB = p.q + ((long long)g * p.Lq + prow(rowB)) * p.q_ld + h * HD;
#pragma unroll
            for (int ks = 0; ks < HD / 16; ++ks) {
                const int d = ks * 16 + c0;
                qa[mt][ks][0] = rowA < Lq ? *reinterpret_cast<const uint32_t*>(qA + d) : 0u;
                qa[mt][ks][1] = rowB < Lq ? *reinterpret_cast<const uint32_t*>(qB + d) : 0u;
                qa[mt][ks][2] = rowA < Lq ? *reinterpret_cast<const uint32_t*>(qA + d + 8) : 0u;
                qa[mt][ks][3] = rowB < Lq ? *reinterpret_cast<const uint32_t*>(qB + d + 8) : 0u;
            }
        }
        cp_async_wait_all();
        __syncthreads();

        // ---- phase A ------------------------------------------------------------------------------
        for (int j0 = 0; j0 < kA_end; j0 += KTA) {
            if (j0 > 0) {   // sequences longer than one window (not reached by this model's shapes)
                __syncthreads();
                stage_A(j0, 0);
                cp_async_wait_all();
                __syncthreads();
            }
            const int nk = min(min(KTA, kA_end - j0), s_last_key - j0);
            if (warp_live) {
#pragma unroll 1
                for (int kb = 0; kb < nk; kb += 32) {
                    if (p.causal) {
                        if (j0 + kb > wrow_last) break;
#pragma unroll
                        for (int mt = 0; mt < 2; ++mt) {
                            const int rowA = wrow0 + mt * 16 + rA;
                            const int colbase = j0 + kb;
                            process_block<HD>(tileA, kb, qa[mt], o[mt], m[mt][0], m[mt][1], l[mt][0], l[mt][1], p.scale_log2e, lane,
                                              [&](int rs, int col) { return colbase + col > rowA + rs * 8; });
                        }
                    } else {
#pragma unroll
                        for (int mt = 0; mt < 2; ++mt)
                            process_block<HD>(tileA, kb, qa[mt], o[mt], m[mt][0], m[mt][1], l[mt][0], l[mt][1], p.scale_log2e, lane, NoMask());
                    }
                }
            }
        }

        // ---- phase B ------------------------------------------------------------------------------
        if (fastB) {
            if (warp_live) {
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    const int row0 = wrow0 + mt * 16;
                    if (row0 >= Lq) continue;
                    const int kstart = (row0 / RL) * RL;      // first key row the tile can see
                    const int rowA = row0 + rA;
                    const int startA = (rowA / RL) * RL, startB = ((rowA + 8) / RL) * RL;
                    process_block<HD>(tileB, kstart - firstB, qa[mt], o[mt], m[mt][0], m[mt][1], l[mt][0], l[mt][1], p.scale_log2e, lane,
                                      [&](int rs, int col) {
                                          const int qr = rowA + rs * 8, kr = kstart + col;
                                          return kr < (rs ? startB : startA) || kr > qr;
                                      });
                }
            }
        } else if (p.spec) {
            const int lo = warp_live ? (wrow0 / RL) * RL : 0;
            const int hi = warp_live ? min(Lq, (wrow_last / RL + 1) * RL) : 0;
            for (int u0 = firstB; u0 < endB; u0 += KTB) {
                if (u0 > firstB) {
                    __syncthreads();
                    stage_B(u0);
                    cp_async_wait_all();
                    __syncthreads();
                }
                const int nk = min(KTB, endB - u0);
                if (warp_live) {
#pragma unroll 1
                    for (int kb = 0; kb < nk; kb += 32) {
                        const int u = u0 + kb;
                        if (u + 32 <= lo || u >= hi || u > wrow_last) continue;
#pragma unroll
                        for (int mt = 0; mt < 2; ++mt) {
                            const int rowA = wrow0 + mt * 16 + rA;
                            // a key row is visible iff it lies in the query's own draft row and not after it
                            const int startA = (rowA / RL) * RL, startB = ((rowA + 8) / RL) * RL;
                            process_block<HD>(tileB, kb, qa[mt], o[mt], m[mt][0], m[mt][1], l[mt][0], l[mt][1], p.scale_log2e, lane,
                                              [&](int rs, int col) {
                                                  const int qr = rowA + rs * 8, kr = u + col;
                                                  return kr < (rs ? startB : startA) || kr > qr;
                                              });
                        }
                    }
                }
            }
        }

        // ---- finalize ---------------------------------------------------------------------------
        if (warp_live) {
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                float lA = l[mt][0], lB = l[mt][1];
                lA += __shfl_xor_sync(0xffffffffu, lA, 1);
                lA += __shfl_xor_sync(0xffffffffu, lA, 2);
                lB += __shfl_xor_sync(0xffffffffu, lB, 1);
                lB += __shfl_xor_sync(0xffffffffu, lB, 2);
                const float nanv = __int_as_float(0x7fc00000);
                const float iA = 1.0f / lA, iB = 1.0f / lB;
                const int rowA = wrow0 + mt * 16 + rA, rowB = rowA + 8;
                __nv_bfloat16* oA = p.out + ((long long)g * p.Lq + prow(rowA)) * p.out_ld + h * HD;
                __nv_bfloat16* oB = p.out + ((long long)g * p.Lq + prow(rowB)) * p.out_ld + h * HD;
#pragma unroll
                for (int nd = 0; nd < HD / 8; ++nd) {
                    const int d = nd * 8 + c0;
                    if (rowA < Lq)
                        *reinterpret_cast<uint32_t*>(oA + d) = lA == 0.f ? pack_bf16(nanv, nanv) : pack_bf16(o[mt][nd][0] * iA, o[mt][nd][1] * iA);
                    if (rowB < Lq)
                        *reinterpret_cast<uint32_t*>(oB + d) = lB == 0.f ? pack_bf16(nanv, nanv) : pack_bf16(o[mt][nd][2] * iB, o[mt][nd][3] * iB);
                }
            }
        }
    }
}

template <bool GRP>
static void launch(const Params& p, int heads, int head_dim, int n_groups_max, cudaStream_t s) {
    dim3 grid(heads, n_groups_max, (p.Lq + ROWS_PER_CTA - 1) / ROWS_PER_CTA);
    if (head_dim == 16) { if (!ensure_dyn_smem(attn_mma_kernel<16, GRP>, (int)smem_bytes<16>())) launch_pdl(attn_mma_kernel<16, GRP>, grid, dim3(THREADS), smem_bytes<16>(), s, p); }
    else if (head_dim == 32) { if (!ensure_dyn_smem(attn_mma_kernel<32, GRP>, (int)smem_bytes<32>())) launch_pdl(attn_mma_kernel<32, GRP>, grid, dim3(THREADS), smem_bytes<32>(), s, p); }
    else if (head_dim == 64) { if (!ensure_dyn_smem(attn_mma_kernel<64, GRP>, (int)smem_bytes<64>())) launch_pdl(attn_mma_kernel<64, GRP>, grid, dim3(THREADS), smem_bytes<64>(), s, p); }
}
}  // namespace amma

void launch_attention_mma(const __nv_bfloat16* q, int q_ld, const __nv_bfloat16* k, const __nv_bfloat16* v, int kv_ld,
                          __nv_bfloat16* out, int out_ld, int n_groups_max, const int* n_groups_dev,
                          int Lq, int Lk, long long kv_group_stride, const int* kvmap,
                          const int* key_tok, int key_tok_stride, int pad_id, bool causal,
                          int heads, int head_dim, cudaStream_t s, const int* lk_dev, const int* lk_group, const int4* desc) {
    if (n_groups_max <= 0 || Lq <= 0) return;
    amma::Params p{};
    p.lk_dev = lk_dev;
    p.lk_group = lk_group;
    p.desc = desc;
    p.q = q; p.q_ld = q_ld; p.k = k; p.v = v; p.kv_ld = kv_ld; p.out = out; p.out_ld = out_ld;
    p.n_groups_dev = n_groups_dev; p.Lq = Lq; p.Lk = Lk; p.kv_group_stride = kv_group_stride; p.kvmap = kvmap;
    p.key_tok = key_tok; p.key_tok_stride = key_tok_stride; p.pad_id = pad_id; p.causal = causal ? 1 : 0;
    p.scale_log2e = 1.4426950408889634f / sqrtf((float)head_dim);
    p.spec = 0;
    amma::launch<false>(p, heads, head_dim, n_groups_max, s);
}

void launch_spec_self_attention_mma(const __nv_bfloat16* qkv, int qkv_ld, const __nv_bfloat16* kcache, const __nv_bfloat16* vcache,
                                    long long cache_query_stride, int cache_ld, __nv_bfloat16* out, int out_ld,
                                    int B_max, const int* n_active_dev, const int* active, const int* front,
                                    const int* gen, int gen_ld, int pad_id, int N, int D,
                                    int heads, int head_dim, cudaStream_t s, const int4* desc, bool group_row_len) {
    if (B_max <= 0) return;
    const int E = heads * head_dim;
    amma::Params p{};
    p.desc = desc;
    p.q = qkv; p.q_ld = qkv_ld; p.k = kcache; p.v = vcache; p.kv_ld = cache_ld; p.out = out; p.out_ld = out_ld;
    p.n_groups_dev = n_active_dev; p.Lq = N * (D + 1); p.Lk = 0;
    p.kv_group_stride = cache_query_stride / cache_ld;   // rows per query in the cache
    p.kvmap = nullptr; p.key_tok = nullptr; p.key_tok_stride = 0; p.pad_id = pad_id; p.causal = 0;
    p.scale_log2e = 1.4426950408889634f / sqrtf((float)head_dim);
    p.spec = 1; p.active = active; p.front = front; p.gen = gen; p.gen_ld = gen_ld;
    p.newk = qkv + E; p.newv = qkv + 2 * E; p.new_ld = qkv_ld; p.row_len = D + 1;
    if (group_row_len && desc) amma::launch<true>(p, heads, head_dim, B_max, s);
    else amma::launch<false>(p, heads, head_dim, B_max, s);
}

}  // namespace ttb
