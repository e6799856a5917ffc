// bf16 GEMM on the 5th-generation tensor cores: C[M,N] = A[M,K] * W[N,K]^T + bias (+ReLU).
//
//   * operands: both K-major bf16 (activations [M,K], nn.Linear weights [N,K]) -> no transposes;
//   * TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) stages 128 x 64 A tiles and BN x 64 W tiles
//     into a 3-deep shared-memory ring guarded by full/empty mbarriers;
//   * one elected thread issues tcgen05.mma (cta_group::1, kind::f16, M=128, N=BN, K=16) with the
//     fp32 accumulator tile in TMEM; tcgen05.commit releases ring slots and signals the epilogue;
//   * four epilogue warps read the accumulator with tcgen05.ld (32 lanes x 32 columns per warp
//     instruction), add bias, apply ReLU, convert and store full 32-byte sectors per thread.
// One output tile per CTA, two CTAs per SM (96 KB smem, 128 TMEM columns each) so that the epilogue
// of one tile overlaps the main loop of another.  The live row count is read on the device
// (RowCount): CTAs beyond it exit before touching any barrier.
#include "kernels.cuh"
#include "philox.cuh"

#include <cuda.h>
#include <cstdlib>
#include <atomic>
#include <map>
#include <mutex>
#include <tuple>
#include <type_traits>

namespace ttb {

namespace tc {
constexpr int BM = 128, BN = 128, BK = 64, STAGES = 3, UMMA_K = 16;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int THREADS = 192;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 128 /*barriers*/;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor of a K-major tile stored with the 128-byte swizzle: rows of 128
// bytes, 8-row atoms 1024 bytes apart (SBO), descriptor version 1 (Blackwell), layout type 2.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;                 // leading byte offset (unused for swizzled K-major), 16 B
    d |= (uint64_t)(1024 >> 4) << 32;       // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                 // descriptor version
    d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
    return d;
}
// Instruction descriptor: D=f32, A=B=bf16, both K-major, N>>3 at bit 17, M>>4 at bit 24.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32"
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
        " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 32 fp32 accumulator values of one row -> staging row in shared memory (already bias/ReLU'd)
template <typename OutT>
__device__ __forceinline__ void stage_chunk(uint8_t* dst, const float (&v)[32]);
template <>
__device__ __forceinline__ void stage_chunk<float>(uint8_t* dst, const float (&v)[32]) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
        reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
template <>
__device__ __forceinline__ void stage_chunk<__nv_bfloat16>(uint8_t* dst, const float (&v)[32]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint4 u;
        __nv_bfloat162 p0 = __floats2bfloat162_rn(v[8 * j + 0], v[8 * j + 1]);
        __nv_bfloat162 p1 = __floats2bfloat162_rn(v[8 * j + 2], v[8 * j + 3]);
        __nv_bfloat162 p2 = __floats2bfloat162_rn(v[8 * j + 4], v[8 * j + 5]);
        __nv_bfloat162 p3 = __floats2bfloat162_rn(v[8 * j + 6], v[8 * j + 7]);
        u.x = *reinterpret_cast<uint32_t*>(&p0);
        u.y = *reinterpret_cast<uint32_t*>(&p1);
        u.z = *reinterpret_cast<uint32_t*>(&p2);
        u.w = *reinterpret_cast<uint32_t*>(&p3);
        reinterpret_cast<uint4*>(dst)[j] = u;
    }
}

template <typename OutT>
__global__ void __launch_bounds__(THREADS, 2)
gemm_bf16_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const float* __restrict__ bias, OutT* __restrict__ C, int ldc, RowCount rows, int N, int K, int relu) {
    const int M = rows.live();
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    if (m0 >= M) return;  // uniform per CTA, before any barrier / TMEM allocation

    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;  // 128B-swizzle atoms need 1024-byte alignment
    uint8_t* gen_base = smem_raw + (base - raw);
    const uint32_t bar_base = base + STAGES * STAGE_BYTES;
    // barriers: full[0..S), empty[S..2S), tmem_full[2S]; tmem base pointer slot after them
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
    const uint32_t tmem_full_bar = bar_base + 8u * (2 * STAGES);
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen_base + STAGES * STAGE_BYTES + 8 * (2 * STAGES + 1));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int KB = K / BK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
            mbar_init(tmem_full_bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"((uint32_t)BN) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer =====
            for (int kb = 0; kb < KB; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(empty_bar(s), ph ^ 1);
                mbar_expect_tx(full_bar(s), STAGE_BYTES);
                const uint32_t a_dst = base + s * STAGE_BYTES, b_dst = a_dst + A_BYTES;
                tma_load_2d(a_dst, &tmA, kb * BK, m0, full_bar(s));
                tma_load_2d(b_dst, &tmB, kb * BK, n0, full_bar(s));
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {  // ===== MMA issuer =====
            constexpr uint32_t idesc = umma_idesc_bf16(BM, BN);
            for (int kb = 0; kb < KB; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(full_bar(s), ph);
                tcgen05_fence_after();
                const uint32_t a_src = base + s * STAGE_BYTES, b_src = a_src + A_BYTES;
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t adesc = umma_desc_sw128(a_src + k * UMMA_K * 2);
                    const uint64_t bdesc = umma_desc_sw128(b_src + k * UMMA_K * 2);
                    umma_bf16(tmem_base, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                }
                umma_commit(empty_bar(s));  // slot reusable once these MMAs have read it
            }
            umma_commit(tmem_full_bar);     // accumulator complete
        }
    } else {  // ===== epilogue: warps 2..5 own TMEM lane quarters (warp % 4) =====
        // TMEM -> registers (one row per thread) -> bias/ReLU/convert -> per-warp staging tile in the
        // (now idle) pipeline shared memory -> fully coalesced 16-byte global stores, whole rows per
        // warp instruction.  All TMA loads and MMAs have completed once tmem_full fires, so the ring
        // buffers are free to reuse.
        const int q = warp & 3;
        constexpr int ESZ = (int)sizeof(OutT);
        constexpr int PITCH = BN * ESZ + 16;          // +16 B: conflict-free 16-byte row-strided writes
        uint8_t* stage = gen_base + q * 32 * PITCH;
        mbar_wait(tmem_full_bar, 0);
        tcgen05_fence_after();
        const int n_cols = min(BN, N - n0);
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
            if (c0 >= n_cols) break;
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                float t = __uint_as_float(r[j]);
                if (bias && c0 + j < n_cols) t += __ldg(bias + n0 + c0 + j);
                if (relu) t = fmaxf(t, 0.f);
                v[j] = t;
            }
            stage_chunk<OutT>(stage + lane * PITCH + c0 * ESZ, v);
        }
        __syncwarp();
        const int row_base = m0 + q * 32;
        constexpr int EPC = 16 / ESZ;                 // elements per 16-byte chunk
        constexpr int CH = BN / EPC;                  // chunks per row: 16 (bf16) or 32 (fp32)
        constexpr int RPI = 32 / CH;                  // rows per warp instruction: 2 or 1
        const bool vec_ok = ((long long)ldc * ESZ) % 16 == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0;
        if (vec_ok) {
#pragma unroll 4
            for (int rr = 0; rr < 32; rr += RPI) {
                const int rl = rr + lane / CH, ch = lane % CH;
                const int row = row_base + rl, col = ch * EPC;
                if (row < M && col < n_cols) {
                    const uint8_t* sp = stage + rl * PITCH + ch * 16;
                    OutT* gp = C + (long long)row * ldc + n0 + col;
                    if (col + EPC <= n_cols) {
                        *reinterpret_cast<uint4*>(gp) = *reinterpret_cast<const uint4*>(sp);
                    } else {
                        for (int j = 0; j < n_cols - col; ++j) gp[j] = reinterpret_cast<const OutT*>(sp)[j];
                    }
                }
            }
        } else {
            for (int rl = 0; rl < 32; ++rl) {
                const int row = row_base + rl;
                if (row >= M) break;
                const OutT* sp = reinterpret_cast<const OutT*>(stage + rl * PITCH);
                for (int c = lane; c < n_cols; c += 32) C[(long long)row * ldc + n0 + c] = sp[c];
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)BN) : "memory");
    }
}

// =====================================================================================================
// Persistent, warp-specialised variant (default).  One CTA per SM loops over output tiles:
//   warp 0      TMA producer     (4-stage smem ring, runs ahead across tile boundaries)
//   warp 1      MMA issuer       (tcgen05.mma into one of two TMEM accumulator buffers)
//   warps 2..9  epilogue         (TMEM lane quarter = warp % 4, column half = (warp - 2) / 4)
// so the loads and MMAs of tile i+1 overlap the epilogue of tile i (smem full/empty and TMEM
// full/empty mbarrier pipelines).  Epilogue: tcgen05.ld -> bias/ReLU/convert -> per-warp staging tile
// -> coalesced 16-byte stores of whole row segments.
namespace pers {
constexpr int PSTAGES = 4;
constexpr int EPI_WARPS = 8;
constexpr int THREADS = 64 + EPI_WARPS * 32;
template <typename OutT, int BN_> constexpr int pitch() { return (BN_ / 2) * (int)sizeof(OutT) + 16; }
template <int BN_> constexpr int stage_bytes() { return A_BYTES + BN_ * BK * 2; }
template <typename OutT, int BN_> constexpr int smem_bytes() {
    return PSTAGES * stage_bytes<BN_>() + EPI_WARPS * 32 * pitch<OutT, BN_>() + EPI_WARPS * (BN_ / 2) * 4 + 1024 + 256;
}
}  // namespace pers

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

template <typename OutT, int BN_>
__global__ void __launch_bounds__(pers::THREADS, 1)
gemm_bf16_tc_persistent_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                               const float* __restrict__ bias, OutT* __restrict__ C, int ldc, RowCount rows, int N, int K, int relu) {
    using namespace pers;
    constexpr int NST = pers::PSTAGES;
    constexpr int BN = BN_;                                  // shadows tc::BN inside this kernel
    constexpr int COLS_PER_WARP = BN_ / 2;
    constexpr int STAGE_BYTES = pers::stage_bytes<BN_>();   // shadows tc::STAGE_BYTES
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gen_base = smem_raw + (base - raw);
    constexpr int ESZ = (int)sizeof(OutT);
    constexpr int PITCH = pitch<OutT, BN_>();
    constexpr int STAGING_BYTES = EPI_WARPS * 32 * PITCH;
    constexpr int BIAS_BYTES = EPI_WARPS * COLS_PER_WARP * 4;
    uint8_t* staging = gen_base + NST * STAGE_BYTES;
    float* bias_sm = reinterpret_cast<float*>(staging + STAGING_BYTES);
    const uint32_t bar_base = base + NST * STAGE_BYTES + STAGING_BYTES + BIAS_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (NST + s); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * NST + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * NST + 2 + a); };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(staging + STAGING_BYTES + BIAS_BYTES + 8 * (2 * NST + 4));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int KB = K / BK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < NST; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
            for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), EPI_WARPS); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"((uint32_t)(2 * BN)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // everything above is independent of earlier kernels; from here on their results are needed
    pdl_launch_dependents();
    const int M = rows.live();   // written before this programmatic chain started (see gemm_pair_k256_kernel): fetched ahead of the wait
    pdl_wait();
    const int n_tiles_n = (N + BN - 1) / BN;
    const int total_tiles = ((M + BM - 1) / BM) * n_tiles_n;   // CTAs beyond it skip straight to the teardown

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer =====
            int it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int m0 = (tile / n_tiles_n) * BM, n0 = (tile % n_tiles_n) * BN;
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    const int s = it % NST;
                    const uint32_t ph = (it / NST) & 1;
                    mbar_wait(empty_bar(s), ph ^ 1);
                    mbar_expect_tx(full_bar(s), STAGE_BYTES);
                    const uint32_t a_dst = base + s * STAGE_BYTES, b_dst = a_dst + A_BYTES;
                    tma_load_2d(a_dst, &tmA, kb * BK, m0, full_bar(s));
                    tma_load_2d(b_dst, &tmB, kb * BK, n0, full_bar(s));
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {  // ===== MMA issuer =====
            constexpr uint32_t idesc = umma_idesc_bf16(BM, BN);
            int it = 0, lt = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
                const int acc = lt & 1;
                const uint32_t acc_ph = (lt >> 1) & 1;
                mbar_wait(tempty_bar(acc), acc_ph ^ 1);      // epilogue has drained this accumulator buffer
                tcgen05_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < KB; ++kb, ++it) {
                    const int s = it % NST;
                    const uint32_t ph = (it / NST) & 1;
                    mbar_wait(full_bar(s), ph);
                    tcgen05_fence_after();
                    const uint32_t a_src = base + s * STAGE_BYTES, b_src = a_src + A_BYTES;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t adesc = umma_desc_sw128(a_src + k * UMMA_K * 2);
                        const uint64_t bdesc = umma_desc_sw128(b_src + k * UMMA_K * 2);
                        umma_bf16(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    umma_commit(empty_bar(s));
                }
                umma_commit(tfull_bar(acc));
            }
        }
    } else {  // ===== epilogue warps =====
        const int ew = warp - 2;
        const int q = warp & 3;                 // TMEM lane quarter this warp may access
        const int half = ew >> 2;               // which 64 columns of the tile
        uint8_t* stage = staging + ew * 32 * PITCH;
        float* my_bias = bias_sm + ew * COLS_PER_WARP;
        constexpr int EPC = 16 / ESZ;                 // elements per 16-byte chunk
        constexpr int CH = COLS_PER_WARP / EPC;       // chunks per row segment: 8 (bf16) or 16 (fp32)
        constexpr int RPI = 32 / CH;                  // rows per warp store instruction: 4 or 2
        const bool vec_ok = ((long long)ldc * ESZ) % 16 == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0;
        int lt = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
            const int m0 = (tile / n_tiles_n) * BM, n0 = (tile % n_tiles_n) * BN + half * COLS_PER_WARP;
            const int acc = lt & 1;
            const uint32_t acc_ph = (lt >> 1) & 1;
            const int n_cols = max(0, min(COLS_PER_WARP, N - n0));
            // bias slice of this warp's columns (overlaps the wait for the accumulator)
            for (int c = lane; c < COLS_PER_WARP; c += 32) my_bias[c] = (bias && c < n_cols) ? __ldg(bias + n0 + c) : 0.f;
            __syncwarp();
            mbar_wait(tfull_bar(acc), acc_ph);
            tcgen05_fence_after();
#pragma unroll
            for (int c0 = 0; c0 < COLS_PER_WARP; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + half * COLS_PER_WARP + c0), r);
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float t = __uint_as_float(r[j]) + my_bias[c0 + j];
                    if (relu) t = fmaxf(t, 0.f);
                    v[j] = t;
                }
                stage_chunk<OutT>(stage + lane * PITCH + c0 * ESZ, v);
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));   // accumulator buffer may be overwritten
            const int row_base = m0 + q * 32;
            if (vec_ok) {
#pragma unroll 4
                for (int rr = 0; rr < 32; rr += RPI) {
                    const int rl = rr + lane / CH, ch = lane % CH;
                    const int row = row_base + rl, col = ch * EPC;
                    if (row < M && col < n_cols) {
                        const uint8_t* sp = stage + rl * PITCH + ch * 16;
                        OutT* gp = C + (long long)row * ldc + n0 + col;
                        if (col + EPC <= n_cols) {
                            *reinterpret_cast<uint4*>(gp) = *reinterpret_cast<const uint4*>(sp);
                        } else {
                            for (int j = 0; j < n_cols - col; ++j) gp[j] = reinterpret_cast<const OutT*>(sp)[j];
                        }
                    }
                }
            } else {
                for (int rl = 0; rl < 32; ++rl) {
                    const int row = row_base + rl;
                    if (row >= M) break;
                    const OutT* sp = reinterpret_cast<const OutT*>(stage + rl * PITCH);
                    for (int c = lane; c < n_cols; c += 32) C[(long long)row * ldc + n0 + c] = sp[c];
                }
            }
            __syncwarp();   // staging tile is rewritten by the next iteration
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BN)) : "memory");
    }
}

// ---- host: tensor-map cache -----------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

// 2-D tensor [rows, cols] with row stride ld (elements); box = box_rows x 128 bytes (64 bf16 or 32 fp32
// elements), 128-byte swizzle
static int get_tensor_map(const void* ptr, int rows, int cols, int ld, int box_rows, CUtensorMap* out, bool f32 = false) {
    using Key = std::tuple<const void*, int, int, int, int, bool>;
    static std::map<Key, CUtensorMap> cache;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    Key key{ptr, rows, cols, ld, box_rows, f32};
    auto it = cache.find(key);
    if (it != cache.end()) {
        *out = it->second;
        return 0;
    }
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        set_last_error("cuTensorMapEncodeTiled is not available from the driver");
        return 4;
    }
    CUtensorMap m;
    const int esz = f32 ? 4 : 2;
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * esz};
    cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride,
                     box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r) + " (rows=" + std::to_string(rows) +
                       " cols=" + std::to_string(cols) + " ld=" + std::to_string(ld) + ")");
        return 4;
    }
    if (cache.size() > 4096) cache.clear();
    cache[key] = m;
    *out = m;
    return 0;
}

// =====================================================================================================
// GEMM + bias + residual + LayerNorm (+ optional second LayerNorm) for E = 256 rows:
//     x <- LN2?( LN1( x + A W^T + bias ) ),  written as fp32 (x, in place) and bf16 (xh)
// One cluster of two CTAs per 128-row tile; CTA r owns output columns [128 r, 128 r + 128):
//   warp 0      TMA producer: K-blocks of A (128 x 64) and of the CTA's W slice (128 x 64) into a 4-stage ring,
//               plus the fp32 residual tile (four 128 x 32 boxes, 128-byte swizzle)
//   warp 1      tcgen05.mma issuer, 128 x 128 fp32 accumulator in TMEM
//   warps 2..9  epilogue: one thread per (row, 64-column half).  tcgen05.ld -> + bias + residual (swizzled
//               shared-memory reads are conflict-free for a row-per-lane pattern) -> local mean / M2 ->
//               the four partial statistics of a row (2 CTAs x 2 halves) are exchanged through
//               distributed shared memory + one cluster barrier and combined with Chan's formula ->
//               normalise -> write fp32 / bf16 tiles back into swizzled shared memory -> TMA stores.
// The LayerNorm kernels, the fp32 GEMM output round trip through HBM/L2 and one launch per
// sub-layer disappear.
namespace lnk {
constexpr int NST = 4;
constexpr int BNL = 128;                               // output columns per CTA
constexpr int STAGE = A_BYTES + BNL * BK * 2;          // 32 KB
constexpr int RESID_BYTES = BM * BNL * 4;              // 64 KB
constexpr int PART_BYTES = 4 * BM * 8;                 // float2[4][128]
constexpr int PARAM_FLOATS = 6 * BNL;                  // bias, g1, b1, g2, b2 slices, bias of the chained GEMM
constexpr int THREADS = 320;
constexpr int SMEM = NST * STAGE + RESID_BYTES + 2 * PART_BYTES + PARAM_FLOATS * 4 + 256 + 1024;
}  // namespace lnk

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_peer_f32x2(uint32_t local_addr, uint32_t peer_rank, float a, float b) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_addr), "r"(peer_rank));
    asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(remote), "f"(a), "f"(b) : "memory");
}

// (a, b) into the same shared-memory offset of CTA `peer_rank`, its 8 bytes counted on that CTA's mbarrier `bar` (same
// offset there): the receiver waits on its own barrier and needs no cluster-scope release / acquire pair, which costs
// 1.1-1.9 k cycles per CTA on this chip (in-kernel stamps, profiles/r2_ffn_pair_timeline.txt)
__device__ __forceinline__ void st_async_peer_f32x2(uint32_t local_addr, uint32_t bar, uint32_t peer_rank, float a, float b) {
    uint32_t raddr, rbar;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(local_addr), "r"(peer_rank));
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rbar) : "r"(bar), "r"(peer_rank));
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(raddr), "f"(a), "f"(b), "r"(rbar)
                 : "memory");
}
__device__ __forceinline__ void cluster_sync_relaxed() {   // execution barrier only: orders no memory
    asm volatile("barrier.cluster.arrive.relaxed.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
}

// ---- LayerNorm tail shared by the fused kernels: one thread = (row, 64-column half h of the CTA's 128 columns) ----
// Packed fp32 arithmetic (FFMA2 / FADD2: two lanes per issue slot).  The LayerNorm phases of the fused kernels are bound by
// the issue rate of their eight epilogue warps (in-kernel stamps: doubling the warps changes nothing), so halving the
// instruction count is what shortens them.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra, rb, rc, rd;
    float2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
    return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    unsigned long long ra, rb, rd;
    float2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
    return d;
}
// acc + bias + residual for four columns, in that order (two packed adds per pair)
__device__ __forceinline__ void add3_f32x4(float* v, const uint32_t* r, const float4& bv, const float4& rv) {
    const float2 lo = fadd2(fadd2(make_float2(__uint_as_float(r[0]), __uint_as_float(r[1])), make_float2(bv.x, bv.y)), make_float2(rv.x, rv.y));
    const float2 hi = fadd2(fadd2(make_float2(__uint_as_float(r[2]), __uint_as_float(r[3])), make_float2(bv.z, bv.w)), make_float2(rv.z, rv.w));
    v[0] = lo.x; v[1] = lo.y; v[2] = hi.x; v[3] = hi.y;
}
// mean and sum of squared deviations of 64 values: four partial sums (two packed accumulators), chains of 16
__device__ __forceinline__ void ln_local_stats(const float (&v)[64], float& mean, float& m2) {
    float2 s0 = make_float2(0.f, 0.f), s1 = s0;
#pragma unroll
    for (int j = 0; j < 64; j += 4) {
        s0 = fadd2(s0, make_float2(v[j], v[j + 1]));
        s1 = fadd2(s1, make_float2(v[j + 2], v[j + 3]));
    }
    mean = ((s0.x + s0.y) + (s1.x + s1.y)) * (1.0f / 64.0f);
    const float2 nm = make_float2(-mean, -mean);
    float2 q0 = make_float2(0.f, 0.f), q1 = q0;
#pragma unroll
    for (int j = 0; j < 64; j += 4) {
        const float2 d0 = fadd2(make_float2(v[j], v[j + 1]), nm), d1 = fadd2(make_float2(v[j + 2], v[j + 3]), nm);
        q0 = ffma2(d0, d0, q0);
        q1 = ffma2(d1, d1, q1);
    }
    m2 = (q0.x + q0.y) + (q1.x + q1.y);
}
// partial statistics of group pidx = 2 * rank + h into both CTAs' tables (float2[4][128])
__device__ __forceinline__ void ln_publish(float2* part, int pidx, int row, uint32_t rank, float mean, float m2) {
    part[pidx * BM + row] = make_float2(mean, m2);
    st_peer_f32x2(smem_u32(&part[pidx * BM + row]), rank ^ 1u, mean, m2);
}
// Chan's combination of the four equally sized groups (64 values each) of a 256-wide row, then scale/shift:
// ((v - mean) rstd) g + b as two packed FMAs per pair: t = v rstd - mean rstd, t g + b
__device__ __forceinline__ void ln_normalise(float (&v)[64], const float2* part, int row, const float* gg, const float* bb) {
    const float2 p0 = part[row], p1 = part[BM + row], p2 = part[2 * BM + row], p3 = part[3 * BM + row];
    const float mean = 0.25f * (p0.x + p1.x + p2.x + p3.x);
    const float d0 = p0.x - mean, d1 = p1.x - mean, d2 = p2.x - mean, d3 = p3.x - mean;
    const float m2 = p0.y + p1.y + p2.y + p3.y + 64.0f * (d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3);
    const float rstd = rsqrtf(m2 * (1.0f / 256.0f) + 1e-5f);
    const float2 rs = make_float2(rstd, rstd), nmr = make_float2(-mean * rstd, -mean * rstd);
    const float4* g4 = reinterpret_cast<const float4*>(gg);   // 16-byte aligned parameter slices: 32 broadcast
    const float4* b4 = reinterpret_cast<const float4*>(bb);   // LDS.128 per thread instead of 128 LDS.32
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float4 g = g4[j], b = b4[j];
        const float2 lo = ffma2(ffma2(make_float2(v[4 * j], v[4 * j + 1]), rs, nmr), make_float2(g.x, g.y), make_float2(b.x, b.y));
        const float2 hi = ffma2(ffma2(make_float2(v[4 * j + 2], v[4 * j + 3]), rs, nmr), make_float2(g.z, g.w), make_float2(b.z, b.w));
        v[4 * j + 0] = lo.x;
        v[4 * j + 1] = lo.y;
        v[4 * j + 2] = hi.x;
        v[4 * j + 3] = hi.y;
    }
}
// fp32 values into two [128 x 32] boxes and bf16 values into one [128 x 64] box (128-byte swizzle, TMA-store layout)
__device__ __forceinline__ void ln_store_tiles(const float (&v)[64], uint8_t* f32_box0, uint8_t* bf16_box, int row) {
    const int swz = row & 7;
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 32) {
        uint8_t* box = f32_box0 + (c0 / 32) * (BM * 128) + row * 128;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int j = c0 + 4 * c;
            *reinterpret_cast<float4*>(box + ((c ^ swz) << 4)) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
    }
    uint8_t* hbox = bf16_box + row * 128;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        uint4 u;
        __nv_bfloat162 p0 = __floats2bfloat162_rn(v[8 * c + 0], v[8 * c + 1]);
        __nv_bfloat162 p1 = __floats2bfloat162_rn(v[8 * c + 2], v[8 * c + 3]);
        __nv_bfloat162 p2 = __floats2bfloat162_rn(v[8 * c + 4], v[8 * c + 5]);
        __nv_bfloat162 p3 = __floats2bfloat162_rn(v[8 * c + 6], v[8 * c + 7]);
        u.x = *reinterpret_cast<uint32_t*>(&p0);
        u.y = *reinterpret_cast<uint32_t*>(&p1);
        u.z = *reinterpret_cast<uint32_t*>(&p2);
        u.w = *reinterpret_cast<uint32_t*>(&p3);
        *reinterpret_cast<uint4*>(hbox + ((c ^ swz) << 4)) = u;
    }
}

#ifdef TTB_LNK_TIMELINE
// Debug build only: clock64 stamps of thread 64 of CTA 0
__device__ long long g_lnk_ts[16];
#define LNK_TS(i) do { if (blockIdx.x == 0 && threadIdx.x == 64) g_lnk_ts[i] = clock64(); } while (0)
#else
#define LNK_TS(i) do { } while (0)
#endif

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(lnk::THREADS, 1)
gemm_resid_ln_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmXh,
                     const float* __restrict__ bias, const float* __restrict__ g1, const float* __restrict__ b1,
                     const float* __restrict__ g2, const float* __restrict__ b2, RowCount rows, int K,
                     const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmQ,
                     const float* __restrict__ bias2, int chain) {
    using namespace lnk;
    const int m0 = (blockIdx.x >> 1) * BM;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int n0 = (int)rank * BNL;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gen_base = smem_raw + (base - raw);
    uint8_t* resid_sm = gen_base + NST * STAGE;
    const uint32_t resid_u32 = base + NST * STAGE;
    float2* part1 = reinterpret_cast<float2*>(resid_sm + RESID_BYTES);
    float2* part2 = part1 + 4 * BM;
    float* prm = reinterpret_cast<float*>(part2 + 4 * BM);
    const uint32_t bar_base = base + NST * STAGE + RESID_BYTES + 2 * PART_BYTES + PARAM_FLOATS * 4;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (NST + s); };
    const uint32_t tfull_bar = bar_base + 8u * (2 * NST);
    const uint32_t resid_bar = bar_base + 8u * (2 * NST + 1);
    const uint32_t w2_bar = bar_base + 8u * (2 * NST + 2);        // chained GEMM: its weight slice has landed
    const uint32_t a2_peer_bar = bar_base + 8u * (2 * NST + 3);   //   the peer's half of the LayerNorm output has landed
    const uint32_t a2_own_bar = bar_base + 8u * (2 * NST + 4);    //   this CTA's half is written
    const uint32_t acc2_bar = bar_base + 8u * (2 * NST + 5);      //   its accumulator is complete
    // LayerNorm statistics of the peer (same rows, other 128 columns): 256 x 8 bytes by st.async per exchange (see ffn_pair_kernel)
    auto stat_bar = [&](int i) { return bar_base + 8u * (2 * NST + 6 + i); };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen_base + (bar_base - base) + 8 * (2 * NST + 8));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int KB = K / BK;
    LNK_TS(0);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmX)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmXh)) : "memory");
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < NST; ++s) { mbar_init(full_bar(s), 2); mbar_init(empty_bar(s), 1); }   // full: A and W arrive separately
            mbar_init(tfull_bar, 1);
            mbar_init(resid_bar, 1);
            mbar_init(w2_bar, 1);
            mbar_init(a2_peer_bar, 1);
            mbar_init(a2_own_bar, 1);
            mbar_init(acc2_bar, 1);
            mbar_init(stat_bar(0), 1);
            mbar_init(stat_bar(1), 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            // The weights do not depend on earlier kernels: the W K-blocks of the first ring fill are requested right here,
            // at the very top of the CTA (before the tensor-memory allocation, the parameter loads and the dependency
            // wait), so they are in flight during the whole prologue of every CTA, also of those that only get their SM
            // when a CTA of the preceding kernel exits.
            for (int kb = 0; kb < (KB < NST ? KB : NST); ++kb) {
                mbar_expect_tx(full_bar(kb), BNL * BK * 2);
                tma_load_2d(base + kb * STAGE + A_BYTES, &tmB, kb * BK, n0, full_bar(kb));
            }
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"((uint32_t)(2 * BNL)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (warp >= 2) {   // parameter slices of this CTA's columns
        const int t = threadIdx.x - 64;
        if (t < BNL) {
            prm[t] = bias ? __ldg(bias + n0 + t) : 0.f;
            prm[BNL + t] = __ldg(g1 + n0 + t);
            prm[2 * BNL + t] = __ldg(b1 + n0 + t);
            prm[3 * BNL + t] = g2 ? __ldg(g2 + n0 + t) : 1.f;
            prm[4 * BNL + t] = g2 ? __ldg(b2 + n0 + t) : 0.f;
            prm[5 * BNL + t] = (chain && bias2) ? __ldg(bias2 + n0 + t) : 0.f;
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // phase 0 of the cluster barrier: "this CTA is running" (its shared memory may be written by the peer);
    // the matching wait sits right before the first remote store
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    // everything above is independent of earlier kernels (weights only); from here on their results are needed
    pdl_launch_dependents();
    const int live_rows = rows.live();   // written before this programmatic chain started (see gemm_pair_k256_kernel): fetched ahead of the wait
    LNK_TS(1);
    pdl_wait();
    LNK_TS(2);
    const bool live = m0 < live_rows;    // uniform per cluster: dead tiles only take part in the barriers

    const int n_pre = KB < NST ? KB : NST;   // W K-blocks requested in the prologue
    if (warp == 0) {
        if (lane == 0 && !live) {   // requested weights must land before the CTA may exit
            for (int kb = 0; kb < n_pre; ++kb) { mbar_arrive(full_bar(kb)); mbar_wait(full_bar(kb), 0); }
        }
        if (lane == 0 && live) {  // ===== TMA producer =====
            for (int kb = 0; kb < KB; ++kb) {
                const int s = kb % NST;
                const uint32_t ph = (kb / NST) & 1;
                mbar_wait(empty_bar(s), ph ^ 1);
                const uint32_t a_dst = base + s * STAGE, b_dst = a_dst + A_BYTES;
                mbar_expect_tx(full_bar(s), A_BYTES);
                tma_load_2d(a_dst, &tmA, kb * BK, m0, full_bar(s));
                if (kb >= n_pre) {
                    mbar_expect_tx(full_bar(s), BNL * BK * 2);
                    tma_load_2d(b_dst, &tmB, kb * BK, n0, full_bar(s));
                }
                if (kb == (KB < NST ? KB : NST) - 1) {   // residual tile: queued behind the first ring fill
                    mbar_expect_tx(resid_bar, RESID_BYTES);
                    for (int bx = 0; bx < 4; ++bx) tma_load_2d(resid_u32 + bx * (BM * 128), &tmX, n0 + 32 * bx, m0, resid_bar);
                }
            }
            if (chain) {   // weight slice of the chained GEMM into ring stages 2-3 once GEMM1 has released the ring
                mbar_wait(tfull_bar, 0);
                mbar_expect_tx(w2_bar, 4 * 16384);
                for (int kb = 0; kb < 4; ++kb) tma_load_2d(base + 2 * STAGE + kb * 16384, &tmW2, kb * BK, n0, w2_bar);
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && live) {  // ===== MMA issuer =====
            constexpr uint32_t idesc = umma_idesc_bf16(BM, BNL);
            for (int kb = 0; kb < KB; ++kb) {
                const int s = kb % NST;
                const uint32_t ph = (kb / NST) & 1;
                mbar_wait(full_bar(s), ph);
                tcgen05_fence_after();
                const uint32_t a_src = base + s * STAGE, b_src = a_src + A_BYTES;
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t adesc = umma_desc_sw128(a_src + k * UMMA_K * 2);
                    const uint64_t bdesc = umma_desc_sw128(b_src + k * UMMA_K * 2);
                    umma_bf16(tmem_base, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                }
                umma_commit(empty_bar(s));
            }
            umma_commit(tfull_bar);
        }
    }

    // ===== epilogue (warps 2..9); warps 0/1 only take part in the cluster barriers =====
    const bool epi = warp >= 2 && live;
    const int q = warp & 3;
    const int h = epi ? ((warp - 2) >> 2) : 0;
    const int row = q * 32 + lane;
    const int swz = row & 7;
    const int pidx = (int)rank * 2 + h;
    float v[64];
    if (epi) {
        mbar_wait(tfull_bar, 0);
        tcgen05_fence_after();
        LNK_TS(3);
        mbar_wait(resid_bar, 0);
        LNK_TS(4);
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(h * 64 + c0), r);
            const uint8_t* box = resid_sm + (2 * h + c0 / 32) * (BM * 128) + row * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float4 rv = *reinterpret_cast<const float4*>(box + ((c ^ swz) << 4));
                const int j = c0 + 4 * c;
                const float4 bv = *reinterpret_cast<const float4*>(prm + h * 64 + j);
                add3_f32x4(v + j, r + 4 * c, bv, rv);
            }
        }
        float mean, m2;
        ln_local_stats(v, mean, m2);
        LNK_TS(5);
        asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");   // phase 0: the peer is running
        part1[pidx * BM + row] = make_float2(mean, m2);
        st_async_peer_f32x2(smem_u32(&part1[pidx * BM + row]), stat_bar(0), rank ^ 1u, mean, m2);
        if (threadIdx.x == 64) {
            mbar_expect_tx(stat_bar(0), 2048);
            // chained GEMM: expect the peer's half of the normalised tile.  The peer sends it after it has received THESE
            // statistics, which leave after this CTA's GEMM has completed: the ring stages it lands in are free by then.
            if (chain) mbar_expect_tx(a2_peer_bar, 2 * 16384);
        }
        LNK_TS(6);
        asm volatile("bar.sync 1, 256;" ::: "memory");   // this CTA's two groups per row
        mbar_wait(stat_bar(0), 0);                       // the peer's two groups
        LNK_TS(7);
    } else {
        __syncwarp();
        asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    }
    __syncwarp();
    if (epi) ln_normalise(v, part1, row, prm + BNL + h * 64, prm + 2 * BNL + h * 64);
    if (g2) {   // final LayerNorm of the stack on top (uniform branch)
        if (epi) {
            float mean, m2;
            ln_local_stats(v, mean, m2);
            part2[pidx * BM + row] = make_float2(mean, m2);
            st_async_peer_f32x2(smem_u32(&part2[pidx * BM + row]), stat_bar(1), rank ^ 1u, mean, m2);
            if (threadIdx.x == 64) mbar_expect_tx(stat_bar(1), 2048);
            asm volatile("bar.sync 1, 256;" ::: "memory");
            mbar_wait(stat_bar(1), 0);
        }
        __syncwarp();
        if (epi) ln_normalise(v, part2, row, prm + 3 * BNL + h * 64, prm + 4 * BNL + h * 64);
    }
    if (chain && live && warp == 1 && lane == 0) {
        // chained GEMM:
        // q2 = LN(x) . W2^T with A = the full 128 x 256 bf16 tile (own + peer halves) in ring stages 0-1
        constexpr uint32_t idesc2 = umma_idesc_bf16(BM, BNL);
        mbar_wait(w2_bar, 0);
        mbar_wait(a2_own_bar, 0);
        mbar_wait(a2_peer_bar, 0);
        tcgen05_fence_after();
#pragma unroll
        for (int kb = 0; kb < 4; ++kb)
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k)
                umma_bf16(tmem_base + (uint32_t)BNL, umma_desc_sw128(base + kb * 16384 + k * UMMA_K * 2),
                          umma_desc_sw128(base + 2 * STAGE + kb * 16384 + k * UMMA_K * 2), idesc2, (kb | k) != 0 ? 1u : 0u);
        umma_commit(acc2_bar);
    }
    if (epi) {
        // fp32 tile back into the residual boxes (in place), bf16 tile into the idle ring: K-block slots 2*rank + h of
        // the 128 x 256 tile that the chained GEMM reads as its A operand (slots 0, 1 without a chained GEMM)
        const int slot0 = chain ? 2 * (int)rank : 0;
        LNK_TS(8);
        ln_store_tiles(v, resid_sm + 2 * h * (BM * 128), gen_base + (slot0 + h) * (BM * 128), row);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, 256;" ::: "memory");
        LNK_TS(9);
        if (threadIdx.x == 64) {
            if (chain) {
                // first (it gates the chained GEMM of the peer): this CTA's two K-blocks to the same slots of the peer, one
                // 32 KB bulk copy through DSMEM
                uint32_t r_dst, r_bar;
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r_dst) : "r"(base + slot0 * 16384), "r"(rank ^ 1u));
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r_bar) : "r"(a2_peer_bar), "r"(rank ^ 1u));
                asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(r_dst),
                             "r"(base + slot0 * 16384), "r"(2 * 16384), "r"(r_bar)
                             : "memory");
                mbar_arrive(a2_own_bar);
            }
            for (int bx = 0; bx < 4; ++bx) tma_store_2d(&tmX, resid_u32 + bx * (BM * 128), n0 + 32 * bx, m0);
            for (int hb = 0; hb < 2; ++hb) tma_store_2d(&tmXh, base + (slot0 + hb) * (BM * 128), n0 + 64 * hb, m0);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (chain) {
            // epilogue of the chained GEMM: + bias, bf16, staged in ring stage 2 (the weight slice is consumed), TMA store
            LNK_TS(10);
            mbar_wait(acc2_bar, 0);
            tcgen05_fence_after();
            LNK_TS(11);
            uint32_t pk[32];
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(BNL + h * 64 + c0), r);
                const float4* bb = reinterpret_cast<const float4*>(prm + 5 * BNL + h * 64 + c0);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 bv = bb[j >> 2];
                    __nv_bfloat162 p01 = __floats2bfloat162_rn(__uint_as_float(r[j]) + bv.x, __uint_as_float(r[j + 1]) + bv.y);
                    __nv_bfloat162 p23 = __floats2bfloat162_rn(__uint_as_float(r[j + 2]) + bv.z, __uint_as_float(r[j + 3]) + bv.w);
                    pk[(c0 + j) >> 1] = *reinterpret_cast<uint32_t*>(&p01);
                    pk[((c0 + j) >> 1) + 1] = *reinterpret_cast<uint32_t*>(&p23);
                }
            }
            uint8_t* qrow = gen_base + 2 * STAGE + h * 16384 + row * 128;
#pragma unroll
            for (int ch = 0; ch < 8; ++ch)
                *reinterpret_cast<uint4*>(qrow + ((ch ^ swz) << 4)) = make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (threadIdx.x == 64) {
                for (int hb = 0; hb < 2; ++hb) tma_store_2d(&tmQ, base + 2 * STAGE + hb * 16384, n0 + 64 * hb, m0);
                LNK_TS(12);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
    }
    // the peer reads this CTA's shared memory (bulk copy above) until its own chained GEMM has started
    if (chain) { __syncwarp(); cluster_sync_relaxed(); }
    LNK_TS(14);
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BNL)) : "memory");
    }
    if (threadIdx.x == 64 && live) {   // the staging tiles must outlive the TMA stores that read them
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        LNK_TS(13);
    }
}

// =====================================================================================================
// Fused feed-forward sub-layer for E = 256:
//     x <- LN2?( LN1( x + relu(xh W1^T + b1) W2^T + b2 ) ),  x fp32 in place, xh = bf16 copy (in place)
// The hidden activations never leave the SM.  One cluster of two CTAs per 128-row tile; CTA r owns the
// hidden units [r F/2, (r+1) F/2) in chunks of 128:
//   GEMM1(c)  acc1[c&1] (128 x 128, TMEM) = X (128 x 256, resident in smem) . W1[chunk]^T
//   epilogue  acc1 -> + b1 -> ReLU -> bf16 -> H (128 x 128, two swizzled K-blocks in smem)
//   GEMM2(c)  acc2 (128 x 256, TMEM) += H . W2[:, chunk]^T
// issued as G1(0) G1(1) G2(0) G1(2) G2(1) ... so that the tensor pipe works on the next chunk while the
// epilogue warps convert the current one.  W1/W2 stream through a ring of three 32 KB slots (TMA).  At the
// end each CTA holds a partial sum over its half of the hidden units: the half of it that belongs to the
// peer's output columns is pushed through distributed shared memory, the own half is combined with the
// peer's push, bias and residual, and the LayerNorm tail is the one of gemm_resid_ln_kernel.
#ifdef TTB_FFN_TIMELINE
// Debug build only: (event id, clock64) pairs of CTA 0 per role -> g_ffn_ts[role][256][2]
__device__ long long g_ffn_ts[3][256][2];
#define FFN_TS(role, cnt, id)                                                   \
    do {                                                                        \
        if (blockIdx.x == 0 && (cnt) < 256) {                                   \
            g_ffn_ts[role][cnt][0] = (id);                                      \
            g_ffn_ts[role][cnt][1] = clock64();                                 \
            ++(cnt);                                                            \
        }                                                                       \
    } while (0)
#else
#define FFN_TS(role, cnt, id) do { } while (0)
#endif

namespace ffn {
constexpr int NSLOT = 3, SLOT = 32768;
constexpr int X_BYTES = 65536, H_BYTES = 32768;
constexpr int THREADS = 320;
constexpr int OFF_H = X_BYTES, OFF_RING = X_BYTES + H_BYTES, OFF_PART = OFF_RING + NSLOT * SLOT;
constexpr int PART_BYTES = 4 * BM * 8;
constexpr int OFF_PRM = OFF_PART + 3 * PART_BYTES;           // three statistics tables (the third: chained pre-phase)
constexpr int OFF_B1 = OFF_PRM + 8 * 128 * 4;                // b2, g1, b1, g2, b2', pre-phase bias, g, b slices: 8 * 128 floats
constexpr int MAX_HALF = 2048;
constexpr int OFF_BAR = OFF_B1 + MAX_HALF * 4;
constexpr int SMEM = OFF_BAR + 256 + 1024;
}  // namespace ffn

__device__ __forceinline__ void st_peer_f32x4(uint32_t local_addr, uint32_t peer_rank, float a, float b, float c, float d) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_addr), "r"(peer_rank));
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(remote), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(ffn::THREADS, 1)
ffn_fused_kernel(const __grid_constant__ CUtensorMap tmXh, const __grid_constant__ CUtensorMap tmW1,
                 const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmX,
                 const float* __restrict__ bias1, const float* __restrict__ bias2, const float* __restrict__ g1,
                 const float* __restrict__ b1, const float* __restrict__ g2, const float* __restrict__ b2, RowCount rows, int F, int dbg) {
    using namespace ffn;
    const int m0 = (blockIdx.x >> 1) * BM;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int half = F / 2;                 // hidden units of this CTA
    const int n_chunks = half / 128;
    const int j_base = (int)rank * half;    // first hidden unit of this CTA
    const int n0 = (int)rank * 128;         // output columns owned by this CTA

    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gen = smem_raw + (base - raw);
    float2* part1 = reinterpret_cast<float2*>(gen + OFF_PART);
    float2* part2 = part1 + 4 * BM;
    float* prm = reinterpret_cast<float*>(gen + OFF_PRM);
    float* b1s = reinterpret_cast<float*>(gen + OFF_B1);
    const uint32_t bar_base = base + OFF_BAR;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (NSLOT + s); };
    const uint32_t x_full = bar_base + 8u * (2 * NSLOT);
    auto acc1_full = [&](int b) { return bar_base + 8u * (2 * NSLOT + 1 + b); };
    auto acc1_empty = [&](int b) { return bar_base + 8u * (2 * NSLOT + 3 + b); };
    const uint32_t h_full = bar_base + 8u * (2 * NSLOT + 5);
    const uint32_t h_empty = bar_base + 8u * (2 * NSLOT + 6);
    const uint32_t acc2_full = bar_base + 8u * (2 * NSLOT + 7);
    const uint32_t resid_bar = bar_base + 8u * (2 * NSLOT + 8);
    const uint32_t recv_bar = bar_base + 8u * (2 * NSLOT + 9);
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen + OFF_BAR + 8 * (2 * NSLOT + 10));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmXh)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW1)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW2)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmX)) : "memory");
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < NSLOT; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
            mbar_init(x_full, 1);
            for (int b = 0; b < 2; ++b) { mbar_init(acc1_full(b), 1); mbar_init(acc1_empty(b), 8); }
            mbar_init(h_full, 8);
            mbar_init(h_empty, 1);
            mbar_init(acc2_full, 1);
            mbar_init(resid_bar, 1);
            mbar_init(recv_bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (warp >= 2) {   // parameter slices (weights only: independent of earlier kernels)
        const int t = threadIdx.x - 64;
        if (t < 128) {
            prm[t] = bias2 ? __ldg(bias2 + n0 + t) : 0.f;
            prm[128 + t] = __ldg(g1 + n0 + t);
            prm[256 + t] = __ldg(b1 + n0 + t);
            prm[384 + t] = g2 ? __ldg(g2 + n0 + t) : 1.f;
            prm[512 + t] = g2 ? __ldg(b2 + n0 + t) : 0.f;
        }
        for (int i = t; i < half; i += 256) b1s[i] = bias1 ? __ldg(bias1 + j_base + i) : 0.f;
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tm_acc2 = tmem_base, tm_acc1 = tmem_base + 256u;
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");   // phase 0: "this CTA is running"
    pdl_launch_dependents();
    const int live_rows = rows.live();   // written before this programmatic chain started: fetched ahead of the wait
    pdl_wait();
#ifdef TTB_FFN_TIMELINE
    if (blockIdx.x == 0 && threadIdx.x == 96) { g_ffn_ts[2][255][0] = 7; g_ffn_ts[2][255][1] = clock64(); }
#endif
    const bool live = m0 < live_rows;   // uniform per cluster: dead tiles only take part in the barriers

    if (warp == 0) {
        if (lane == 0 && live) {  // ===== TMA producer =====
            [[maybe_unused]] int tsn = 0;
            FFN_TS(0, tsn, 1);
            mbar_expect_tx(x_full, X_BYTES);
            for (int kb = 0; kb < 4; ++kb) tma_load_2d(base + kb * 16384, &tmXh, kb * BK, m0, x_full);
            int it = 0;
            auto take_slot = [&]() -> uint32_t {
                const int s = it % NSLOT;
                const uint32_t ph = (it / NSLOT) & 1;
                mbar_wait(empty_bar(s), ph ^ 1);
                FFN_TS(0, tsn, 100 + it);
                if ((dbg & 1) && it >= NSLOT) { mbar_expect_tx(full_bar(s), 0); ++it; return 0xffffffffu; }   // timing experiment: no reload
                mbar_expect_tx(full_bar(s), SLOT);
                ++it;
                return (uint32_t)s;
            };
            auto load_w1 = [&](int c) {    // two slots, each two K-blocks [128 x 64] of the chunk's W1 rows
                const int j0 = j_base + c * 128;
                for (int j = 0; j < 2; ++j) {
                    const uint32_t sl = take_slot();
                    if (sl == 0xffffffffu) continue;
                    const uint32_t dst = base + OFF_RING + sl * SLOT;
                    tma_load_2d(dst, &tmW1, (2 * j) * BK, j0, full_bar(sl));
                    tma_load_2d(dst + 16384, &tmW1, (2 * j + 1) * BK, j0, full_bar(sl));
                }
            };
            auto load_w2 = [&](int c) {    // two slots, each one K-block [256 x 64] of W2 (two boxes of 128 rows)
                const int j0 = j_base + c * 128;
                for (int kk = 0; kk < 2; ++kk) {
                    const uint32_t sl = take_slot();
                    if (sl == 0xffffffffu) continue;
                    const uint32_t dst = base + OFF_RING + sl * SLOT;
                    tma_load_2d(dst, &tmW2, j0 + kk * BK, 0, full_bar(sl));
                    tma_load_2d(dst + 16384, &tmW2, j0 + kk * BK, 128, full_bar(sl));
                }
            };
            load_w1(0);
            for (int c = 0; c < n_chunks; ++c) {
                if (c + 1 < n_chunks) load_w1(c + 1);
                load_w2(c);
            }
            // residual tile into the (now idle) X region once every MMA has completed
            mbar_wait(acc2_full, 0);
            mbar_expect_tx(resid_bar, 65536);
            for (int bx = 0; bx < 4; ++bx) tma_load_2d(base + bx * 16384, &tmX, n0 + 32 * bx, m0, resid_bar);
        }
    } else if (warp == 1) {
        if (lane == 0 && live) {  // ===== MMA issuer =====
            constexpr uint32_t idesc1 = umma_idesc_bf16(BM, 128);
            constexpr uint32_t idesc2 = umma_idesc_bf16(BM, 256);
            int it = 0;
            [[maybe_unused]] int tsn = 0;
            FFN_TS(1, tsn, 1);
            mbar_wait(x_full, 0);
            tcgen05_fence_after();
            FFN_TS(1, tsn, 2);
            auto gemm1 = [&](int c) {
                const int b = c & 1;
                mbar_wait(acc1_empty(b), ((c >> 1) & 1) ^ 1);
                tcgen05_fence_after();
                FFN_TS(1, tsn, 1000 + c);
                const uint32_t d = tm_acc1 + (uint32_t)(128 * b);
                for (int j = 0; j < 2; ++j, ++it) {
                    const int s = it % NSLOT;
                    mbar_wait(full_bar(s), (it / NSLOT) & 1);
                    tcgen05_fence_after();
                    FFN_TS(1, tsn, 2000 + it);
                    const uint32_t slot = base + OFF_RING + s * SLOT;
#pragma unroll
                    for (int kq = 0; kq < 2; ++kq) {
                        const int kb = 2 * j + kq;
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k) {
                            const uint64_t adesc = umma_desc_sw128(base + kb * 16384 + k * UMMA_K * 2);
                            const uint64_t bdesc = umma_desc_sw128(slot + kq * 16384 + k * UMMA_K * 2);
                            umma_bf16(d, adesc, bdesc, idesc1, (kb | k) != 0 ? 1u : 0u);
                        }
                    }
                    umma_commit(empty_bar(s));
                }
                umma_commit(acc1_full(b));
            };
            auto gemm2 = [&](int c) {
                mbar_wait(h_full, c & 1);
                tcgen05_fence_after();
                FFN_TS(1, tsn, 3000 + c);
                for (int kk = 0; kk < 2; ++kk, ++it) {
                    const int s = it % NSLOT;
                    mbar_wait(full_bar(s), (it / NSLOT) & 1);
                    tcgen05_fence_after();
                    FFN_TS(1, tsn, 2000 + it);
                    const uint32_t slot = base + OFF_RING + s * SLOT;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t adesc = umma_desc_sw128(base + OFF_H + kk * 16384 + k * UMMA_K * 2);
                        const uint64_t bdesc = umma_desc_sw128(slot + k * UMMA_K * 2);
                        umma_bf16(tm_acc2, adesc, bdesc, idesc2, (c | kk | k) != 0 ? 1u : 0u);
                    }
                    umma_commit(empty_bar(s));
                }
                umma_commit(h_empty);
            };
            gemm1(0);
            for (int c = 0; c < n_chunks; ++c) {
                if (c + 1 < n_chunks) gemm1(c + 1);
                gemm2(c);
            }
            umma_commit(acc2_full);
            FFN_TS(1, tsn, 9);
        }
    }

    // ===== epilogue warps 2..9: thread = (row, 64-column half hh) =====
    [[maybe_unused]] int tse = 0;
    [[maybe_unused]] const bool ts_on = threadIdx.x == 64;
    const bool epi = warp >= 2 && live;
    const int q = warp & 3;
    const int hh = warp >= 2 ? ((warp - 2) >> 2) : 0;
    const int row = q * 32 + lane;
    const int swz = row & 7;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    if (epi) {
        for (int c = 0; c < n_chunks; ++c) {
            const int b = c & 1;
            if (ts_on) FFN_TS(2, tse, 100 + c);
            mbar_wait(acc1_full(b), (c >> 1) & 1);
            tcgen05_fence_after();
            if (ts_on) FFN_TS(2, tse, 200 + c);
            uint32_t pk[32];   // 64 bf16 values
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32(tm_acc1 + lane_base + (uint32_t)(128 * b + hh * 64 + c0), r);
                const float4* bb = reinterpret_cast<const float4*>(b1s + c * 128 + hh * 64 + c0);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 bv = bb[j >> 2];
                    const float v0 = fmaxf(__uint_as_float(r[j]) + bv.x, 0.f);
                    const float v1 = fmaxf(__uint_as_float(r[j + 1]) + bv.y, 0.f);
                    const float v2 = fmaxf(__uint_as_float(r[j + 2]) + bv.z, 0.f);
                    const float v3 = fmaxf(__uint_as_float(r[j + 3]) + bv.w, 0.f);
                    __nv_bfloat162 p01 = __floats2bfloat162_rn(v0, v1), p23 = __floats2bfloat162_rn(v2, v3);
                    pk[(c0 + j) >> 1] = *reinterpret_cast<uint32_t*>(&p01);
                    pk[((c0 + j) >> 1) + 1] = *reinterpret_cast<uint32_t*>(&p23);
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc1_empty(b));        // accumulator buffer may be overwritten
            if (ts_on) FFN_TS(2, tse, 300 + c);
            mbar_wait(h_empty, (c & 1) ^ 1);                  // GEMM2 of the previous chunk has read H
            if (ts_on) FFN_TS(2, tse, 400 + c);
            uint8_t* hrow = gen + OFF_H + hh * 16384 + row * 128;
#pragma unroll
            for (int ch = 0; ch < 8; ++ch)
                *reinterpret_cast<uint4*>(hrow + ((ch ^ swz) << 4)) = make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(h_full);
            if (ts_on) FFN_TS(2, tse, 500 + c);
        }
        mbar_wait(acc2_full, 0);
        tcgen05_fence_after();
        if (ts_on) FFN_TS(2, tse, 600);
    }
    // ---- cross-CTA reduction of the two partial sums -------------------------------------------------
    // Each CTA stages the half of its partial sum that belongs to the peer's output columns in its own shared
    // memory (idle ring slots 1-2) and ships it with one asynchronous bulk copy per 16 KB into the peer's
    // receive buffer (idle H + ring slot 0); the copy signals the peer's recv_bar.  Cluster barrier A ("my main
    // loop is over, my buffers may be written") is split into arrive / wait around the staging.
    uint8_t* recv = gen + OFF_H;             // [128 rows][32 chunks of 16 B], chunk index XOR (row & 31)
    uint8_t* send = gen + OFF_RING + SLOT;   // same layout
    if (threadIdx.x == 64 && live) mbar_expect_tx(recv_bar, 65536);
    __syncwarp();
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");     // phase 0
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");   // barrier A (arrive)
    if (epi) {
        const int pcol = (int)(rank ^ 1u) * 128 + hh * 64;   // the peer's output columns handled by this thread
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
            uint32_t r[32];
            tmem_ld_32x32(tm_acc2 + lane_base + (uint32_t)(pcol + c0), r);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int chunk = hh * 16 + (c0 >> 2) + i;
                *reinterpret_cast<uint4*>(send + row * 512 + ((chunk ^ (row & 31)) << 4)) = make_uint4(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    __syncwarp();
    if (ts_on) FFN_TS(2, tse, 700);
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");     // barrier A (wait): the peer's buffers are free
    if (ts_on) FFN_TS(2, tse, 701);
    if (threadIdx.x == 64 && live) {
        uint32_t r_recv, r_bar;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r_recv) : "r"(base + OFF_H), "r"(rank ^ 1u));
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r_bar) : "r"(recv_bar), "r"(rank ^ 1u));
        for (int i = 0; i < 4; ++i)
            asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(r_recv + i * 16384),
                         "r"(base + OFF_RING + SLOT + i * 16384), "r"(16384), "r"(r_bar)
                         : "memory");
    }
    float v[64];
    const int pidx = (int)rank * 2 + hh;
    if (epi) {
        mbar_wait(resid_bar, 0);
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
            uint32_t r[32];
            tmem_ld_32x32(tm_acc2 + lane_base + (uint32_t)(n0 + hh * 64 + c0), r);
            const uint8_t* box = gen + (2 * hh + c0 / 32) * 16384 + row * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float4 rv = *reinterpret_cast<const float4*>(box + ((c ^ swz) << 4));
                const int j = c0 + 4 * c;
                const float4 bv = *reinterpret_cast<const float4*>(prm + hh * 64 + j);
                add3_f32x4(v + j, r + 4 * c, bv, rv);
            }
        }
        mbar_wait(recv_bar, 0);   // the peer's partial sum has landed (its flight overlapped the loads above)
        if (ts_on) FFN_TS(2, tse, 702);
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const int chunk = hh * 16 + c;
            const float4 pv = *reinterpret_cast<const float4*>(recv + row * 512 + ((chunk ^ (row & 31)) << 4));
            {
                const float2 lo = fadd2(make_float2(v[4 * c], v[4 * c + 1]), make_float2(pv.x, pv.y));
                const float2 hi = fadd2(make_float2(v[4 * c + 2], v[4 * c + 3]), make_float2(pv.z, pv.w));
                v[4 * c] = lo.x; v[4 * c + 1] = lo.y; v[4 * c + 2] = hi.x; v[4 * c + 3] = hi.y;
            }
        }
        float mean, m2;
        ln_local_stats(v, mean, m2);
        ln_publish(part1, pidx, row, rank, mean, m2);
    }
    __syncwarp();
    if (ts_on) FFN_TS(2, tse, 800);
    cluster_sync_all();                                                         // barrier C
    if (ts_on) FFN_TS(2, tse, 801);
    if (epi) ln_normalise(v, part1, row, prm + 128 + hh * 64, prm + 256 + hh * 64);
    if (ts_on) FFN_TS(2, tse, 810);
    if (g2) {
        if (epi) {
            float mean, m2;
            ln_local_stats(v, mean, m2);
            ln_publish(part2, pidx, row, rank, mean, m2);
        }
        __syncwarp();
        cluster_sync_all();
        if (epi) ln_normalise(v, part2, row, prm + 384 + hh * 64, prm + 512 + hh * 64);
    }
    if (ts_on) FFN_TS(2, tse, 811);
    if (epi) {
        // fp32 tile back into the residual boxes (X region, in place), bf16 tile into ring slot 1 (the send buffer:
        // the peer has consumed it before it arrived at barrier C)
        ln_store_tiles(v, gen + 2 * hh * 16384, gen + OFF_RING + SLOT + hh * 16384, row);
        if (ts_on) FFN_TS(2, tse, 820);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (ts_on) FFN_TS(2, tse, 830);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (threadIdx.x == 64) {
            if (ts_on) FFN_TS(2, tse, 850);
            for (int bx = 0; bx < 4; ++bx) tma_store_2d(&tmX, base + bx * 16384, n0 + 32 * bx, m0);
            for (int hb = 0; hb < 2; ++hb) tma_store_2d(&tmXh, base + OFF_RING + SLOT + hb * 16384, n0 + 64 * hb, m0);
            if (ts_on) FFN_TS(2, tse, 860);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            if (ts_on) FFN_TS(2, tse, 900);
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// =====================================================================================================
// Fused feed-forward sub-layer on CTA PAIRS (tcgen05 cta_group::2), same contract as ffn_fused_kernel.
// One cluster of FOUR CTAs per 256-row block: rank = 2 p + t, t = row tile (128 rows) and position in the MMA pair,
// p = half of the hidden units.  The pair {2p, 2p+1} runs M = 256 MMAs: each CTA keeps its own 128 rows of X / H as
// the A operand and stages only HALF of every weight tile (B operand: W1 chunk 64 of 128 hidden rows, W2 chunk 128 of
// 256 output rows), so the shared-memory and L2 traffic of the weights per row halves against the cta_group::1 kernel
// (whose main loop is bound by exactly that traffic).  The even CTA of a pair issues every MMA; its mbarriers collect
// the TMA bytes of both CTAs and the "H written" / "accumulator drained" arrivals of both CTAs' epilogue warps;
// tcgen05.commit multicasts the "slot free" / "accumulator ready" signals to both.  The partial sums over the two
// hidden halves are exchanged between ranks r and r ^ 2 (same rows) exactly as in ffn_fused_kernel.
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    // default semantics (release at CTA scope), like CUTLASS's ClusterBarrier::arrive: the data handed over is either
    // tensor memory (tcgen05.fence::before_thread_sync) or shared memory already fenced into the async proxy; a
    // cluster-scope release here stalls the arriving thread for ~1000 cycles per arrival
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {   // acquires arrivals of the peer CTA
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
// TMA load into this CTA's shared memory whose bytes are counted on an mbarrier of the pair's even CTA
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar_cluster_addr) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar_cluster_addr)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t cta_mask) {   // same barrier offset in every CTA of the mask
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(cta_mask)
                 : "memory");
}

// A operand from tensor memory (this CTA's 128 rows, 16 K elements = 8 columns per instruction), B from shared memory
__device__ __forceinline__ void umma_bf16_pair_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16,"
        " %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
        "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// one K-block (64 bf16 = 32 words of this thread's row, 128-byte swizzle) from shared memory into 32 tensor-memory columns
__device__ __forceinline__ void smem_kblock_to_tmem(const uint8_t* kblock, int row, uint32_t taddr) {
    const int swz = row & 7;
    uint32_t w[32];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const uint4 u = *reinterpret_cast<const uint4*>(kblock + row * 128 + ((c ^ swz) << 4));
        w[4 * c] = u.x; w[4 * c + 1] = u.y; w[4 * c + 2] = u.z; w[4 * c + 3] = u.w;
    }
    tmem_st_32x32(taddr, w);
}

__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(ffn::THREADS, 1)
ffn_pair_kernel(const __grid_constant__ CUtensorMap tmXh, const __grid_constant__ CUtensorMap tmW1h,
                const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmX,
                const float* __restrict__ bias1, const float* __restrict__ bias2, const float* __restrict__ g1,
                const float* __restrict__ b1, const float* __restrict__ g2, const float* __restrict__ b2, RowCount rows, int F,
                const __grid_constant__ CUtensorMap tmAtt, const __grid_constant__ CUtensorMap tmWoh,
                const float* __restrict__ bias_o, const float* __restrict__ g0, const float* __restrict__ b0, int chain) {
    using namespace ffn;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const uint32_t t = rank & 1u, p = rank >> 1;      // row tile / position in the MMA pair, hidden half
    const uint32_t leader = rank & ~1u;               // even CTA of the pair: issues the MMAs, owns the pair's barriers
    const uint32_t xpeer = rank ^ 2u;                 // same rows, other hidden half
    const uint16_t pair_mask = (uint16_t)(3u << leader);
    const int mblk = (blockIdx.x >> 2) * (2 * BM);
    const int m0 = mblk + (int)t * BM;
    const int half = F / 2;                 // hidden units of this pair
    const int n_chunks = half / 128;
    const int j_base = (int)p * half;       // first hidden unit of this pair
    const int n0 = (int)p * 128;            // output columns finalised by this CTA

    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gen = smem_raw + (base - raw);
    float2* part1 = reinterpret_cast<float2*>(gen + OFF_PART);
    float2* part2 = part1 + 4 * BM;
    float2* part0 = part2 + 4 * BM;         // statistics of the chained pre-phase
    float* prm = reinterpret_cast<float*>(gen + OFF_PRM);
    float* b1s = reinterpret_cast<float*>(gen + OFF_B1);
    const uint32_t bar_base = base + OFF_BAR;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };                           // used in the even CTA only
    auto empty_bar = [&](int s) { return bar_base + 8u * (NSLOT + s); };
    const uint32_t x_full = bar_base + 8u * (2 * NSLOT);   // chained: even CTA only (att tiles of both CTAs); else local (own X tile)
    auto acc1_full = [&](int b) { return bar_base + 8u * (2 * NSLOT + 1 + b); };
    auto acc1_empty = [&](int b) { return bar_base + 8u * (2 * NSLOT + 3 + b); };       // even CTA only (16 arrivals)
    const uint32_t h_full = bar_base + 8u * (2 * NSLOT + 5);                             // even CTA only (16 arrivals)
    const uint32_t h_empty = bar_base + 8u * (2 * NSLOT + 6);
    const uint32_t acc2_full = bar_base + 8u * (2 * NSLOT + 7);
    const uint32_t resid_bar = bar_base + 8u * (2 * NSLOT + 8);
    const uint32_t recv_bar = bar_base + 8u * (2 * NSLOT + 9);
    // chained pre-phase (x <- LN0(x + att Wo^T + bo) computed by this kernel, see below)
    const uint32_t pre_full = bar_base + 8u * (2 * NSLOT + 10);     // even CTA only: Wo halves of both CTAs have landed
    const uint32_t pre_acc = bar_base + 8u * (2 * NSLOT + 11);      // its accumulator is complete
    const uint32_t pre_done = bar_base + 8u * (2 * NSLOT + 12);     // ring slots 1-2 (residual tile) are free again
    const uint32_t x2_recv = bar_base + 8u * (2 * NSLOT + 13);      // the partner's half of the normalised tile has landed
    const uint32_t x2_full = bar_base + 8u * (2 * NSLOT + 14);      // even CTA only: both CTAs hold the A operand of GEMM1 in TMEM
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen + OFF_BAR + 8 * (2 * NSLOT + 15));
    // LayerNorm statistics of the partner CTA (same rows, other 128 columns): 256 x 8 bytes by st.async per exchange
    auto stat_bar = [&](int i) { return bar_base + 8u * (2 * NSLOT + 16 + i); };   // 0: pre-phase, 1: LayerNorm, 2: final LayerNorm

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef TTB_FFN_TIMELINE
    if (blockIdx.x == 0 && threadIdx.x == 96) { g_ffn_ts[2][253][0] = 5; g_ffn_ts[2][253][1] = clock64(); }
#endif

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmXh)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW1h)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW2)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmX)) : "memory");
        if (chain) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmAtt)) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmWoh)) : "memory");
        }
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < NSLOT; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
            mbar_init(x_full, 1);
            for (int b = 0; b < 2; ++b) { mbar_init(acc1_full(b), 1); mbar_init(acc1_empty(b), 16); }
            mbar_init(h_full, 16);
            mbar_init(h_empty, 1);
            mbar_init(acc2_full, 1);
            mbar_init(resid_bar, 1);
            mbar_init(recv_bar, 1);
            mbar_init(pre_full, 1);
            mbar_init(pre_acc, 1);
            mbar_init(pre_done, 1);
            mbar_init(x2_recv, 1);
            mbar_init(x2_full, 16);
            for (int i = 0; i < 3; ++i) mbar_init(stat_bar(i), 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    if (warp >= 2) {   // parameter slices (weights only: independent of earlier kernels)
        const int tt = threadIdx.x - 64;
        if (tt < 128) {
            prm[tt] = bias2 ? __ldg(bias2 + n0 + tt) : 0.f;
            prm[128 + tt] = __ldg(g1 + n0 + tt);
            prm[256 + tt] = __ldg(b1 + n0 + tt);
            prm[384 + tt] = g2 ? __ldg(g2 + n0 + tt) : 1.f;
            prm[512 + tt] = g2 ? __ldg(b2 + n0 + tt) : 0.f;
            if (chain) {
                prm[640 + tt] = bias_o ? __ldg(bias_o + n0 + tt) : 0.f;
                prm[768 + tt] = __ldg(g0 + n0 + tt);
                prm[896 + tt] = __ldg(b0 + n0 + tt);
            }
        }
        for (int i = tt; i < half; i += 256) b1s[i] = bias1 ? __ldg(bias1 + j_base + i) : 0.f;
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // tensor memory: acc2 (256 columns), acc1 (128, ONE buffer: the tensor pipe runs GEMM2 of the previous chunk while the
    // epilogue warps drain it), and the A operand of GEMM1 (this CTA's 128 rows x 256 bf16 = 128 columns, two K elements
    // per 32-bit cell): GEMM1 reads it from tensor memory instead of 64 KB of shared memory per hidden chunk
    const uint32_t tm_acc2 = tmem_base, tm_acc1 = tmem_base + 256u, tm_xa = tmem_base + 384u;
    // every CTA of the cluster has initialised its barriers and owns its tensor memory before any remote signal
    cluster_sync_all();                                                      // cluster barrier phase 0
#ifdef TTB_FFN_TIMELINE
    if (blockIdx.x == 0 && threadIdx.x == 96) { g_ffn_ts[2][254][0] = 6; g_ffn_ts[2][254][1] = clock64(); }
#endif
    pdl_launch_dependents();
    const int live_rows = rows.live();   // written before this programmatic chain started: fetched ahead of the wait
    const bool live = mblk < live_rows;   // uniform per cluster: dead blocks only take part in the cluster barriers

    // ---- roles, phase 1 (chained launches only): operands and GEMM of the pre-phase.  The producer / issuer threads come
    // back to the cluster barrier of the pre-phase before they start the feed-forward main loop.
    int prod_it = 0;
    [[maybe_unused]] int tsn = 0;
    const bool producer = warp == 0 && lane == 0 && live;
    const bool issuer = warp == 1 && lane == 0 && live && t == 0;
    auto take_slot = [&]() -> int {
        const int s = prod_it % NSLOT;
        const uint32_t ph = (prod_it / NSLOT) & 1;
        if (chain && prod_it == 1) mbar_wait(pre_done, 0);   // slots 1-2: the pre-phase has stored its fp32 tile
        mbar_wait(empty_bar(s), ph ^ 1);
        FFN_TS(0, tsn, 100 + prod_it);
        if (t == 0) mbar_expect_tx(full_bar(s), 2 * SLOT);
        ++prod_it;
        return s;
    };
    auto load_w1 = [&](int c) {    // this CTA's 64 of the chunk's 128 hidden rows: four K-blocks [64 x 64]
        const int s = take_slot();
        const uint32_t dst = base + OFF_RING + s * SLOT, fl = mapa_u32(full_bar(s), leader);
        const int j0 = j_base + c * 128 + (int)t * 64;
        for (int kb = 0; kb < 4; ++kb) tma_load_2d_pair(dst + kb * 8192, &tmW1h, kb * BK, j0, fl);
    };
    auto load_w2 = [&](int c) {    // this CTA's 128 of the 256 output rows: two K-blocks [128 x 64] of the chunk
        const int s = take_slot();
        const uint32_t dst = base + OFF_RING + s * SLOT, fl = mapa_u32(full_bar(s), leader);
        const int j0 = j_base + c * 128;
        for (int kk = 0; kk < 2; ++kk) tma_load_2d_pair(dst + kk * 16384, &tmW2, j0 + kk * BK, (int)t * 128, fl);
    };
    constexpr uint32_t idesc1 = umma_idesc_bf16(2 * BM, 128);
    constexpr uint32_t idesc2 = umma_idesc_bf16(2 * BM, 256);
    // Weights do not depend on earlier kernels: the out-projection tile of the pre-phase and the first W1 chunk are requested
    // ahead of the dependency wait (every barrier of the pair exists since the cluster barrier above)
    if (producer) {
        if (chain) {
            const uint32_t pf_l = mapa_u32(pre_full, leader);
            if (t == 0) mbar_expect_tx(pre_full, 2 * 32768);
            for (int kb = 0; kb < 4; ++kb) tma_load_2d_pair(base + OFF_H + kb * 8192, &tmWoh, kb * BK, n0 + (int)t * 64, pf_l);
        }
        load_w1(0);   // ring slot 0 is free from the start
    }
    pdl_wait();
#ifdef TTB_FFN_TIMELINE
    if (blockIdx.x == 0 && threadIdx.x == 96) { g_ffn_ts[2][255][0] = 7; g_ffn_ts[2][255][1] = clock64(); }
#endif

    if (producer) {   // ===== TMA producer (both CTAs of a pair: own rows of the A operand, own half of every weight tile) =====
        FFN_TS(0, tsn, 1);
        if (!chain) {   // own X tile: copied into tensor memory by this CTA's epilogue warps
            mbar_expect_tx(x_full, X_BYTES);
            for (int kb = 0; kb < 4; ++kb) tma_load_2d(base + kb * 16384, &tmXh, kb * BK, m0, x_full);
        } else {
            const uint32_t x_full_l = mapa_u32(x_full, leader);
            if (t == 0) mbar_expect_tx(x_full, 2 * X_BYTES);
            for (int kb = 0; kb < 4; ++kb) tma_load_2d_pair(base + kb * 16384, &tmAtt, kb * BK, m0, x_full_l);
            // pre-phase operands: this CTA's 64 of the pair's 128 rows of Wo are on their way into the (still idle) H region
            // since before the wait; the fp32 residual tile of its 128 output columns goes into ring slots 1-2
            mbar_expect_tx(resid_bar, 65536);
            for (int bx = 0; bx < 4; ++bx) tma_load_2d(base + OFF_RING + SLOT + bx * 16384, &tmX, n0 + 32 * bx, m0, resid_bar);
        }
    }
    if (issuer) {     // ===== MMA issuer: even CTA of the pair =====
        FFN_TS(1, tsn, 1);
        if (chain) {   // pre-phase GEMM: att (X region) . Wo[128 p .. 128 p + 128)^T -> acc1
            mbar_wait(x_full, 0);
            tcgen05_fence_after();
            FFN_TS(1, tsn, 2);
            mbar_wait(pre_full, 0);
            tcgen05_fence_after();
#pragma unroll
            for (int kb = 0; kb < 4; ++kb) {
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t adesc = umma_desc_sw128(base + kb * 16384 + k * UMMA_K * 2);
                    const uint64_t bdesc = umma_desc_sw128(base + OFF_H + kb * 8192 + k * UMMA_K * 2);
                    umma_bf16_pair(tm_acc1, adesc, bdesc, idesc1, (kb | k) != 0 ? 1u : 0u);
                }
            }
            umma_commit_pair(pre_acc, pair_mask);
        }
    }
    __syncwarp();

    // ===== epilogue warps 2..9: thread = (row, 64-column half hh) =====
    [[maybe_unused]] int tse = 0;
    [[maybe_unused]] const bool ts_on = threadIdx.x == 64;
    const bool epi = warp >= 2 && live;
    const int q = warp & 3;
    const int hh = warp >= 2 ? ((warp - 2) >> 2) : 0;
    const int row = q * 32 + lane;
    const int swz = row & 7;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    if (chain) {
        // ---- chained pre-phase: x <- LN0(x + att Wo^T + bo) for this CTA's 128 rows x 128 columns; the fp32 tile goes back
        // to global memory (it is the residual of the feed-forward block), the bf16 tile becomes K-blocks 2p, 2p+1 of the
        // A operand in the X region of this CTA and (bulk copy through DSMEM) of the partner with the other columns
        float v[64];
        const int pidx0 = (int)p * 2 + hh;
        if (epi) {
            mbar_wait(pre_acc, 0);
            tcgen05_fence_after();
            if (ts_on) FFN_TS(2, tse, 10);
            mbar_wait(resid_bar, 0);
            if (ts_on) FFN_TS(2, tse, 11);
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32(tm_acc1 + lane_base + (uint32_t)(hh * 64 + c0), r);
                const uint8_t* box = gen + OFF_RING + SLOT + (2 * hh + c0 / 32) * 16384 + row * 128;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float4 rv = *reinterpret_cast<const float4*>(box + ((c ^ swz) << 4));
                    const int j = c0 + 4 * c;
                    const float4 bv = *reinterpret_cast<const float4*>(prm + 640 + hh * 64 + j);
                    add3_f32x4(v + j, r + 4 * c, bv, rv);
                }
            }
            if (ts_on) FFN_TS(2, tse, 12);
            float mean, m2;
            ln_local_stats(v, mean, m2);
            if (ts_on) FFN_TS(2, tse, 13);
            part0[pidx0 * BM + row] = make_float2(mean, m2);
            st_async_peer_f32x2(smem_u32(&part0[pidx0 * BM + row]), stat_bar(0), xpeer, mean, m2);
            if (threadIdx.x == 64) { mbar_expect_tx(x2_recv, 32768); mbar_expect_tx(stat_bar(0), 2048); }
            // the partner's statistics only leave after its threads have seen ITS pre-phase accumulator complete, so their
            // arrival also says that the partner pair's GEMM has finished reading its X regions (written below through DSMEM)
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (ts_on) FFN_TS(2, tse, 14);
            mbar_wait(stat_bar(0), 0);
            if (ts_on) FFN_TS(2, tse, 15);
        }
        __syncwarp();
        if (epi) {
            ln_normalise(v, part0, row, prm + 768 + hh * 64, prm + 896 + hh * 64);
            if (ts_on) FFN_TS(2, tse, 16);
            ln_store_tiles(v, gen + OFF_RING + SLOT + 2 * hh * 16384, gen + (2 * (int)p + hh) * 16384, row);
            if (ts_on) FFN_TS(2, tse, 17);
            {   // own 64 columns of the normalised row -> A operand in tensor memory (K elements 128 p + 64 hh ..)
                uint32_t w[32];
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) {
                    __nv_bfloat162 pp = __floats2bfloat162_rn(v[2 * jj], v[2 * jj + 1]);
                    w[jj] = *reinterpret_cast<uint32_t*>(&pp);
                }
                tmem_st_32x32(tm_xa + lane_base + (uint32_t)(64 * (int)p + 32 * hh), w);
            }
            if (ts_on) FFN_TS(2, tse, 18);
            tcgen05_fence_before();
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (ts_on) FFN_TS(2, tse, 19);
            if (threadIdx.x == 64) {
                // the tile halves first: they gate GEMM1; the fp32 store only gates ring slots 1-2 (second weight tile)
                const uint32_t own = base + 2 * p * 16384;
                asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(mapa_u32(own, xpeer)),
                             "r"(own), "r"(32768), "r"(mapa_u32(x2_recv, xpeer))
                             : "memory");
                for (int bx = 0; bx < 4; ++bx) tma_store_2d(&tmX, base + OFF_RING + SLOT + bx * 16384, n0 + 32 * bx, m0);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            // the partner's 128 columns (K-blocks 2(1-p), 2(1-p)+1 of the X region, landed through DSMEM) -> tensor memory
            if (ts_on) FFN_TS(2, tse, 20);
            mbar_wait(x2_recv, 0);
            if (ts_on) FFN_TS(2, tse, 21);
            smem_kblock_to_tmem(gen + (2 * (int)(p ^ 1u) + hh) * 16384, row, tm_xa + lane_base + (uint32_t)(64 * (int)(p ^ 1u) + 32 * hh));
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(mapa_u32(x2_full, leader));
            if (ts_on) FFN_TS(2, tse, 22);
            if (threadIdx.x == 64) {   // ring slots 1-2 are free once the fp32 store has read them
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                mbar_arrive(pre_done);
            }
        }
    } else if (epi) {
        // own X tile (TMA, swizzled shared memory) -> A operand in tensor memory: K-blocks 2 hh, 2 hh + 1 of this thread's row
        mbar_wait(x_full, 0);
        smem_kblock_to_tmem(gen + (2 * hh) * 16384, row, tm_xa + lane_base + (uint32_t)(64 * hh));
        smem_kblock_to_tmem(gen + (2 * hh + 1) * 16384, row, tm_xa + lane_base + (uint32_t)(64 * hh + 32));
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(mapa_u32(x2_full, leader));
    }
    // ---- roles, phase 2: the feed-forward main loop
    if (producer) {
        for (int c = 0; c < n_chunks; ++c) {
            if (c + 1 < n_chunks) load_w1(c + 1);
            load_w2(c);
        }
        // residual tile into the (now idle) X region once every MMA has completed
        mbar_wait(acc2_full, 0);
        mbar_expect_tx(resid_bar, 65536);
        for (int bx = 0; bx < 4; ++bx) tma_load_2d(base + bx * 16384, &tmX, n0 + 32 * bx, m0, resid_bar);
    }
    if (issuer) {
        int it = 0;
        mbar_wait(x2_full, 0);     // the A operand of GEMM1 is complete in the tensor memory of both CTAs
        tcgen05_fence_after();
        FFN_TS(1, tsn, 3);
        auto gemm1 = [&](int c) {
            if (c > 0) mbar_wait_cluster(acc1_empty(0), (c - 1) & 1);   // the epilogue warps of both CTAs have drained chunk c-1
            tcgen05_fence_after();
            FFN_TS(1, tsn, 1000 + c);
            const uint32_t d = tm_acc1;
            const int s = it % NSLOT;
            mbar_wait(full_bar(s), (it / NSLOT) & 1);
            tcgen05_fence_after();
            FFN_TS(1, tsn, 2000 + it);
            const uint32_t slot = base + OFF_RING + s * SLOT;
#pragma unroll
            for (int kb = 0; kb < 4; ++kb) {
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t bdesc = umma_desc_sw128(slot + kb * 8192 + k * UMMA_K * 2);
                    umma_bf16_pair_ts(d, tm_xa + (uint32_t)(kb * 32 + k * 8), bdesc, idesc1, (kb | k) != 0 ? 1u : 0u);
                }
            }
            umma_commit_pair(empty_bar(s), pair_mask);
            umma_commit_pair(acc1_full(0), pair_mask);
            ++it;
        };
        auto gemm2 = [&](int c) {
            mbar_wait_cluster(h_full, c & 1);
            tcgen05_fence_after();
            FFN_TS(1, tsn, 3000 + c);
            const int s = it % NSLOT;
            mbar_wait(full_bar(s), (it / NSLOT) & 1);
            tcgen05_fence_after();
            FFN_TS(1, tsn, 2000 + it);
            const uint32_t slot = base + OFF_RING + s * SLOT;
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t adesc = umma_desc_sw128(base + OFF_H + kk * 16384 + k * UMMA_K * 2);
                    const uint64_t bdesc = umma_desc_sw128(slot + kk * 16384 + k * UMMA_K * 2);
                    umma_bf16_pair(tm_acc2, adesc, bdesc, idesc2, (c | kk | k) != 0 ? 1u : 0u);
                }
            }
            umma_commit_pair(empty_bar(s), pair_mask);
            umma_commit_pair(h_empty, pair_mask);
            ++it;
        };
        gemm1(0);
        for (int c = 0; c < n_chunks; ++c) {
            if (c + 1 < n_chunks) gemm1(c + 1);
            gemm2(c);
        }
        umma_commit_pair(acc2_full, pair_mask);
        FFN_TS(1, tsn, 9);
    }

    if (epi) {
        const uint32_t acc1_empty_l0 = mapa_u32(acc1_empty(0), leader);
        const uint32_t h_full_l = mapa_u32(h_full, leader);
        for (int c = 0; c < n_chunks; ++c) {
            if (ts_on) FFN_TS(2, tse, 100 + c);
            mbar_wait(acc1_full(0), c & 1);
            tcgen05_fence_after();
            if (ts_on) FFN_TS(2, tse, 200 + c);
            uint32_t pk[32];   // 64 bf16 values
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32(tm_acc1 + lane_base + (uint32_t)(hh * 64 + c0), r);
                const float4* bb = reinterpret_cast<const float4*>(b1s + c * 128 + hh * 64 + c0);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 bv = bb[j >> 2];
                    const float v0 = fmaxf(__uint_as_float(r[j]) + bv.x, 0.f);
                    const float v1 = fmaxf(__uint_as_float(r[j + 1]) + bv.y, 0.f);
                    const float v2 = fmaxf(__uint_as_float(r[j + 2]) + bv.z, 0.f);
                    const float v3 = fmaxf(__uint_as_float(r[j + 3]) + bv.w, 0.f);
                    __nv_bfloat162 p01 = __floats2bfloat162_rn(v0, v1), p23 = __floats2bfloat162_rn(v2, v3);
                    pk[(c0 + j) >> 1] = *reinterpret_cast<uint32_t*>(&p01);
                    pk[((c0 + j) >> 1) + 1] = *reinterpret_cast<uint32_t*>(&p23);
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(acc1_empty_l0);   // accumulator may be overwritten
            if (ts_on) FFN_TS(2, tse, 300 + c);
            mbar_wait(h_empty, (c & 1) ^ 1);                  // GEMM2 of the previous chunk has read H (of both CTAs)
            if (ts_on) FFN_TS(2, tse, 400 + c);
            uint8_t* hrow = gen + OFF_H + hh * 16384 + row * 128;
#pragma unroll
            for (int ch = 0; ch < 8; ++ch)
                *reinterpret_cast<uint4*>(hrow + ((ch ^ swz) << 4)) = make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(h_full_l);
            if (ts_on) FFN_TS(2, tse, 500 + c);
        }
        mbar_wait(acc2_full, 0);
        tcgen05_fence_after();
        if (ts_on) FFN_TS(2, tse, 600);
    }
    // ---- reduction of the two partial sums (ranks r and r ^ 2), see ffn_fused_kernel ------------------------
    uint8_t* recv = gen + OFF_H;             // [128 rows][32 chunks of 16 B], chunk index XOR (row & 31)
    uint8_t* send = gen + OFF_RING + SLOT;   // same layout
    if (threadIdx.x == 64 && live) mbar_expect_tx(recv_bar, 65536);
    __syncwarp();
    // barrier A ("my main loop is over: my H / ring may be written"), split into arrive / wait around the staging; an
    // execution hand-over (nothing is published by it), hence relaxed: the release form costs 1.9 k cycles here.
    // (Measured and not adopted: the partial sums sent straight from registers with st.async.v4 instead of staging tile +
    // bulk copy -- 16 instructions per thread take 5.8 k cycles to issue, ~11 B/clk against ~21 B/clk of the bulk copy.)
    asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
    if (epi) {
        const int pcol = (int)(p ^ 1u) * 128 + hh * 64;   // the partner's output columns handled by this thread
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
            uint32_t r[32];
            tmem_ld_32x32(tm_acc2 + lane_base + (uint32_t)(pcol + c0), r);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int chunk = hh * 16 + (c0 >> 2) + i;
                *reinterpret_cast<uint4*>(send + row * 512 + ((chunk ^ (row & 31)) << 4)) = make_uint4(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    __syncwarp();
    if (ts_on) FFN_TS(2, tse, 700);
    asm volatile("barrier.cluster.wait.aligned;" ::: "memory");             // barrier A (wait): the partner's buffers are free
    if (ts_on) FFN_TS(2, tse, 701);
    if (threadIdx.x == 64 && live) {
        const uint32_t r_recv = mapa_u32(base + OFF_H, xpeer), r_bar = mapa_u32(recv_bar, xpeer);
        for (int i = 0; i < 4; ++i)
            asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(r_recv + i * 16384),
                         "r"(base + OFF_RING + SLOT + i * 16384), "r"(16384), "r"(r_bar)
                         : "memory");
    }
    float v[64];
    const int pidx = (int)p * 2 + hh;
    if (epi) {
        mbar_wait(resid_bar, chain ? 1u : 0u);
#pragma unroll
        for (int c0 = 0; c0 < 64; c0 += 32) {
            uint32_t r[32];
            tmem_ld_32x32(tm_acc2 + lane_base + (uint32_t)(n0 + hh * 64 + c0), r);
            const uint8_t* box = gen + (2 * hh + c0 / 32) * 16384 + row * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float4 rv = *reinterpret_cast<const float4*>(box + ((c ^ swz) << 4));
                const int j = c0 + 4 * c;
                const float4 bv = *reinterpret_cast<const float4*>(prm + hh * 64 + j);
                add3_f32x4(v + j, r + 4 * c, bv, rv);
            }
        }
        mbar_wait_cluster(recv_bar, 0);   // the partner's partial sum has landed (its flight overlapped the loads above)
        if (ts_on) FFN_TS(2, tse, 702);
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const int chunk = hh * 16 + c;
            const float4 pv = *reinterpret_cast<const float4*>(recv + row * 512 + ((chunk ^ (row & 31)) << 4));
            {
                const float2 lo = fadd2(make_float2(v[4 * c], v[4 * c + 1]), make_float2(pv.x, pv.y));
                const float2 hi = fadd2(make_float2(v[4 * c + 2], v[4 * c + 3]), make_float2(pv.z, pv.w));
                v[4 * c] = lo.x; v[4 * c + 1] = lo.y; v[4 * c + 2] = hi.x; v[4 * c + 3] = hi.y;
            }
        }
        float mean, m2;
        ln_local_stats(v, mean, m2);
        part1[pidx * BM + row] = make_float2(mean, m2);
        st_async_peer_f32x2(smem_u32(&part1[pidx * BM + row]), stat_bar(1), xpeer, mean, m2);
        if (threadIdx.x == 64) mbar_expect_tx(stat_bar(1), 2048);
        if (ts_on) FFN_TS(2, tse, 800);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        mbar_wait(stat_bar(1), 0);
    }
    __syncwarp();
    if (ts_on) FFN_TS(2, tse, 801);
    if (epi) ln_normalise(v, part1, row, prm + 128 + hh * 64, prm + 256 + hh * 64);
    if (ts_on) FFN_TS(2, tse, 810);
    if (g2) {
        if (epi) {
            float mean, m2;
            ln_local_stats(v, mean, m2);
            part2[pidx * BM + row] = make_float2(mean, m2);
            st_async_peer_f32x2(smem_u32(&part2[pidx * BM + row]), stat_bar(2), xpeer, mean, m2);
            if (threadIdx.x == 64) mbar_expect_tx(stat_bar(2), 2048);
            asm volatile("bar.sync 1, 256;" ::: "memory");
            mbar_wait(stat_bar(2), 0);
        }
        __syncwarp();
        if (epi) ln_normalise(v, part2, row, prm + 384 + hh * 64, prm + 512 + hh * 64);
    }
    if (epi) {
        // fp32 tile back into the residual boxes (X region, in place), bf16 tile into ring slot 1 (the send buffer: the
        // partner's statistics are computed from the partial sum this CTA sent, so their arrival says it has been consumed)
        if (ts_on) FFN_TS(2, tse, 811);
        ln_store_tiles(v, gen + 2 * hh * 16384, gen + OFF_RING + SLOT + hh * 16384, row);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (ts_on) FFN_TS(2, tse, 850);
        if (threadIdx.x == 64) {
            for (int bx = 0; bx < 4; ++bx) tma_store_2d(&tmX, base + bx * 16384, n0 + 32 * bx, m0);
            for (int hb = 0; hb < 2; ++hb) tma_store_2d(&tmXh, base + OFF_RING + SLOT + hb * 16384, n0 + 64 * hb, m0);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    // the tensor memory of a pair is released together: both CTAs are past their last tcgen05.ld
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_relaxed();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
    // the staging tiles must outlive the TMA stores that read them: the storing thread waits here, behind the barrier and
    // the release of the tensor memory instead of in front of them
    if (threadIdx.x == 64 && live) {
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        if (ts_on) FFN_TS(2, tse, 900);
    }
}

// =====================================================================================================
// Wide projection with K = 256 on CTA pairs (cta_group::2):  C[M, N] = A[M, 256] W[N, 256]^T + bias (+ReLU), bf16 out.
// The persistent kernel re-loads the A tile for every 128-column tile of the output (QKV: six times) and every CTA
// stages whole weight tiles, so a QKV launch moves ~50 MB from L2 into shared memory and is bound by exactly that.
// Here one pair owns 256 rows x (CHUNKS x 128) columns: each CTA keeps its own 128 rows of A (64 KB, loaded once) and
// HALF of the pair's weight rows (CHUNKS x 32 KB), everything resident at once (no ring), M = 256 MMAs into CHUNKS
// accumulator tiles of 128 columns.  Traffic per QKV launch: 20 MB.  Epilogue per chunk as soon as its accumulator is
// complete: + bias -> bf16 -> swizzled staging tile in the (consumed) weight region of the chunk -> TMA store.
namespace pgk {
constexpr int THREADS = 320;
constexpr int MAXC = 3;
constexpr int OFF_W = 65536;                                  // after the A tile
constexpr int OFF_BIAS = OFF_W + MAXC * 32768;
constexpr int OFF_BAR = OFF_BIAS + MAXC * 128 * 4;
constexpr int SMEM = OFF_BAR + 128 + 1024;
}  // namespace pgk

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(pgk::THREADS, 1)
gemm_pair_k256_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmWh,
                      const __grid_constant__ CUtensorMap tmC, const float* __restrict__ bias, RowCount rows, int chunks,
                      int pairs_per_block, int relu) {
    using namespace pgk;
    uint32_t t;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(t));
    const int pair = blockIdx.x >> 1;
    const int mblk = (pair / pairs_per_block) * (2 * BM);
    const int m0 = mblk + (int)t * BM;
    const int col0 = (pair % pairs_per_block) * chunks * 128;   // first output column of the pair
    const uint16_t pair_mask = 3;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gen = smem_raw + (base - raw);
    float* bias_sm = reinterpret_cast<float*>(gen + OFF_BIAS);
    const uint32_t bar_base = base + OFF_BAR;
    const uint32_t a_full = bar_base;                                       // even CTA: A tiles of both CTAs
    auto w_full = [&](int c) { return bar_base + 8u * (1 + c); };          // even CTA: weight halves of chunk c
    auto acc_full = [&](int c) { return bar_base + 8u * (1 + MAXC + c); }; // both CTAs: accumulator of chunk c complete
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen + OFF_BAR + 8 * (1 + 2 * MAXC));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmWh)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmC)) : "memory");
    }
    if (warp == 1) {
        if (lane == 0) {
            mbar_init(a_full, 1);
            for (int c = 0; c < MAXC; ++c) { mbar_init(w_full(c), 1); mbar_init(acc_full(c), 1); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    if (warp >= 2) {
        const int tt = threadIdx.x - 64;
        for (int i = tt; i < chunks * 128; i += 256) bias_sm[i] = bias ? __ldg(bias + col0 + i) : 0.f;
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    cluster_sync_all();   // both CTAs have initialised their barriers and own their tensor memory
    pdl_launch_dependents();
    // the weights do not depend on earlier kernels: they are requested before the dependency wait
    const bool producer = warp == 0 && lane == 0;
    if (producer) {
        for (int c = 0; c < chunks; ++c) {
            const uint32_t wl = mapa_u32(w_full(c), 0);
            if (t == 0) mbar_expect_tx(w_full(c), 2 * 32768);
            for (int kb = 0; kb < 4; ++kb)
                tma_load_2d_pair(base + OFF_W + c * 32768 + kb * 8192, &tmWh, kb * BK, col0 + c * 128 + (int)t * 64, wl);
        }
    }
    // The live row count is written by the bookkeeping kernel that ends the previous decoding iteration (or opens this
    // one); the launch right behind that kernel is a fully serialised one, so no kernel of a programmatic chain can run
    // ahead of it: the count is fetched before the dependency wait (its ~1000-cycle round trip leaves the critical path).
    const int live_rows = rows.live();
    pdl_wait();
    const bool live = mblk < live_rows;   // uniform per pair
    if (producer) {
        if (live) {
            const uint32_t al = mapa_u32(a_full, 0);
            if (t == 0) mbar_expect_tx(a_full, 2 * 65536);
            for (int kb = 0; kb < 4; ++kb) tma_load_2d_pair(base + kb * 16384, &tmA, kb * BK, m0, al);
        } else if (t == 0) {
            for (int c = 0; c < chunks; ++c) mbar_wait(w_full(c), 0);   // requested weights must land before the pair may exit
        }
    } else if (warp == 1 && lane == 0 && live && t == 0) {   // ===== MMA issuer: even CTA =====
        constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, 128);
        mbar_wait(a_full, 0);
        tcgen05_fence_after();
        for (int c = 0; c < chunks; ++c) {
            mbar_wait(w_full(c), 0);
            tcgen05_fence_after();
#pragma unroll
            for (int kb = 0; kb < 4; ++kb) {
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t adesc = umma_desc_sw128(base + kb * 16384 + k * UMMA_K * 2);
                    const uint64_t bdesc = umma_desc_sw128(base + OFF_W + c * 32768 + kb * 8192 + k * UMMA_K * 2);
                    umma_bf16_pair(tmem_base + (uint32_t)(c * 128), adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                }
            }
            umma_commit_pair(acc_full(c), pair_mask);
        }
    }
    // ===== epilogue warps 2..9: thread = (row, 64-column half hh of the chunk) =====
    if (warp >= 2 && live) {
        const int q = warp & 3, hh = (warp - 2) >> 2;
        const int row = q * 32 + lane, swz = row & 7;
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        for (int c = 0; c < chunks; ++c) {
            mbar_wait(acc_full(c), 0);
            tcgen05_fence_after();
            uint32_t pk[32];   // 64 bf16 values
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32(tmem_base + lane_base + (uint32_t)(c * 128 + hh * 64 + c0), r);
                const float4* bb = reinterpret_cast<const float4*>(bias_sm + c * 128 + hh * 64 + c0);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 bv = bb[j >> 2];
                    float v0 = __uint_as_float(r[j]) + bv.x, v1 = __uint_as_float(r[j + 1]) + bv.y;
                    float v2 = __uint_as_float(r[j + 2]) + bv.z, v3 = __uint_as_float(r[j + 3]) + bv.w;
                    if (relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f); }
                    __nv_bfloat162 p01 = __floats2bfloat162_rn(v0, v1), p23 = __floats2bfloat162_rn(v2, v3);
                    pk[(c0 + j) >> 1] = *reinterpret_cast<uint32_t*>(&p01);
                    pk[((c0 + j) >> 1) + 1] = *reinterpret_cast<uint32_t*>(&p23);
                }
            }
            // the weight halves of chunk c (32 KB) are consumed: they become the two [128 x 64] output boxes of the chunk
            uint8_t* orow = gen + OFF_W + c * 32768 + hh * 16384 + row * 128;
#pragma unroll
            for (int ch = 0; ch < 8; ++ch)
                *reinterpret_cast<uint4*>(orow + ((ch ^ swz) << 4)) = make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (threadIdx.x == 64) {
                for (int hb = 0; hb < 2; ++hb) tma_store_2d(&tmC, base + OFF_W + c * 32768 + hb * 16384, col0 + c * 128 + hb * 64, m0);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_relaxed();   // the tensor memory of a pair is released together (execution order only: no release fence)
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
    if (threadIdx.x == 64 && live) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging tiles outlive their stores
}

// =====================================================================================================
// Vocabulary projection + arg-max for the greedy loop:  pred[row] = argmax_v (xh[row] . Wc[v] + bc[v])
// (first maximal index, like torch.argmax).  The logits never leave the SM: one CTA per 128 rows keeps
// the whole [V x K] classifier weight and its A tile in shared memory (K = 256: 64 KB + 144 KB for V = 288),
// accumulates all V_pad <= 512 columns in TMEM (one N <= 256 MMA group plus a tail group), and each row's
// maximum is found by two threads scanning disjoint column ranges straight out of TMEM.
//
// The same kernel draws the sampling decoding's tokens (DESIGN.md section 15) with another epilogue, EPI:
//   CLS_ARGMAX       the arg-max above (the greedy loops);
//   CLS_SAMPLE       top_k = 0: one pass, z = (logit + bias) / T + Gumbel noise (one Philox call per 4 columns), running
//                    arg-max of z; the halves merge as the arg-max does (a strictly larger upper-half z wins);
//   CLS_SAMPLE_TOPK  1 <= top_k <= 8: the sorted 8-entry list pass of classifier_stats_kernel, the two lists merged in
//                    shared memory (the A tiles are dead by then), noise for the first top_k entries only.
namespace cls {
constexpr int THREADS = 320;
enum Epi : int { CLS_ARGMAX = 0, CLS_SAMPLE = 1, CLS_SAMPLE_TOPK = 2 };
constexpr int SAMPLE_KT = 8;
}
template <int EPI>
__global__ void __launch_bounds__(cls::THREADS, 1)
classifier_argmax_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                         const __grid_constant__ CUtensorMap tmWtail, const float* __restrict__ bias, int* __restrict__ pred,
                         RowCount rows, int V, int V_pad, int KB, SampleArgs sa) {
    const int m0 = blockIdx.x * BM;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gen = smem_raw + (base - raw);
    const int w_kb_bytes = V_pad * 128;                       // one K-block of the weight: V_pad rows x 64 bf16
    const uint32_t w_base = base + KB * A_BYTES;
    float* bias_sm = reinterpret_cast<float*>(gen + KB * A_BYTES + KB * w_kb_bytes);
    float2* half_best = reinterpret_cast<float2*>(bias_sm + V_pad);
    const uint32_t bar_base = base + KB * A_BYTES + KB * w_kb_bytes + V_pad * 4 + BM * 8;
    auto full_bar = [&](int kb) { return bar_base + 8u * kb; };
    const uint32_t tfull_bar = bar_base + 8u * 16;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen + (bar_base - base) + 8 * 17);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_main = V_pad < 256 ? V_pad : 256, n_tail = V_pad - n_main;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmWtail)) : "memory");
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int kb = 0; kb < KB; ++kb) mbar_init(full_bar(kb), 1);
            mbar_init(tfull_bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (warp >= 2)
        for (int c = threadIdx.x - 64; c < V_pad; c += 256) bias_sm[c] = (bias && c < V) ? __ldg(bias + c) : 0.f;
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_launch_dependents();
    const int M = rows.live();   // written before this programmatic chain started (see gemm_pair_k256_kernel): fetched ahead of the wait
    pdl_wait();
    const bool live = m0 < M;

    if (warp == 0) {
        if (lane == 0 && live) {  // ===== TMA producer: everything at once, one barrier per K-block =====
            for (int kb = 0; kb < KB; ++kb) {
                mbar_expect_tx(full_bar(kb), A_BYTES + w_kb_bytes);
                tma_load_2d(base + kb * A_BYTES, &tmA, kb * BK, m0, full_bar(kb));
                const uint32_t wdst = w_base + kb * w_kb_bytes;
                int r0 = 0;
                for (; r0 + 128 <= V_pad; r0 += 128) tma_load_2d(wdst + r0 * 128, &tmW, kb * BK, r0, full_bar(kb));
                if (r0 < V_pad) tma_load_2d(wdst + r0 * 128, &tmWtail, kb * BK, r0, full_bar(kb));
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && live) {  // ===== MMA issuer =====
            const uint32_t idesc_main = umma_idesc_bf16(BM, n_main);
            const uint32_t idesc_tail = umma_idesc_bf16(BM, n_tail > 0 ? n_tail : 16);
            for (int kb = 0; kb < KB; ++kb) {
                mbar_wait(full_bar(kb), 0);
                tcgen05_fence_after();
                const uint32_t a_src = base + kb * A_BYTES, b_src = w_base + kb * w_kb_bytes;
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t adesc = umma_desc_sw128(a_src + k * UMMA_K * 2);
                    umma_bf16(tmem_base, adesc, umma_desc_sw128(b_src + k * UMMA_K * 2), idesc_main, (kb | k) != 0 ? 1u : 0u);
                    if (n_tail > 0)
                        umma_bf16(tmem_base + 256u, adesc, umma_desc_sw128(b_src + 256 * 128 + k * UMMA_K * 2), idesc_tail, (kb | k) != 0 ? 1u : 0u);
                }
            }
            umma_commit(tfull_bar);
        }
    } else if (live && EPI == cls::CLS_ARGMAX) {  // ===== arg-max: thread = (row, column range) =====
        const int q = warp & 3, hh = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        const int n32 = V_pad / 32, c_half = (n32 + 1) / 2;
        const int c_begin = hh == 0 ? 0 : c_half, c_end = hh == 0 ? c_half : n32;
        float best = -INFINITY;
        int bi = c_begin * 32;
        mbar_wait(tfull_bar, 0);
        tcgen05_fence_after();
        for (int ch = c_begin; ch < c_end; ++ch) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * 32), r);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int col = ch * 32 + j;
                const float v = __uint_as_float(r[j]) + bias_sm[col];
                if (col < V && v > best) { best = v; bi = col; }
            }
        }
        if (hh == 1) half_best[row] = make_float2(best, __int_as_float(bi));
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (hh == 0) {
            if (c_end < n32) {   // columns of the upper half exist: a strictly larger value there wins
                const float2 o = half_best[row];
                if (o.x > best) { best = o.x; bi = __float_as_int(o.y); }
            }
            if (m0 + row < M) pred[m0 + row] = bi;
        }
    } else if (live) {  // ===== draw of the sampling decoding: thread = (row, column half) =====
      if constexpr (EPI != cls::CLS_ARGMAX) {
        const int q = warp & 3, hh = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        const int grow = m0 + row;
        const int n32 = V_pad / 32, c_half = (n32 + 1) / 2;
        const int c_begin = hh == 0 ? 0 : c_half, c_end = hh == 0 ? c_half : n32;
        int4 d = make_int4(0, 0, 0, 0);
        unsigned long long key = 0;
        if (grow < M) {
            d = sa.desc[grow];
            key = sa.keys[d.x / sa.S];
        }
        const int t = d.y + 1, smp = d.x % sa.S;
        const float T = sa.temperature;
        const uint32_t tm_row = tmem_base + ((uint32_t)(q * 32) << 16);
        mbar_wait(tfull_bar, 0);
        tcgen05_fence_after();
        if constexpr (EPI == cls::CLS_SAMPLE) {
            float best = -INFINITY;
            int bi = 0x7fffffff;
            for (int ch = c_begin; ch < c_end; ++ch) {
                uint32_t r[32];
                tmem_ld_32x32(tm_row + (uint32_t)(ch * 32), r);
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const Philox4 nz = sample_noise_bits(t, smp, ch * 8 + j4, key);
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int col = ch * 32 + j4 * 4 + u;
                        const float z = (__uint_as_float(r[j4 * 4 + u]) + bias_sm[col]) / T + gumbel(nz.x[u]);
                        if (col < V && sample_better(z, col, best, bi)) { best = z; bi = col; }
                    }
                }
            }
            if (hh == 1) half_best[row] = make_float2(best, __int_as_float(bi));
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (hh == 0) {
                if (c_end < n32) {   // a strictly larger upper-half z wins (its ids are all above the lower half's)
                    const float2 o = half_best[row];
                    if (o.x > best || bi >= V) { best = o.x; bi = __float_as_int(o.y); }
                }
                if (grow < M) sa.pred[grow] = bi < V ? bi : 0;   // no candidate only with NaN logits
            }
        } else {
            constexpr int KT = cls::SAMPLE_KT;
            float* xv = reinterpret_cast<float*>(gen);                    // [2][KT][128] list values (aliases the A tiles)
            int* xi = reinterpret_cast<int*>(gen + 2 * KT * BM * 4);      // [2][KT][128] list token ids
            float tv[KT];
            int ti[KT];
#pragma unroll
            for (int i = 0; i < KT; ++i) { tv[i] = -INFINITY; ti[i] = -1; }
            for (int ch = c_begin; ch < c_end; ++ch) {
                uint32_t r[32];
                tmem_ld_32x32(tm_row + (uint32_t)(ch * 32), r);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int col = ch * 32 + j;
                    if (col < V) topk_list_insert<KT>(tv, ti, __uint_as_float(r[j]) + bias_sm[col], col);
                }
            }
#pragma unroll
            for (int i = 0; i < KT; ++i) { xv[(hh * KT + i) * BM + row] = tv[i]; xi[(hh * KT + i) * BM + row] = ti[i]; }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (hh == 0 && grow < M) {
                // merge of the two sorted lists (equal values: the lower column half first = lower token id); the first top_k
                // entries are the candidate set
                int a = 0, b = 0;
                float best = -INFINITY;
                int bi = 0x7fffffff;
#pragma unroll
                for (int j = 0; j < KT; ++j) {
                    const float va = a < KT ? xv[a * BM + row] : -INFINITY;
                    const float vb = b < KT ? xv[(KT + b) * BM + row] : -INFINITY;
                    const int ia = a < KT ? xi[a * BM + row] : -1;
                    const int ib = b < KT ? xi[(KT + b) * BM + row] : -1;
                    const bool take_a = ia >= 0 && (ib < 0 || va >= vb);
                    const float mv = take_a ? va : vb;
                    const int mi = take_a ? ia : ib;
                    a += take_a ? 1 : 0;
                    b += take_a ? 0 : 1;
                    if (j < sa.top_k && mi >= 0) {
                        const float z = mv / T + gumbel(philox_word(sample_noise_bits(t, smp, mi >> 2, key), mi & 3));
                        if (sample_better(z, mi, best, bi)) { best = z; bi = mi; }
                    }
                }
                sa.pred[grow] = bi < V ? bi : 0;
            }
        }
      }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// =====================================================================================================
// Vocabulary projection fused with the per-distribution statistics of the speculative beam search (bf16 path): the
// logits of a 128-row tile stay in tensor memory (as in classifier_argmax_kernel) and the epilogue reduces every row to
// what beam_choose / beam_expand read (beam.cu): soft-max maximum and sum, the K largest logits in descending order
// (ties: lower token id first) with their token ids, the size of the nucleus-truncated support, and the logit of the
// row's own next draft token.  The (rows x V) fp32 logits matrix never exists in memory.
//   thread = (row, half of the columns): pass 1 streams its columns through a sorted KT-entry list held in registers
//   (an element enters only when it beats the current KT-th best: ~KT (1 + ln(columns / KT)) insertions per thread),
//   the two halves meet in shared memory (the A tiles are dead once the accumulator is complete), pass 2 adds
//   exp(logit - max) over the same columns, the lower half merges the two lists and writes the results.
template <int KT>
__global__ void __launch_bounds__(cls::THREADS, 1)
classifier_stats_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                        const __grid_constant__ CUtensorMap tmWtail, const float* __restrict__ bias, RowCount rows, int V, int V_pad, int KB,
                        int K, const int* __restrict__ row_tok, float* __restrict__ tokv, float* __restrict__ lmax, float* __restrict__ lsum,
                        int* __restrict__ nkeep, float* __restrict__ topv, int* __restrict__ topi) {
    const int m0 = blockIdx.x * BM;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* gen = smem_raw + (base - raw);
    const int w_kb_bytes = V_pad * 128;
    const uint32_t w_base = base + KB * A_BYTES;
    float* bias_sm = reinterpret_cast<float*>(gen + KB * A_BYTES + KB * w_kb_bytes);
    const uint32_t bar_base = base + KB * A_BYTES + KB * w_kb_bytes + V_pad * 4 + BM * 8;
    auto full_bar = [&](int kb) { return bar_base + 8u * kb; };
    const uint32_t tfull_bar = bar_base + 8u * 16;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen + (bar_base - base) + 8 * 17);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_main = V_pad < 256 ? V_pad : 256, n_tail = V_pad - n_main;
    // exchange area of the two column halves (aliases the A tiles): [2][128] {max, token logit, found, partial sum},
    // [2][KT][128] list values, [2][KT][128] list token ids
    float4* xinfo = reinterpret_cast<float4*>(gen);
    float* xv = reinterpret_cast<float*>(gen + 4096);
    int* xi = reinterpret_cast<int*>(gen + 4096 + 2 * KT * BM * 4);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmWtail)) : "memory");
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int kb = 0; kb < KB; ++kb) mbar_init(full_bar(kb), 1);
            mbar_init(tfull_bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (warp >= 2)
        for (int c = threadIdx.x - 64; c < V_pad; c += 256) bias_sm[c] = (bias && c < V) ? __ldg(bias + c) : 0.f;
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_launch_dependents();
    pdl_wait();                  // the live row count of the beam search is written inside the iteration: read it behind the wait
    const int M = rows.live();
    const bool live = m0 < M;

    if (warp == 0) {
        if (lane == 0 && live) {  // ===== TMA producer: everything at once, one barrier per K-block =====
            for (int kb = 0; kb < KB; ++kb) {
                mbar_expect_tx(full_bar(kb), A_BYTES + w_kb_bytes);
                tma_load_2d(base + kb * A_BYTES, &tmA, kb * BK, m0, full_bar(kb));
                const uint32_t wdst = w_base + kb * w_kb_bytes;
                int r0 = 0;
                for (; r0 + 128 <= V_pad; r0 += 128) tma_load_2d(wdst + r0 * 128, &tmW, kb * BK, r0, full_bar(kb));
                if (r0 < V_pad) tma_load_2d(wdst + r0 * 128, &tmWtail, kb * BK, r0, full_bar(kb));
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && live) {  // ===== MMA issuer =====
            const uint32_t idesc_main = umma_idesc_bf16(BM, n_main);
            const uint32_t idesc_tail = umma_idesc_bf16(BM, n_tail > 0 ? n_tail : 16);
            for (int kb = 0; kb < KB; ++kb) {
                mbar_wait(full_bar(kb), 0);
                tcgen05_fence_after();
                const uint32_t a_src = base + kb * A_BYTES, b_src = w_base + kb * w_kb_bytes;
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    const uint64_t adesc = umma_desc_sw128(a_src + k * UMMA_K * 2);
                    umma_bf16(tmem_base, adesc, umma_desc_sw128(b_src + k * UMMA_K * 2), idesc_main, (kb | k) != 0 ? 1u : 0u);
                    if (n_tail > 0)
                        umma_bf16(tmem_base + 256u, adesc, umma_desc_sw128(b_src + 256 * 128 + k * UMMA_K * 2), idesc_tail, (kb | k) != 0 ? 1u : 0u);
                }
            }
            umma_commit(tfull_bar);
        }
    } else if (live) {  // ===== statistics: thread = (row, column half) =====
        const int q = warp & 3, hh = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        const int grow = m0 + row;
        const int n32 = V_pad / 32, c_half = (n32 + 1) / 2;
        const int c_begin = hh == 0 ? 0 : c_half, c_end = hh == 0 ? c_half : n32;
        const int tok = grow < M ? row_tok[grow] : -1;
        float tv[KT];
        int ti[KT];
#pragma unroll
        for (int i = 0; i < KT; ++i) { tv[i] = -INFINITY; ti[i] = -1; }
        float mx = -INFINITY, tokval = 0.f, found = 0.f;
        mbar_wait(tfull_bar, 0);
        tcgen05_fence_after();
        const uint32_t tm_row = tmem_base + ((uint32_t)(q * 32) << 16);
        for (int ch = c_begin; ch < c_end; ++ch) {
            uint32_t r[32];
            tmem_ld_32x32(tm_row + (uint32_t)(ch * 32), r);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int col = ch * 32 + j;
                const float v = __uint_as_float(r[j]) + bias_sm[col];
                if (col < V) {
                    mx = fmaxf(mx, v);
                    if (col == tok) { tokval = v; found = 1.f; }
                    topk_list_insert<KT>(tv, ti, v, col);   // sift down from the top (equal values stay behind earlier ones)
                }
            }
        }
#pragma unroll
        for (int i = 0; i < KT; ++i) { xv[(hh * KT + i) * BM + row] = tv[i]; xi[(hh * KT + i) * BM + row] = ti[i]; }
        xinfo[hh * BM + row] = make_float4(mx, tokval, found, 0.f);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const float4 i0 = xinfo[row], i1 = xinfo[BM + row];
        const float gmax = fmaxf(i0.x, i1.x);
        float part = 0.f;
        for (int ch = c_begin; ch < c_end; ++ch) {
            uint32_t r[32];
            tmem_ld_32x32(tm_row + (uint32_t)(ch * 32), r);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int col = ch * 32 + j;
                if (col < V) part += expf(__uint_as_float(r[j]) + bias_sm[col] - gmax);
            }
        }
        if (hh == 1) xinfo[BM + row].w = part;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (hh == 0 && grow < M) {
            const float sum = part + xinfo[BM + row].w;
            // merge of the two sorted lists (equal values: the lower column half first = lower token id)
            int a = 0, b = 0;
            float mv[KT];
            int mi[KT];
#pragma unroll
            for (int j = 0; j < KT; ++j) {
                const float va = a < KT ? xv[a * BM + row] : -INFINITY;
                const float vb = b < KT ? xv[(KT + b) * BM + row] : -INFINITY;
                const int ia = a < KT ? xi[a * BM + row] : -1;
                const int ib = b < KT ? xi[(KT + b) * BM + row] : -1;
                const bool take_a = ia >= 0 && (ib < 0 || va >= vb);
                mv[j] = take_a ? va : vb;
                mi[j] = take_a ? ia : ib;
                a += take_a ? 1 : 0;
                b += take_a ? 0 : 1;
            }
            int keep = 1;
            float cum = 0.f;
            bool open = true;
#pragma unroll
            for (int j = 0; j < KT; ++j) {
                if (j < K) {
                    topv[(long long)grow * K + j] = mv[j];
                    topi[(long long)grow * K + j] = mi[j];
                    // truncated support: entry j is kept while the exclusive cumulative probability of entries 0..j-1 is < 0.9975
                    if (j >= 1 && open) {
                        if (mi[j] < 0) {
                            open = false;
                        } else {
                            cum += expf(mv[j - 1] - gmax) / sum;
                            if (cum < 0.9975f) keep = j + 1; else open = false;
                        }
                    }
                }
            }
            lmax[grow] = gmax;
            lsum[grow] = sum;
            nkeep[grow] = keep;
            tokv[grow] = i0.z != 0.f ? i0.y : i1.y;
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}
}  // namespace tc

template <typename OutT>
int launch_gemm_bf16_tc(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias,
                        OutT* C, int ldc, RowCount rows, int N, int K, bool relu, cudaStream_t s) {
    using namespace tc;
    if (rows.max_rows <= 0 || N <= 0) return 0;
    if (K % BK != 0 || lda % 8 != 0 || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(W) & 15)) {
        set_last_error("tcgen05 GEMM needs K % 64 == 0, lda % 8 == 0 and 16-byte aligned operands");
        return 4;
    }
    CUtensorMap tmA, tmB;
    if (int rc = get_tensor_map(A, rows.max_rows, K, lda, BM, &tmA)) return rc;
    if constexpr (std::is_same<OutT, __nv_bfloat16>::value) {
        // wide K = 256 projections (QKV, cross K/V): CTA-pair kernel, every operand resident, A loaded once per row
        static const bool pair_off = [] { const char* v = getenv("TTB_GEMM_PAIR"); return v && v[0] == '0'; }();
        const int chunks = N % 384 == 0 ? 3 : (N % 256 == 0 && N >= 512 ? 2 : 0);
        if (!pair_off && K == 256 && chunks && ldc % 8 == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0 && rows.max_rows >= 1024) {
            if (int rc = ensure_dyn_smem(gemm_pair_k256_kernel, pgk::SMEM)) return rc;
            CUtensorMap tmWh, tmC;
            if (int rc = get_tensor_map(W, N, K, K, 64, &tmWh)) return rc;
            if (int rc = get_tensor_map(C, rows.max_rows, N, ldc, BM, &tmC)) return rc;
            const int blocks = (rows.max_rows + 2 * BM - 1) / (2 * BM), ppb = N / (chunks * 128);
            launch_pdl(gemm_pair_k256_kernel, dim3(2 * blocks * ppb), dim3(pgk::THREADS), (size_t)pgk::SMEM, s, tmA, tmWh, tmC, bias, rows, chunks, ppb,
                       relu ? 1 : 0);
            return 0;
        }
    }
    if (int rc = get_tensor_map(W, N, K, K, BN, &tmB)) return rc;
    static const bool use_v1 = [] { const char* v = getenv("TTB_GEMM_V1"); return v && v[0] == '1'; }();
    if (!use_v1) {
        // narrow GEMMs (N <= 256 at full batch) get 64-column tiles so that every SM owns more than one
        // tile and the epilogue/main-loop overlap of the persistent kernel has something to overlap
        const int tiles128 = ((N + 127) / 128) * ((rows.max_rows + BM - 1) / BM);
        const bool narrow = tiles128 < 2 * kNumSMs && K <= 512;   // long-K GEMMs (FFN2) would double their A re-reads
        const int bn = narrow ? 64 : 128;
        if (int rc = get_tensor_map(W, N, K, K, bn, &tmB)) return rc;
        const int max_tiles = ((N + bn - 1) / bn) * ((rows.max_rows + BM - 1) / BM);
        const int grid = max_tiles < kNumSMs ? max_tiles : kNumSMs;
        auto launch = [&](auto kernel, int smem) -> int {
            if (int rc = ensure_dyn_smem(kernel, smem)) return rc;
            launch_pdl(kernel, dim3(grid), dim3(pers::THREADS), (size_t)smem, s, tmA, tmB, bias, C, ldc, rows, N, K, relu ? 1 : 0);
            return 0;
        };
        if (narrow) return launch(gemm_bf16_tc_persistent_kernel<OutT, 64>, pers::smem_bytes<OutT, 64>());
        return launch(gemm_bf16_tc_persistent_kernel<OutT, 128>, pers::smem_bytes<OutT, 128>());
    }
    if (int rc = ensure_dyn_smem(gemm_bf16_tc_kernel<OutT>, SMEM_BYTES)) return rc;
    dim3 grid((N + BN - 1) / BN, (rows.max_rows + BM - 1) / BM);
    gemm_bf16_tc_kernel<OutT><<<grid, THREADS, SMEM_BYTES, s>>>(tmA, tmB, bias, C, ldc, rows, N, K, relu ? 1 : 0);
    return 0;
}
// returns 0 on success, -1 when the shape does not fit the fused kernel (caller falls back to GEMM + argmax)
int launch_classifier_argmax(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias, int* pred, RowCount rows,
                             int V, int K, cudaStream_t s) {
    using namespace tc;
    if (rows.max_rows <= 0) return 0;
    const int V_pad = (V + 31) / 32 * 32, KB = K / BK;
    const int smem = KB * A_BYTES + KB * V_pad * 128 + V_pad * 4 + BM * 8 + 8 * 18 + 64 + 1024;
    if (K % BK != 0 || KB > 16 || V_pad > 512 || smem > 227 * 1024 || lda % 8 != 0 || (reinterpret_cast<uintptr_t>(A) & 15) ||
        (reinterpret_cast<uintptr_t>(W) & 15))
        return -1;
    CUtensorMap tmA, tmW, tmWtail;
    if (int rc = get_tensor_map(A, rows.max_rows, K, lda, BM, &tmA)) return rc;
    const int tail_rows = V_pad % 128 ? V_pad % 128 : 128;
    if (int rc = get_tensor_map(W, V, K, K, V_pad >= 128 ? 128 : tail_rows, &tmW)) return rc;
    if (int rc = get_tensor_map(W, V, K, K, tail_rows, &tmWtail)) return rc;
    if (int rc = ensure_dyn_smem(classifier_argmax_kernel<cls::CLS_ARGMAX>, smem)) return rc;
    const int tiles = (rows.max_rows + BM - 1) / BM;
    launch_pdl(classifier_argmax_kernel<cls::CLS_ARGMAX>, dim3(tiles), dim3(cls::THREADS), (size_t)smem, s, tmA, tmW, tmWtail, bias, pred, rows, V,
               V_pad, KB, SampleArgs{});
    return 0;
}

// returns 0 on success, -1 where launch_classifier_argmax would and for top_k > 8 (caller: logits GEMM + launch_sample_rows)
int launch_classifier_sample(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias, RowCount rows, int V, int K,
                             const SampleArgs& a, cudaStream_t s) {
    using namespace tc;
    if (rows.max_rows <= 0) return 0;
    const int V_pad = (V + 31) / 32 * 32, KB = K / BK;
    const int smem = KB * A_BYTES + KB * V_pad * 128 + V_pad * 4 + BM * 8 + 8 * 18 + 64 + 1024;
    const bool list = a.top_k > 0 && a.top_k < V;   // top_k = V draws from the whole vocabulary like top_k = 0
    if (K % BK != 0 || KB > 16 || V_pad > 512 || smem > 227 * 1024 || lda % 8 != 0 || (reinterpret_cast<uintptr_t>(A) & 15) ||
        (reinterpret_cast<uintptr_t>(W) & 15) || (list && (a.top_k > cls::SAMPLE_KT || 2 * 2 * cls::SAMPLE_KT * BM * 4 > KB * A_BYTES)))
        return -1;
    CUtensorMap tmA, tmW, tmWtail;
    if (int rc = get_tensor_map(A, rows.max_rows, K, lda, BM, &tmA)) return rc;
    const int tail_rows = V_pad % 128 ? V_pad % 128 : 128;
    if (int rc = get_tensor_map(W, V, K, K, V_pad >= 128 ? 128 : tail_rows, &tmW)) return rc;
    if (int rc = get_tensor_map(W, V, K, K, tail_rows, &tmWtail)) return rc;
    const int tiles = (rows.max_rows + BM - 1) / BM;
    auto launch = [&](auto kernel) -> int {
        if (int rc = ensure_dyn_smem(kernel, smem)) return rc;
        launch_pdl(kernel, dim3(tiles), dim3(cls::THREADS), (size_t)smem, s, tmA, tmW, tmWtail, bias, a.pred, rows, V, V_pad, KB, a);
        return 0;
    };
    return list ? launch(classifier_argmax_kernel<cls::CLS_SAMPLE_TOPK>) : launch(classifier_argmax_kernel<cls::CLS_SAMPLE>);
}


// returns 0 on success, -1 when the shape does not fit the fused kernel (caller falls back to the logits GEMM + beam_stats)
int launch_classifier_stats(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias, RowCount rows, int V, int Kdim, int n_best,
                            const int* row_tok, float* tokv, float* lmax, float* lsum, int* nkeep, float* topv, int* topi, cudaStream_t s) {
    using namespace tc;
    if (rows.max_rows <= 0) return 0;
    const int V_pad = (V + 31) / 32 * 32, KB = Kdim / BK;
    const int smem = KB * A_BYTES + KB * V_pad * 128 + V_pad * 4 + BM * 8 + 8 * 18 + 64 + 1024;
    // one-entry list for n_best = 1 (teacher-forced scoring reads only the maximum, the sum and the token logit): the same
    // outputs as the 8-entry list, without its sift in the column loop.  Which shapes fit is decided with the 8-entry
    // exchange area either way, so that n_best does not move a shape between the fused and the unfused kernels.
    const int KT = n_best == 1 ? 1 : (n_best <= 8 ? 8 : 16), KT_fit = KT < 8 ? 8 : KT;
    // n_best > 8 stays on the unfused kernels unless forced (TTB_FUSED_STATS_WIDE=1): a warp runs the sift of the sorted list
    // whenever ANY of its 32 rows inserts, which at 16 entries is nearly every element -- measured on B200 (retrosynthesis,
    // bs 8, n_best 10): 267 SMILES/s fused against 291 unfused, while n_best 5 is on par (253 / 252) with one launch less
    if (n_best > 8) {
        const char* wide = getenv("TTB_FUSED_STATS_WIDE");
        if (!(wide && wide[0] == '1')) return -1;
    }
    if (Kdim % BK != 0 || KB > 16 || V_pad > 512 || smem > 227 * 1024 || lda % 8 != 0 || (reinterpret_cast<uintptr_t>(A) & 15) ||
        (reinterpret_cast<uintptr_t>(W) & 15) || n_best > 16 || n_best > V || 4096 + 4 * KT_fit * BM * 4 > KB * A_BYTES)
        return -1;
    CUtensorMap tmA, tmW, tmWtail;
    if (int rc = get_tensor_map(A, rows.max_rows, Kdim, lda, BM, &tmA)) return rc;
    const int tail_rows = V_pad % 128 ? V_pad % 128 : 128;
    if (int rc = get_tensor_map(W, V, Kdim, Kdim, V_pad >= 128 ? 128 : tail_rows, &tmW)) return rc;
    if (int rc = get_tensor_map(W, V, Kdim, Kdim, tail_rows, &tmWtail)) return rc;
    const int tiles = (rows.max_rows + BM - 1) / BM;
    if (KT == 1) {
        if (int rc = ensure_dyn_smem(classifier_stats_kernel<1>, smem)) return rc;
        launch_pdl(classifier_stats_kernel<1>, dim3(tiles), dim3(cls::THREADS), (size_t)smem, s, tmA, tmW, tmWtail, bias, rows, V, V_pad, KB, n_best, row_tok,
                   tokv, lmax, lsum, nkeep, topv, topi);
    } else if (KT == 8) {
        if (int rc = ensure_dyn_smem(classifier_stats_kernel<8>, smem)) return rc;
        launch_pdl(classifier_stats_kernel<8>, dim3(tiles), dim3(cls::THREADS), (size_t)smem, s, tmA, tmW, tmWtail, bias, rows, V, V_pad, KB, n_best, row_tok,
                   tokv, lmax, lsum, nkeep, topv, topi);
    } else {
        if (int rc = ensure_dyn_smem(classifier_stats_kernel<16>, smem)) return rc;
        launch_pdl(classifier_stats_kernel<16>, dim3(tiles), dim3(cls::THREADS), (size_t)smem, s, tmA, tmW, tmWtail, bias, rows, V, V_pad, KB, n_best, row_tok,
                   tokv, lmax, lsum, nkeep, topv, topi);
    }
    return 0;
}

// Number of co-resident clusters of the CTA-pair kernel (0: not usable); TTB_FFN_PAIR=0/1 forces the choice.
static int ffn_pair_clusters() {
    // per device (the opt-in and the occupancy answer are properties of the device); slots are written once each
    static std::atomic<int> per_device[64];
    static std::once_flag init;
    std::call_once(init, [] { for (auto& v : per_device) v.store(-1); });
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
    int max_clusters = per_device[dev].load();
    if (max_clusters < 0) {
        cudaError_t e = ensure_dyn_smem(tc::ffn_pair_kernel, tc::ffn::SMEM) ? cudaErrorInvalidValue : cudaSuccess;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(4 * kNumSMs);
        cfg.blockDim = dim3(tc::ffn::THREADS);
        cfg.dynamicSmemBytes = tc::ffn::SMEM;
        int n = 0;
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&n, tc::ffn_pair_kernel, &cfg);
        max_clusters = e == cudaSuccess ? n : 0;
        (void)cudaGetLastError();
        if (getenv("TTB_DEBUG")) fprintf(stderr, "[ttb] ffn_pair_kernel: %d co-resident clusters of 4 on device %d (%s)\n", max_clusters, dev, cudaGetErrorString(e));
        per_device[dev].store(max_clusters);
    }
    return max_clusters;
}
bool ffn_pair_available(int max_rows) {
    static const int pair_env = [] { const char* v = getenv("TTB_FFN_PAIR"); return v ? atoi(v) : -1; }();
    if (pair_env == 0) return false;
    const int clusters = ffn_pair_clusters();
    if (clusters <= 0) return false;
    // also with more 256-row blocks than co-resident clusters (several waves): measured 1.3 % faster than the
    // cta_group::1 kernel + separate out-projection on the retrosynthesis beam search (80 blocks, 33 clusters)
    (void)max_rows;
    return true;
}

int launch_ffn_fused(__nv_bfloat16* xh, const __nv_bfloat16* W1, const float* bias1, const __nv_bfloat16* W2, const float* bias2,
                     float* x, const float* g1, const float* b1, const float* g2, const float* b2, RowCount rows, int F, cudaStream_t s,
                     const __nv_bfloat16* att, const __nv_bfloat16* Wo, const float* bias_o, const float* g0, const float* b0) {
    using namespace tc;
    const bool chain = att && Wo;
    if (chain && !ffn_pair_available(rows.max_rows)) {
        set_last_error("chained feed-forward launch without the CTA-pair kernel");
        return 4;
    }
    if (rows.max_rows <= 0) return 0;
    if (F % 256 != 0 || F / 2 > ffn::MAX_HALF || (reinterpret_cast<uintptr_t>(W1) & 15) || (reinterpret_cast<uintptr_t>(W2) & 15) ||
        (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(xh) & 15)) {
        set_last_error("fused FFN needs feedforward_dim % 256 == 0, <= 4096 and 16-byte aligned operands");
        return 4;
    }
    CUtensorMap tmXh, tmW1, tmW2, tmX;
    if (int rc = get_tensor_map(xh, rows.max_rows, 256, 256, BM, &tmXh)) return rc;
    if (int rc = get_tensor_map(W1, F, 256, 256, 128, &tmW1)) return rc;
    if (int rc = get_tensor_map(W2, 256, F, F, 128, &tmW2)) return rc;
    if (int rc = get_tensor_map(x, rows.max_rows, 256, 256, BM, &tmX, true)) return rc;
    if (int rc = ensure_dyn_smem(ffn_fused_kernel, ffn::SMEM)) return rc;
    const int tiles = (rows.max_rows + BM - 1) / BM;
#ifdef TTB_FFN_TIMELINE
    {
        static int n_launch = 0;
        if (++n_launch == 400) {   // dump the timeline of launch #399 (steady state)
            cudaStreamSynchronize(s);
            static long long h[3][256][2];
            cudaMemcpyFromSymbol(h, g_ffn_ts, sizeof(h));
            FILE* f = fopen("gpurun_out/ffn_timeline.txt", "w");
            if (f) {
                for (int r = 0; r < 3; ++r)
                    for (int i = 0; i < 256; ++i)
                        if (h[r][i][1]) fprintf(f, "%d %lld %lld\n", r, h[r][i][0], h[r][i][1]);
                fclose(f);
            }
        }
    }
#endif
    // CTA-pair kernel (cta_group::2, clusters of four) whenever all of its clusters are co-resident
    if (ffn_pair_available(rows.max_rows)) {
        const int blocks = (rows.max_rows + 2 * BM - 1) / (2 * BM);
        CUtensorMap tmW1h, tmAtt = tmXh, tmWoh = tmXh;
        if (int rc = get_tensor_map(W1, F, 256, 256, 64, &tmW1h)) return rc;
        if (chain) {
            if ((reinterpret_cast<uintptr_t>(att) & 15) || (reinterpret_cast<uintptr_t>(Wo) & 15)) {
                set_last_error("chained feed-forward launch needs 16-byte aligned operands");
                return 4;
            }
            if (int rc = get_tensor_map(att, rows.max_rows, 256, 256, BM, &tmAtt)) return rc;
            if (int rc = get_tensor_map(Wo, 256, 256, 256, 64, &tmWoh)) return rc;
        }
        launch_pdl(ffn_pair_kernel, dim3(4 * blocks), dim3(ffn::THREADS), (size_t)ffn::SMEM, s, tmXh, tmW1h, tmW2, tmX, bias1, bias2, g1, b1, g2, b2,
                   rows, F, tmAtt, tmWoh, bias_o, g0, b0, chain ? 1 : 0);
        return 0;
    }
    static const int ffn_dbg = [] { const char* v = getenv("TTB_FFN_DBG"); return v ? atoi(v) : 0; }();
    launch_pdl(ffn_fused_kernel, dim3(2 * tiles), dim3(ffn::THREADS), (size_t)ffn::SMEM, s, tmXh, tmW1, tmW2, tmX, bias1, bias2, g1, b1, g2, b2, rows, F, ffn_dbg);
    return 0;
}

int launch_gemm_resid_ln(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, const float* bias, float* x, __nv_bfloat16* xh,
                         const float* g1, const float* b1, const float* g2, const float* b2, RowCount rows, int K, cudaStream_t s,
                         const __nv_bfloat16* W2, const float* bias2, __nv_bfloat16* q2) {
    using namespace tc;
    if (rows.max_rows <= 0) return 0;
    if (K % BK != 0 || lda % 8 != 0 || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(W) & 15) ||
        (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(xh) & 15)) {
        set_last_error("fused GEMM+LayerNorm needs K % 64 == 0, lda % 8 == 0 and 16-byte aligned operands");
        return 4;
    }
    const int chain = (W2 && q2) ? 1 : 0;
    if (chain && (K != 256 || (reinterpret_cast<uintptr_t>(W2) & 15) || (reinterpret_cast<uintptr_t>(q2) & 15))) {
        set_last_error("the chained projection of the fused GEMM+LayerNorm kernel needs K == 256 and 16-byte aligned operands");
        return 4;
    }
    CUtensorMap tmA, tmB, tmX, tmXh, tmW2, tmQ;
    if (int rc = get_tensor_map(A, rows.max_rows, K, lda, BM, &tmA)) return rc;
    if (int rc = get_tensor_map(W, 256, K, K, lnk::BNL, &tmB)) return rc;
    if (int rc = get_tensor_map(x, rows.max_rows, 256, 256, BM, &tmX, true)) return rc;
    if (int rc = get_tensor_map(xh, rows.max_rows, 256, 256, BM, &tmXh)) return rc;
    tmW2 = tmB;
    tmQ = tmXh;
    if (chain) {
        if (int rc = get_tensor_map(W2, 256, 256, 256, lnk::BNL, &tmW2)) return rc;
        if (int rc = get_tensor_map(q2, rows.max_rows, 256, 256, BM, &tmQ)) return rc;
    }
    if (int rc = ensure_dyn_smem(gemm_resid_ln_kernel, lnk::SMEM)) return rc;
    const int tiles = (rows.max_rows + BM - 1) / BM;
#ifdef TTB_LNK_TIMELINE
    {
        static int n_launch = 0;
        if (++n_launch == 400) {
            cudaStreamSynchronize(s);
            long long h[16];
            cudaMemcpyFromSymbol(h, g_lnk_ts, sizeof(h));
            FILE* f = fopen("gpurun_out/lnk_timeline.txt", "w");
            if (f) { for (int i = 0; i < 15; ++i) fprintf(f, "%d %lld\n", i, h[i] ? h[i] - h[2] : -1); fclose(f); }
        }
    }
#endif
    launch_pdl(gemm_resid_ln_kernel, dim3(2 * tiles), dim3(lnk::THREADS), (size_t)lnk::SMEM, s, tmA, tmB, tmX, tmXh, bias, g1, b1, g2, b2, rows, K,
               tmW2, tmQ, bias2, chain);
    return 0;
}

template int launch_gemm_bf16_tc<float>(const __nv_bfloat16*, int, const __nv_bfloat16*, const float*, float*, int, RowCount, int, int, bool, cudaStream_t);
template int launch_gemm_bf16_tc<__nv_bfloat16>(const __nv_bfloat16*, int, const __nv_bfloat16*, const float*, __nv_bfloat16*, int, RowCount, int, int, bool, cudaStream_t);

}  // namespace ttb
