// Common device/host helpers for libttb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <string>
#include <utility>

namespace ttb {

// ---- error plumbing (C ABI returns int, message kept per thread) -------------------------
void set_last_error(const std::string& msg);

#define TTB_CUDA_OK(expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            ttb::set_last_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + \
                                " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")");    \
            return 1;                                                                       \
        }                                                                                   \
    } while (0)

#define TTB_CHECK(cond, msg)                                                          \
    do {                                                                              \
        if (!(cond)) {                                                                \
            ttb::set_last_error(std::string(msg) + " (" + __FILE__ + ":" +            \
                                std::to_string(__LINE__) + ")");                      \
            return 2;                                                                 \
        }                                                                             \
    } while (0)

// ---- storage-type conversion -----------------------------------------------------------
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

constexpr int kNumSMs = 148;  // B200

// ---- continuous batching (beam.cu, std_beam.cu) --------------------------------------------------------------------
// exclusive prefix sums of (a, b) over the threads of the block (blockDim.x a multiple of 32); totals in ta, tb
__device__ __forceinline__ void block_scan2(int a, int b, int& ea, int& eb, int& ta, int& tb) {
    __shared__ int s_a[32], s_b[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int ia = a, ib = b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, ia, o), y = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += x; ib += y; }
    }
    if (lane == 31) { s_a[warp] = ia; s_b[warp] = ib; }
    __syncthreads();
    if (warp == 0) {
        int va = lane < nw ? s_a[lane] : 0, vb = lane < nw ? s_b[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, va, o), y = __shfl_up_sync(0xffffffffu, vb, o);
            if (lane >= o) { va += x; vb += y; }
        }
        s_a[lane] = va; s_b[lane] = vb;
    }
    __syncthreads();
    ea = (warp ? s_a[warp - 1] : 0) + ia - a;
    eb = (warp ? s_b[warp - 1] : 0) + ib - b;
    ta = s_a[nw - 1];
    tb = s_b[nw - 1];
    __syncthreads();
}

// One warp: the first n free slots (slot_group[i] < 0) of S, in slot order, into slots[0 .. n); returns the number of free
// slots seen (the scan stops once n are found)
__device__ __forceinline__ int take_free_slots(const int* slot_group, int S, int n, int* slots) {
    const int lane = threadIdx.x & 31;
    int taken = 0;
    for (int i0 = 0; i0 < S && taken < n; i0 += 32) {
        const int i = i0 + lane;
        const bool fr = i < S && slot_group[i] < 0;
        const unsigned m = __ballot_sync(0xffffffffu, fr);
        const int pos = taken + __popc(m & ((1u << lane) - 1u));
        if (fr && pos < n) slots[pos] = i;
        taken += __popc(m);
    }
    return taken;
}

// ---- programmatic dependent launch (PDL) --------------------------------------------------------
// Kernels of the decoding iteration are launched with the programmatic-stream-serialization attribute:
// a kernel may be scheduled while its predecessor drains, runs its prologue (barrier init, TMEM
// allocation, descriptor prefetch) and then blocks in pdl_wait() until the predecessor has completed
// and its writes are visible.  Rule: no global-memory access that depends on (or could disturb) an
// earlier kernel before pdl_wait().  Both instructions are no-ops for a plain launch.
#ifdef TTB_PDL_AFTER_WAIT
// A/B build (scripts/build_variant.sh): a kernel releases its dependents only once its own dependency is satisfied, so at
// most ONE successor waits on the SMs instead of the whole downstream chain cascading ahead
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n\tgriddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() {}
#else
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
bool pdl_enabled();   // engine.cu: TTB_NO_PDL=1 switches the attribute off (A/B comparisons)

// Opt-in of `kernel` to `bytes` of dynamic shared memory on the CURRENT device, once per (device, kernel) and for the
// largest size asked so far.  The attribute is per device and engines of several devices / host threads share the
// process, so the bookkeeping is a mutex-protected table keyed by (device, kernel) (engine.cu).  Returns 0 or an error
// code after set_last_error().
int ensure_dyn_smem(const void* kernel, int bytes);
template <typename... KArgs>
inline int ensure_dyn_smem(void (*kernel)(KArgs...), int bytes) { return ensure_dyn_smem(reinterpret_cast<const void*>(kernel), bytes); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}

// Control words of the device-resident decoding loops (int32 each).
enum Ctrl : int {
    CTRL_N_ACTIVE = 0,   // live queries (rows of the compact token matrix = n_active * rows_per_query)
    CTRL_WIDTH = 1,      // width of the reference's token matrix for the coming iteration (Wn)
    CTRL_DONE = 2,       // 1 -> loop finished (all queries done, width limit, or error)
    CTRL_ERROR = 3,      // 0 ok, 1 draft splice out of bounds, 2 finished-row shape mismatch
    CTRL_ITERS = 4,      // decoder calls made
    CTRL_ACCEPTED = 5,   // accepted draft tokens (sum over queries and iterations)
    CTRL_TOKENS = 6,     // tokens produced (accepted + bonus)
    CTRL_PREV_WIDTH = 7, // width before growing (W)
    CTRL_N_SEL = 8,      // rows recorded in GreedyState::sel by the last accept (live queries before retirement)
    CTRL_N_LEFT = 9,     // live queries left when DONE was raised (N_ACTIVE is zeroed then so that every
                         // row-counted kernel of an already-enqueued iteration exits immediately)
    CTRL_LS = 10,        // source length of the batch (read by the cross-attention kernels so that the
                         // captured decoding graph does not depend on it)
    CTRL_ALLEQ_PICK = 11,  // draft index torch-CPU topk(1) returns when all n_drafts accepted lengths are equal
    CTRL_COUNT = 16
};

// Control words of the speculative beam search (read back by the host once per iteration).
enum BeamCtrl : int {
    BC_NLIVE_ROWS = 0,    // (candidate, draft) rows of unfinished candidates = decoder batch of the iteration
    BC_ERROR = 1,         // 0 ok, 3 draft slots not contiguous (PAD inside a hypothesis), 4 fewer leaves than n_best
    BC_ALL_FINISHED = 2,  // every new candidate contains EOS
    BC_EMPTY_COLS = 3,    // min over new candidates of the number of PAD columns
    BC_ACCEPTED = 4,      // accepted draft tokens of the surviving hypotheses (reference accepted_tokens_num)
    BC_PRODUCED = 5,      // reference produced_non_pad_tokens
    BC_NLIVE_CANDS = 6,   // unfinished candidates (groups of the KV-cached decoder pass)
    BC_LMAX = 7,          // smart drafts: drafts of the candidate that has the most (length the tie-break emulation pads to)
    BC_COUNT = 8
};

}  // namespace ttb
