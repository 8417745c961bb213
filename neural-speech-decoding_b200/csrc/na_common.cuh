// Shared helpers for libneuroalpha_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include "../../include/neuroalpha.h"

namespace na {

// ---- error plumbing (thread-local message, integer codes across the ABI) -----------------
char* err_buf();
int fail(int code, const char* fmt, ...);
void count_launch(int n = 1);
// test knob (na_set_tuning "train_max_ctas"): caps the grid of the persistent training kernels so that small batches exercise
// the several-tiles-per-CTA paths (running mbarrier phases across tiles); 0 = one CTA per SM.  Scratch sizes ignore it.
int train_grid_cap(int grid);
int check_launch(const char* what);   // cudaGetLastError -> code + message

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Before a launch of `threads` per block with `smem` bytes of dynamic shared memory: fails with NA_EUNSUPPORTED when the
// kernel as compiled cannot run that many threads (its registers decide), and opts in to shared memory beyond the 48 KB
// default, which covers static and dynamic shared memory together.  A launch that would be refused fails here with a
// message that names the limit instead of as "too many resources requested for launch".
template <typename Kernel>
int prepare_launch(Kernel kern, int threads, size_t smem, const char* what) {
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, kern);
    if (e != cudaSuccess) return fail((int)e, "%s: cudaFuncGetAttributes failed (%s)", what, cudaGetErrorString(e));
    if (threads > a.maxThreadsPerBlock)
        return fail(NA_EUNSUPPORTED, "%s: %d threads per block exceed the kernel's limit of %d (%d registers per thread)", what,
                    threads, a.maxThreadsPerBlock, a.numRegs);
    if (a.sharedSizeBytes + smem > 48 * 1024) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess)
            return fail((int)e, "%s: opt-in to %zu bytes of shared memory failed (%s)", what, smem, cudaGetErrorString(e));
    }
    return NA_OK;
}

#define NA_REQUIRE(cond, code, ...)                          \
    do {                                                     \
        if (!(cond)) return ::na::fail((code), __VA_ARGS__); \
    } while (0)

#define NA_REQUIRE_PTR(p)                                                                \
    do {                                                                                 \
        if ((p) == nullptr) return ::na::fail(NA_EINVAL, "%s: null pointer " #p, __func__); \
        if (!::na::aligned16(p)) return ::na::fail(NA_EALIGN, "%s: " #p " not 16-byte aligned", __func__); \
    } while (0)

#define NA_OPTIONAL_PTR(p)                                                               \
    do {                                                                                 \
        if ((p) != nullptr && !::na::aligned16(p))                                       \
            return ::na::fail(NA_EALIGN, "%s: " #p " not 16-byte aligned", __func__);    \
    } while (0)

inline cudaStream_t as_stream(na_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- activations --------------------------------------------------------------------------
// Exact path: CUDA libm (<= 2 ulp) and IEEE division.  The fp32 contract is 1e-5 relative on
// logits after 1250 dependent cell updates, so no .approx tanh / TF32 here (SURVEY 7.4.2).
__device__ __forceinline__ float sigmoid_acc(float v) { return 1.0f / (1.0f + expf(-v)); }
__device__ __forceinline__ float tanh_acc(float v) { return tanhf(v); }

// Fast-exact path: MUFU.EX2 + MUFU.RCP (each ~1 ulp), absolute error ~1.5e-7 -- the same
// order as the fp32 rounding of the gate pre-activation itself.
__device__ __forceinline__ float ex2_approx(float v) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float rcp_approx(float v) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float sigmoid_fast(float v) {
    return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * v));
}
__device__ __forceinline__ float tanh_fast(float v) {
    // tanh(v) = 2*sigmoid(2v) - 1
    return fmaf(2.0f, rcp_approx(1.0f + ex2_approx(-2.8853900817779268f * v)), -1.0f);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Input range of the 16-bit formats: raw EEG can carry DC offsets of 1e5 uV, beyond fp16's 65,504.  Every fp16 copy of
// the input (K1 with out_dtype NA_F16, the fused producers of the tensor-core kernels) stores x * 2^-4 and the packed
// layer-0 W_ih carries the 2^4 -- both exact powers of two, so nothing changes numerically inside the normal range,
// samples up to 1e6 stay finite, and the layer-0 weight gradient is rescaled by 2^4 where it is reduced.
constexpr float kF16InScale = 0.0625f, kF16InScaleInv = 16.0f;

// nn.RReLU eval slope: torch evaluates (lower+upper)/2 in double, then casts to the tensor dtype
constexpr float kRReluEvalSlope = (float)((1.0 / 8.0 + 1.0 / 3.0) / 2.0);
constexpr float kLnEps = 1e-5f;                                        // nn.LayerNorm default

}  // namespace na
