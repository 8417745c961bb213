// K1: windowing + per-window per-channel z-score (Frontend/app.py:166-170 semantics),
// HBM-bound: one read of the window, one write.  One CTA per window.
#include "na_common.cuh"
#include <cuda_fp16.h>

namespace na {

constexpr int kWinThreads = 256;

__device__ __forceinline__ void store_vec4(void* y, int64_t vec_idx, float4 v, int out_dtype) {
    if (out_dtype == NA_F32) {
        reinterpret_cast<float4*>(y)[vec_idx] = v;
    } else if (out_dtype == NA_F16) {
        __half2 lo = __floats2half2_rn(kF16InScale * v.x, kF16InScale * v.y);
        __half2 hi = __floats2half2_rn(kF16InScale * v.z, kF16InScale * v.w);
        uint2 p;
        p.x = *reinterpret_cast<uint32_t*>(&lo);
        p.y = *reinterpret_cast<uint32_t*>(&hi);
        reinterpret_cast<uint2*>(y)[vec_idx] = p;
    } else {
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y);
        __nv_bfloat162 hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 p;
        p.x = *reinterpret_cast<uint32_t*>(&lo);
        p.y = *reinterpret_cast<uint32_t*>(&hi);
        reinterpret_cast<uint2*>(y)[vec_idx] = p;
    }
}

__device__ __forceinline__ float4 f4add(float4 a, float4 b) {
    return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

// Sum over all threads whose (tid % CQ) is equal; result broadcast to every thread.
// CQ is a power of two <= 32.  `scratch` holds (kWinThreads/32)*CQ float4.
template <int CQ>
__device__ __forceinline__ float4 class_sum(float4 v, float4* scratch) {
#pragma unroll
    for (int o = 16; o >= CQ; o >>= 1) {
        v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
        v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
        v.z += __shfl_xor_sync(0xffffffffu, v.z, o);
        v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane < CQ) scratch[warp * CQ + lane] = v;
    __syncthreads();
    float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
    const int cq = threadIdx.x % CQ;
#pragma unroll
    for (int w = 0; w < kWinThreads / 32; ++w) tot = f4add(tot, scratch[w * CQ + cq]);
    return tot;
}

// Vectorised path: C = 4*CQ channels, the whole window lives in registers (VPT float4 per
// thread), so HBM sees exactly one read and one write of the window.
template <int CQ, int VPT>
__global__ void __launch_bounds__(kWinThreads)
window_zscore_vec_kernel(const float* __restrict__ x, void* __restrict__ y, int64_t B, int64_t T,
                         int64_t hop, int normalize, int out_tmp, int64_t Bp, int out_dtype) {
    __shared__ float4 scratch[2][(kWinThreads / 32) * CQ];
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x;
    const int64_t nvec = T * CQ;
    float4 v[VPT];
    if (b < B) {
        const float4* src = reinterpret_cast<const float4*>(x + b * hop * (4 * CQ));
#pragma unroll
        for (int k = 0; k < VPT; ++k) {
            const int64_t i = tid + (int64_t)k * kWinThreads;
            v[k] = (i < nvec) ? __ldg(src + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (normalize) {
            float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int k = 0; k < VPT; ++k) s = f4add(s, v[k]);
            s = class_sum<CQ>(s, scratch[0]);
            const float fT = (float)T;   // numpy: sum / T (true division), then sqrt(mean(d^2))
            const float4 mu = make_float4(s.x / fT, s.y / fT, s.z / fT, s.w / fT);
            float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int k = 0; k < VPT; ++k) {
                const int64_t i = tid + (int64_t)k * kWinThreads;
                if (i < nvec) {
                    v[k] = make_float4(v[k].x - mu.x, v[k].y - mu.y, v[k].z - mu.z, v[k].w - mu.w);
                    q.x = fmaf(v[k].x, v[k].x, q.x);
                    q.y = fmaf(v[k].y, v[k].y, q.y);
                    q.z = fmaf(v[k].z, v[k].z, q.z);
                    q.w = fmaf(v[k].w, v[k].w, q.w);
                }
            }
            q = class_sum<CQ>(q, scratch[1]);
            // sigma = sqrt(mean((x-mu)^2)) + 1e-6  (epsilon outside the sqrt, app.py:169)
            const float4 sg = make_float4(sqrtf(q.x / fT) + 1e-6f, sqrtf(q.y / fT) + 1e-6f,
                                          sqrtf(q.z / fT) + 1e-6f, sqrtf(q.w / fT) + 1e-6f);
#pragma unroll
            for (int k = 0; k < VPT; ++k)
                v[k] = make_float4(v[k].x / sg.x, v[k].y / sg.y, v[k].z / sg.z, v[k].w / sg.w);
        }
    } else {
#pragma unroll
        for (int k = 0; k < VPT; ++k) v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < VPT; ++k) {
        const int64_t i = tid + (int64_t)k * kWinThreads;
        if (i < nvec) {
            const int64_t t = i / CQ, cq = i % CQ;
            const int64_t o = out_tmp ? ((t * Bp + b) * CQ + cq) : (b * nvec + i);
            store_vec4(y, o, v[k], out_dtype);
        }
    }
}

// 16-bit time-major (TMP) output for C = 8: the input format of the tensor-core tier.  One window-row is
// only 16 B there, so a CTA-per-window kernel would scatter 16-B pieces Bp*16 B apart (half-filled
// sectors; measured 0.39 of HBM peak).  Here a CTA takes 8 consecutive windows, transposes them through
// shared memory and writes 128-B contiguous runs [t][b0..b0+7][8 x 16 bit].
constexpr int kPackWin = 8;
template <int VPT>
__global__ void __launch_bounds__(kWinThreads)
window_pack16_tmp_kernel(const float* __restrict__ x, void* __restrict__ y, int64_t B, int64_t T, int64_t hop,
                         int normalize, int64_t Bp, int out_dtype) {
    extern __shared__ uint2 tile[];                      // [T][kPackWin] : 4 x 16-bit per entry half ... see below
    // tile layout: uint4 per (t, w) = 8 channels x 16 bit; stored as two uint2 halves (cq = 0, 1)
    __shared__ float4 scratch[2][(kWinThreads / 32) * 2];
    const int tid = threadIdx.x;
    const int64_t b0 = (int64_t)blockIdx.x * kPackWin;
    const int64_t nvec = T * 2;
    for (int w = 0; w < kPackWin; ++w) {
        const int64_t b = b0 + w;
        float4 v[VPT];
        if (b < B) {                                      // block-uniform
            const float4* src = reinterpret_cast<const float4*>(x + b * hop * 8);
#pragma unroll
            for (int k = 0; k < VPT; ++k) {
                const int64_t i = tid + (int64_t)k * kWinThreads;
                v[k] = (i < nvec) ? __ldg(src + i) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (normalize) {
                float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int k = 0; k < VPT; ++k) s = f4add(s, v[k]);
                __syncthreads();                          // scratch re-use across windows
                s = class_sum<2>(s, scratch[0]);
                const float fT = (float)T;
                const float4 mu = make_float4(s.x / fT, s.y / fT, s.z / fT, s.w / fT);
                float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int k = 0; k < VPT; ++k) {
                    const int64_t i = tid + (int64_t)k * kWinThreads;
                    if (i < nvec) {
                        v[k] = make_float4(v[k].x - mu.x, v[k].y - mu.y, v[k].z - mu.z, v[k].w - mu.w);
                        q.x = fmaf(v[k].x, v[k].x, q.x); q.y = fmaf(v[k].y, v[k].y, q.y);
                        q.z = fmaf(v[k].z, v[k].z, q.z); q.w = fmaf(v[k].w, v[k].w, q.w);
                    }
                }
                q = class_sum<2>(q, scratch[1]);
                const float4 sg = make_float4(sqrtf(q.x / fT) + 1e-6f, sqrtf(q.y / fT) + 1e-6f,
                                              sqrtf(q.z / fT) + 1e-6f, sqrtf(q.w / fT) + 1e-6f);
#pragma unroll
                for (int k = 0; k < VPT; ++k)
                    v[k] = make_float4(v[k].x / sg.x, v[k].y / sg.y, v[k].z / sg.z, v[k].w / sg.w);
            }
        } else {
#pragma unroll
            for (int k = 0; k < VPT; ++k) v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < VPT; ++k) {
            const int64_t i = tid + (int64_t)k * kWinThreads;      // i = t*2 + cq
            if (i < nvec) {
                uint2 p;
                if (out_dtype == NA_F16) {
                    __half2 lo = __floats2half2_rn(kF16InScale * v[k].x, kF16InScale * v[k].y);
                    __half2 hi = __floats2half2_rn(kF16InScale * v[k].z, kF16InScale * v[k].w);
                    p.x = *reinterpret_cast<uint32_t*>(&lo); p.y = *reinterpret_cast<uint32_t*>(&hi);
                } else {
                    __nv_bfloat162 lo = __floats2bfloat162_rn(v[k].x, v[k].y), hi = __floats2bfloat162_rn(v[k].z, v[k].w);
                    p.x = *reinterpret_cast<uint32_t*>(&lo); p.y = *reinterpret_cast<uint32_t*>(&hi);
                }
                const int64_t t = i >> 1, cq = i & 1;
                tile[(t * kPackWin + w) * 2 + cq] = p;
            }
        }
    }
    __syncthreads();
    // write-out: for each t, 8 windows x 16 B = 128 B contiguous in the TMP layout
    const uint4* tile4 = reinterpret_cast<const uint4*>(tile);
    uint4* out = reinterpret_cast<uint4*>(y);
    for (int64_t idx = tid; idx < T * kPackWin; idx += kWinThreads) {
        const int64_t t = idx / kPackWin, w = idx % kPackWin;
        out[t * Bp + b0 + w] = tile4[idx];
    }
}

// Generic path: any T, any C <= 256.  Three passes over the window (the re-reads hit L1/L2).
__global__ void __launch_bounds__(kWinThreads)
window_zscore_generic_kernel(const float* __restrict__ x, void* __restrict__ y, int64_t B, int64_t T,
                             int64_t C, int64_t hop, int normalize, int out_tmp, int64_t Bp,
                             int out_dtype) {
    __shared__ float red[kWinThreads];
    __shared__ float stat[kWinThreads];
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x;
    const int rows_per_pass = kWinThreads / (int)C;
    const int nactive = rows_per_pass * (int)C;
    const int c = tid % (int)C, r0 = tid / (int)C;
    const bool active = tid < nactive;
    const float* src = x + b * hop * C;
    float mu = 0.f, sg = 1.f;
    if (normalize && b < B) {
        float s = 0.f;
        if (active)
            for (int64_t r = r0; r < T; r += rows_per_pass) s += src[r * C + c];
        red[tid] = active ? s : 0.f;
        __syncthreads();
        if (tid < C) {
            float tot = 0.f;
            for (int k = 0; k < rows_per_pass; ++k) tot += red[tid + k * C];
            stat[tid] = tot / (float)T;
        }
        __syncthreads();
        mu = stat[c];
        float q = 0.f;
        if (active)
            for (int64_t r = r0; r < T; r += rows_per_pass) {
                const float d = src[r * C + c] - mu;
                q = fmaf(d, d, q);
            }
        __syncthreads();
        red[tid] = active ? q : 0.f;
        __syncthreads();
        if (tid < C) {
            float tot = 0.f;
            for (int k = 0; k < rows_per_pass; ++k) tot += red[tid + k * C];
            stat[tid] = sqrtf(tot / (float)T) + 1e-6f;
        }
        __syncthreads();
        sg = stat[c];
    }
    if (!active) return;
    for (int64_t r = r0; r < T; r += rows_per_pass) {
        float v = 0.f;
        if (b < B) {
            v = src[r * C + c];
            if (normalize) v = (v - mu) / sg;
        }
        const int64_t o = out_tmp ? ((r * Bp + b) * C + c) : ((b * T + r) * C + c);
        if (out_dtype == NA_F32) reinterpret_cast<float*>(y)[o] = v;
        else if (out_dtype == NA_F16) reinterpret_cast<__half*>(y)[o] = __float2half_rn(kF16InScale * v);
        else reinterpret_cast<__nv_bfloat16*>(y)[o] = __float2bfloat16_rn(v);
    }
}

// Layout copy (normalize = 0) of windows with more channels than a CTA has threads (the LSTM's input_size reaches 4096):
// thread = channel, strided over the C channels, one time row after another.
__global__ void __launch_bounds__(kWinThreads)
window_copy_wide_kernel(const float* __restrict__ x, void* __restrict__ y, int64_t B, int64_t T, int64_t C, int64_t hop,
                        int out_tmp, int64_t Bp, int out_dtype) {
    const int64_t b = blockIdx.x;
    const float* src = x + b * hop * C;
    for (int64_t r = 0; r < T; ++r)
        for (int64_t c = threadIdx.x; c < C; c += kWinThreads) {
            const float v = (b < B) ? src[r * C + c] : 0.f;
            const int64_t o = out_tmp ? ((r * Bp + b) * C + c) : ((b * T + r) * C + c);
            if (out_dtype == NA_F32) reinterpret_cast<float*>(y)[o] = v;
            else if (out_dtype == NA_F16) reinterpret_cast<__half*>(y)[o] = __float2half_rn(kF16InScale * v);
            else reinterpret_cast<__nv_bfloat16*>(y)[o] = __float2bfloat16_rn(v);
        }
}

}  // namespace na

extern "C" int na_window_zscore(const float* x, void* y, int64_t B, int64_t T, int64_t C, int64_t hop,
                                int normalize, int out_tmp, int64_t Bp, int out_dtype,
                                na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(B >= 0 && T >= 1 && C >= 1 && hop >= 1, NA_EINVAL,
               "na_window_zscore: bad shape B=%lld T=%lld C=%lld hop=%lld", (long long)B, (long long)T,
               (long long)C, (long long)hop);
    NA_REQUIRE(C <= kWinThreads || !normalize, NA_EUNSUPPORTED, "na_window_zscore: C=%lld > %d with normalize", (long long)C,
               kWinThreads);
    NA_REQUIRE(out_dtype == NA_F32 || out_dtype == NA_BF16 || out_dtype == NA_F16, NA_EINVAL, "na_window_zscore: bad out_dtype");
    if (!out_tmp) Bp = B;
    NA_REQUIRE(Bp >= B, NA_EINVAL, "na_window_zscore: Bp < B");
    if (Bp == 0) return NA_OK;
    NA_REQUIRE_PTR(x);
    NA_REQUIRE_PTR(y);
    cudaStream_t st = as_stream(stream);
    const dim3 grid((unsigned)Bp), block(kWinThreads);
    const int64_t nvec = (C % 4 == 0) ? T * (C / 4) : 0;
    const bool hop_ok = ((hop * C) % 4) == 0;   // every window start stays 16-byte aligned
    if (C > kWinThreads) {
        window_copy_wide_kernel<<<grid, block, 0, st>>>(x, y, B, T, C, hop, out_tmp, Bp, out_dtype);
    } else if (C == 8 && hop_ok && out_tmp && out_dtype != NA_F32 && Bp % kPackWin == 0 && nvec <= 5 * kWinThreads &&
        (size_t)T * kPackWin * 16 <= 200 * 1024) {
        const size_t smem = (size_t)T * kPackWin * 16;
        // the attribute is per device: set it on every launch (cheap), like the other wrappers do
        cudaError_t e = cudaFuncSetAttribute(window_pack16_tmp_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return fail((int)e, "na_window_zscore: shared memory opt-in failed (%s)", cudaGetErrorString(e));
        window_pack16_tmp_kernel<5><<<(unsigned)(Bp / kPackWin), block, smem, st>>>(x, y, B, T, hop, normalize, Bp, out_dtype);
    } else if (C == 8 && hop_ok && nvec <= 5 * kWinThreads) {
        window_zscore_vec_kernel<2, 5><<<grid, block, 0, st>>>(x, y, B, T, hop, normalize, out_tmp, Bp, out_dtype);
    } else if (C == 8 && hop_ok && nvec <= 20 * kWinThreads) {
        window_zscore_vec_kernel<2, 20><<<grid, block, 0, st>>>(x, y, B, T, hop, normalize, out_tmp, Bp, out_dtype);
    } else if (C == 4 && hop_ok && nvec <= 8 * kWinThreads) {
        window_zscore_vec_kernel<1, 8><<<grid, block, 0, st>>>(x, y, B, T, hop, normalize, out_tmp, Bp, out_dtype);
    } else if (C == 16 && hop_ok && nvec <= 16 * kWinThreads) {
        window_zscore_vec_kernel<4, 16><<<grid, block, 0, st>>>(x, y, B, T, hop, normalize, out_tmp, Bp, out_dtype);
    } else {
        window_zscore_generic_kernel<<<grid, block, 0, st>>>(x, y, B, T, C, hop, normalize, out_tmp, Bp, out_dtype);
    }
    count_launch();
    return check_launch("na_window_zscore");
}
