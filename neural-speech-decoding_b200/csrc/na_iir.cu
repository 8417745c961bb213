// SURVEY 8(f) rank 4: the collector-side filter chain (Neural_decoding_data_collector.py:109-127) on the GPU.
// Per (window, channel) series: detrend(CONSTANT), then for every filter of the chain a "zero phase" application
// = forward DirectFormII biquad cascade, time reversal, the same cascade again (BrainFlow re-uses the filter object,
// so by default the state of the forward pass is carried into the backward pass), reversal; finally np.round(., d).
// float64 like BrainFlow.
//
// iir_chain_warp_kernel (T <= 2560, the default): ONE WARP per series and the series never leaves the register file.
// Lane l owns the L = ceil(T / 32) consecutive samples [l L, l L + L).  A biquad is a linear recurrence on the state
// s = (w[t-1], w[t-2]), s' = A s + (v, 0), so a section pass over the whole series is
//   (1) every lane runs the recurrence over its own samples from a ZERO state (2 FMA per sample) -> its end state e_l;
//   (2) a warp scan S_l = A^L S_{l-1} + e_l with the constant matrices A^(L 2^j) (5 shuffle rounds; the matrices are
//       computed once per launch by repeated squaring) gives every lane its true incoming state;
//   (3) every lane re-runs the section over its samples from that state -- the same arithmetic, in the same order, as
//       the serial DirectFormII loop -- and overwrites its samples with the outputs.
// The time-reversed pass is the same with the lane order reversed.  7 FMA per sample and section pass instead of 5, but
// the dependent chain is L = 20 samples instead of 625, there is no scratch at all, and DRAM traffic is the algorithmic
// 8 B per sample (one fp32 read, one fp32 write): the bound is the fp64 FMA pipe.  For C = 8 a CTA is one window: it is
// loaded and stored through shared memory with fully coalesced 16-byte accesses.
//
// iir_chain_kernel (longer series): one thread per series, the 2 x nfilt passes go through a per-CTA tiled
// [T][128 series] scratch.
// PARITY UNPINNED (brainflow==5.19.0 is absent from this image): checked against oracle/filter_chain.py, a scipy
// restatement of BrainFlow's published algorithm.
#include "na_common.cuh"

namespace na {

constexpr int kIirMaxF = 8, kIirMaxS = 8;

__global__ void __launch_bounds__(128)
iir_chain_kernel(const float* __restrict__ x, float* __restrict__ y, double* __restrict__ scratch,
                 const double* __restrict__ coef, const int* __restrict__ nsec, int nfilt, int64_t S, int T, int C,
                 int detrend, int round_decimals, int carry_state) {
    __shared__ double s_coef[kIirMaxF * kIirMaxS * 5];
    __shared__ int s_nsec[kIirMaxF];
    int total = 0;
    for (int f = 0; f < nfilt; ++f) total += nsec[f];
    for (int i = threadIdx.x; i < total * 5; i += blockDim.x) s_coef[i] = coef[i];
    if (threadIdx.x < nfilt) s_nsec[threadIdx.x] = nsec[threadIdx.x];
    __syncthreads();
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int64_t b = s / C;
    const int c = (int)(s % C);
    const float* xs = x + (b * T) * C + c;           // element t at xs[t * C]
    float* ys = y + (b * T) * C + c;
    // scratch is tiled per CTA: [S / 128][T][128] -- a CTA walks ONE contiguous T x 1 KB region forwards and backwards
    // (DRAM-page and L2 friendly; the first layout, [T][S], scattered 256-byte accesses over the whole buffer)
    double* sc = scratch + (int64_t)blockIdx.x * T * 128 + threadIdx.x;
    double mean = 0.0;
    if (detrend) {
        for (int t = 0; t < T; ++t) mean += (double)xs[(int64_t)t * C];
        mean /= (double)T;
    }
    double scale = 1.0;
    for (int k = 0; k < round_decimals; ++k) scale *= 10.0;
    if (nfilt == 0) {
        for (int t = 0; t < T; ++t) {
            double v = (double)xs[(int64_t)t * C] - mean;
            if (round_decimals >= 0) v = rint(v * scale) / scale;
            ys[(int64_t)t * C] = (float)(v == 0.0 ? 0.0 : v);
        }
        return;
    }
    int cbase = 0;
    for (int f = 0; f < nfilt; ++f) {
        const int ns = s_nsec[f];
        double b0[kIirMaxS], b1[kIirMaxS], b2[kIirMaxS], a1[kIirMaxS], a2[kIirMaxS], w1[kIirMaxS], w2[kIirMaxS];
#pragma unroll
        for (int k = 0; k < kIirMaxS; ++k) {
            const bool on = k < ns;
            const double* cf = s_coef + (cbase + (on ? k : 0)) * 5;
            b0[k] = on ? cf[0] : 1.0; b1[k] = on ? cf[1] : 0.0; b2[k] = on ? cf[2] : 0.0;
            a1[k] = on ? cf[3] : 0.0; a2[k] = on ? cf[4] : 0.0;
            w1[k] = 0.0; w2[k] = 0.0;
        }
        cbase += ns;
        const bool last = (f == nfilt - 1);
        // forward pass (8 samples fetched ahead of the serial recurrence: the loads are independent of it)
        for (int t0 = 0; t0 < T; t0 += 8) {
            double buf[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int t = t0 + j;
                buf[j] = t < T ? ((f == 0) ? (double)xs[(int64_t)t * C] - mean : sc[(int64_t)t * 128]) : 0.0;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int t = t0 + j;
                if (t >= T) break;
                double v = buf[j];
#pragma unroll
                for (int k = 0; k < kIirMaxS; ++k) {
                    if (k < ns) {                               // DirectFormII: w = v - a1 w1 - a2 w2; out = b0 w + b1 w1 + b2 w2
                        const double w = v - a1[k] * w1[k] - a2[k] * w2[k];
                        v = b0[k] * w + b1[k] * w1[k] + b2[k] * w2[k];
                        w2[k] = w1[k];
                        w1[k] = w;
                    }
                }
                sc[(int64_t)t * 128] = v;
            }
        }
        if (!carry_state) {
#pragma unroll
            for (int k = 0; k < kIirMaxS; ++k) { w1[k] = 0.0; w2[k] = 0.0; }
        }
        // backward pass (the reversed series through the same cascade)
        for (int t0 = T - 1; t0 >= 0; t0 -= 8) {
            double buf[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int t = t0 - j;
                buf[j] = t >= 0 ? sc[(int64_t)t * 128] : 0.0;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int t = t0 - j;
                if (t < 0) break;
                double v = buf[j];
#pragma unroll
                for (int k = 0; k < kIirMaxS; ++k) {
                    if (k < ns) {
                        const double w = v - a1[k] * w1[k] - a2[k] * w2[k];
                        v = b0[k] * w + b1[k] * w1[k] + b2[k] * w2[k];
                        w2[k] = w1[k];
                        w1[k] = w;
                    }
                }
                if (last) {
                    if (round_decimals >= 0) v = rint(v * scale) / scale;      // np.round: multiply, rint, divide
                    ys[(int64_t)t * C] = (float)(v == 0.0 ? 0.0 : v);          // the collector also clears negative zero
                } else {
                    sc[(int64_t)t * 128] = v;
                }
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------------------------
// warp-per-series kernel
// ---------------------------------------------------------------------------------------------------------------
constexpr int kIirWarps = 8;                 // series per CTA (for C == 8: the 8 channels of one window)

struct Mat2 { double a, b, c, d; };          // [[a, b], [c, d]]
__device__ __forceinline__ Mat2 mat_mul(const Mat2& x, const Mat2& y) {
    return Mat2{x.a * y.a + x.b * y.c, x.a * y.b + x.b * y.d, x.c * y.a + x.d * y.c, x.c * y.b + x.d * y.d};
}

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// One section pass over the register-resident series (every lane owns exactly LT samples: the series is padded with
// zeros at the FRONT, see the kernel).  dir = +1: ascending time (lane 0 first), -1: descending (lane 31 first).
// (w1, w2) in: the state the pass starts from (warp-uniform); out: the state after the last sample processed.
template <int LT>
__device__ __forceinline__ void section_pass(double (&v)[LT], const int lane, const int dir,
                                             const double b0, const double b1, const double b2, const double na1, const double na2,
                                             const double* __restrict__ pm,       // 5 x (a, b, c, d): A^(LT 2^j), then A^(LT/2)
                                             double& w1, double& w2) {
    static_assert(LT % 2 == 0, "the lane block is processed as two half blocks");
    constexpr int HB = LT / 2;
    const bool first = dir > 0 ? lane == 0 : lane == 31;          // the block that is processed first carries the initial state
    const double h00 = pm[20], h01 = pm[21], h10 = pm[22], h11 = pm[23];     // A^HB
    // (1) end state of this lane's block from a zero state (the first block: from the true initial state).  The block is
    //     run as TWO independent half-block chains (instruction-level parallelism: the recurrence is latency-bound),
    //     joined by A^HB.  w_t = (v_t - a2 w_{t-2}) - a1 w_{t-1}: only the outer FMA is on a dependent chain.
    double p1 = first ? w1 : 0.0, p2 = first ? w2 : 0.0, q1 = 0.0, q2 = 0.0;
#pragma unroll
    for (int jj = 0; jj < HB; ++jj) {
        const int ja = dir > 0 ? jj : LT - 1 - jj, jb = dir > 0 ? jj + HB : HB - 1 - jj;
        const double wa = fma(na1, p1, fma(na2, p2, v[ja]));
        const double wb = fma(na1, q1, fma(na2, q2, v[jb]));
        p2 = p1; p1 = wa;
        q2 = q1; q1 = wb;
    }
    double e1 = fma(h00, p1, fma(h01, p2, q1)), e2 = fma(h10, p1, fma(h11, p2, q2));
    // (2) scan over the blocks in processing order: S_p = A^LT S_{p-1} + e_p
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const int d = 1 << j;
        const int src = dir > 0 ? lane - d : lane + d;
        const double f1 = shfl_d(e1, src & 31), f2 = shfl_d(e2, src & 31);
        const bool take = dir > 0 ? lane >= d : lane + d <= 31;
        const double g1 = fma(pm[4 * j], f1, pm[4 * j + 1] * f2), g2 = fma(pm[4 * j + 2], f1, pm[4 * j + 3] * f2);
        e1 += take ? g1 : 0.0;
        e2 += take ? g2 : 0.0;
    }
    // incoming state of this lane = end state of the block processed just before it
    const int prev = dir > 0 ? lane - 1 : lane + 1;
    double s1 = shfl_d(e1, prev & 31), s2 = shfl_d(e2, prev & 31);
    if (first) { s1 = w1; s2 = w2; }
    // incoming state of the second half block = A^HB s_in + (zero-state end of the first half); in the first block the
    // first half already ran from the true initial state
    double t1 = first ? p1 : fma(h00, s1, fma(h01, s2, p1)), t2 = first ? p2 : fma(h10, s1, fma(h11, s2, p2));
    // (3) the real pass: DirectFormII, w = v - a1 w1 - a2 w2; out = b0 w + b1 w1 + b2 w2 (two half-block chains again)
#pragma unroll
    for (int jj = 0; jj < HB; ++jj) {
        const int ja = dir > 0 ? jj : LT - 1 - jj, jb = dir > 0 ? jj + HB : HB - 1 - jj;
        const double parta = fma(b1, s1, b2 * s2), partb = fma(b1, t1, b2 * t2);       // off the dependent chains
        const double wa = fma(na1, s1, fma(na2, s2, v[ja]));
        const double wb = fma(na1, t1, fma(na2, t2, v[jb]));
        v[ja] = fma(b0, wa, parta);
        v[jb] = fma(b0, wb, partb);
        s2 = s1; s1 = wa;
        t2 = t1; t1 = wb;
    }
    // state after the last processed sample (end of the second half): ascending -> lane 31, descending -> lane 0
    const int fin = dir > 0 ? 31 : 0;
    w1 = shfl_d(t1, fin);
    w2 = shfl_d(t2, fin);
}

// The series occupies the LAST T of the 32 LT register slots (slot p = pad + t, lane = p / LT): the pad slots in front hold
// zeros.  A zero input on a zero state is an exact no-op, so the ascending pass (which always starts from a zero state) is
// unchanged, the state after the last sample sits at the end of lane 31 where the descending pass picks it up, and what
// the descending pass rings into the pad slots is cleared before the next filter.  Every lane runs identical,
// unpredicated loops.
template <int LT, int MAXS, int OCC>
__global__ void __launch_bounds__(kIirWarps * 32, OCC)
iir_chain_warp_kernel(const float* __restrict__ x, float* __restrict__ y, const double* __restrict__ coef,
                      const int* __restrict__ nsec, int nfilt, int64_t S, int T, int C, int detrend, int round_decimals,
                      int carry_state) {
    __shared__ double s_coef[kIirMaxF * kIirMaxS * 5];
    __shared__ double s_pm[kIirMaxF * kIirMaxS * 24];
    __shared__ int s_nsec[kIirMaxF];
    extern __shared__ __align__(16) float s_io[];                  // C == 8: [8 channels][32 lanes][LT + 1] staging
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int pad = 32 * LT - T;
    int total = 0;
    for (int f = 0; f < nfilt; ++f) total += nsec[f];
    for (int i = tid; i < total * 5; i += blockDim.x) s_coef[i] = coef[i];
    if (tid < nfilt) s_nsec[tid] = nsec[tid];
    if (tid < total) {                                             // A^(LT/2), then A^(LT 2^j), j = 0..4, by repeated squaring
        const double a1 = coef[tid * 5 + 3], a2 = coef[tid * 5 + 4];
        Mat2 base{-a1, -a2, 1.0, 0.0}, acc{1.0, 0.0, 0.0, 1.0};
        for (int e = LT / 2; e > 0; e >>= 1) {
            if (e & 1) acc = mat_mul(acc, base);
            base = mat_mul(base, base);
        }
        double* oh = s_pm + tid * 24 + 20;
        oh[0] = acc.a; oh[1] = acc.b; oh[2] = acc.c; oh[3] = acc.d;
        acc = mat_mul(acc, acc);
        for (int j = 0; j < 5; ++j) {
            double* o = s_pm + tid * 24 + 4 * j;
            o[0] = acc.a; o[1] = acc.b; o[2] = acc.c; o[3] = acc.d;
            acc = mat_mul(acc, acc);
        }
    }
    const int64_t s = (int64_t)blockIdx.x * kIirWarps + warp;
    const bool coop = (C == kIirWarps);                             // CTA = one window: coalesced staging through shared memory
    constexpr int stride = LT + 1;                                 // padding: the 32 lanes of a warp hit distinct banks
    if (coop) {
        const float4* src = reinterpret_cast<const float4*>(x + (int64_t)blockIdx.x * T * 8);
        for (int i = tid; i < T * 2; i += blockDim.x) {
            const float4 q = src[i];
            const int p = pad + (i >> 1), c0 = (i & 1) * 4;
            const int ln = p / LT, j = p - ln * LT;
            s_io[((c0 + 0) * 32 + ln) * stride + j] = q.x;
            s_io[((c0 + 1) * 32 + ln) * stride + j] = q.y;
            s_io[((c0 + 2) * 32 + ln) * stride + j] = q.z;
            s_io[((c0 + 3) * 32 + ln) * stride + j] = q.w;
        }
    }
    __syncthreads();
    const bool active = s < S;
    const int64_t b = active ? s / C : 0;
    const int c = active ? (int)(s % C) : 0;
    const int p0 = lane * LT;                                      // first slot of this lane
    double v[LT];
#pragma unroll
    for (int j = 0; j < LT; ++j) {
        const int t = p0 + j - pad;
        v[j] = 0.0;
        if (active && t >= 0) v[j] = coop ? (double)s_io[(warp * 32 + lane) * stride + j] : (double)x[(b * T + t) * C + c];
    }
    if (detrend) {
        double part = 0.0;
#pragma unroll
        for (int j = 0; j < LT; ++j) part += v[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        const double mean = part / (double)T;
#pragma unroll
        for (int j = 0; j < LT; ++j) if (p0 + j >= pad) v[j] -= mean;
    }
    int cbase = 0;
    for (int f = 0; f < nfilt; ++f) {
        const int ns = s_nsec[f];
        double w1[MAXS], w2[MAXS];
#pragma unroll
        for (int k = 0; k < MAXS; ++k) { w1[k] = 0.0; w2[k] = 0.0; }
        // forward: the cascade section by section over the whole series (same result as sample by sample: section k only
        // consumes the finished output of section k-1)
#pragma unroll
        for (int k = 0; k < MAXS; ++k)
            if (k < ns) {
                const double* cf = s_coef + (cbase + k) * 5;
                section_pass<LT>(v, lane, +1, cf[0], cf[1], cf[2], -cf[3], -cf[4], s_pm + (cbase + k) * 24, w1[k], w2[k]);
            }
        if (!carry_state) {
#pragma unroll
            for (int k = 0; k < MAXS; ++k) { w1[k] = 0.0; w2[k] = 0.0; }
        }
        // the reversed series through the same cascade
#pragma unroll
        for (int k = 0; k < MAXS; ++k)
            if (k < ns) {
                const double* cf = s_coef + (cbase + k) * 5;
                section_pass<LT>(v, lane, -1, cf[0], cf[1], cf[2], -cf[3], -cf[4], s_pm + (cbase + k) * 24, w1[k], w2[k]);
            }
        cbase += ns;
        if (p0 < pad) {                                            // the descending pass rang into the pad slots: clear them
#pragma unroll
            for (int j = 0; j < LT; ++j) if (p0 + j < pad) v[j] = 0.0;
        }
    }
    double scale = 1.0;
    for (int k = 0; k < round_decimals; ++k) scale *= 10.0;
    if (coop) __syncthreads();                                     // every warp has read its inputs from the staging buffer
#pragma unroll
    for (int j = 0; j < LT; ++j) {
        const int t = p0 + j - pad;
        if (active && t >= 0) {
            double o = v[j];
            if (round_decimals >= 0) o = rint(o * scale) / scale;  // np.round: multiply, rint, divide
            const float of = (float)(o == 0.0 ? 0.0 : o);          // the collector also clears negative zero
            if (coop) s_io[(warp * 32 + lane) * stride + j] = of;
            else y[(b * T + t) * C + c] = of;
        }
    }
    if (coop) {
        __syncthreads();
        float4* dst = reinterpret_cast<float4*>(y + (int64_t)blockIdx.x * T * 8);
        for (int i = tid; i < T * 2; i += blockDim.x) {
            const int p = pad + (i >> 1), c0 = (i & 1) * 4;
            const int ln = p / LT, j = p - ln * LT;
            dst[i] = make_float4(s_io[((c0 + 0) * 32 + ln) * stride + j], s_io[((c0 + 1) * 32 + ln) * stride + j],
                                 s_io[((c0 + 2) * 32 + ln) * stride + j], s_io[((c0 + 3) * 32 + ln) * stride + j]);
        }
    }
}

static int g_iir_occ3 = 2;           // LT = 20: CTAs per SM the register allocation aims at (1: 152 registers, 2: <= 128, 3: <= 80 with spills); A/B knob
void set_iir_occ3(int v) { g_iir_occ3 = v; }

// The 48 KB a launch gets without opting in covers static (s_coef, s_pm: 14,880 B) and dynamic shared memory together, so
// the C == 8 staging of LT = 40 (41,984 B) needs the opt-in as well as that of LT = 80 (82,944 B); LT = 20 (21,504 B) fits.
template <typename Kernel>
static int allow_dynamic_smem(Kernel kern, size_t smem) {
    if (smem == 0) return 0;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    return e == cudaSuccess ? 0 : fail((int)e, "na_iir_chain: shared memory opt-in failed (%s)", cudaGetErrorString(e));
}

template <int LT>
static int launch_iir_warp(const float* x, float* y, const double* coef, const int* nsec, int nfilt, int max_sections, int64_t S, int T,
                           int C, int detrend, int round_decimals, int carry_state, cudaStream_t st) {
    const size_t smem = C == kIirWarps ? (size_t)kIirWarps * 32 * (LT + 1) * sizeof(float) : 0;
    const unsigned grid = (unsigned)((S + kIirWarps - 1) / kIirWarps);
    if (max_sections <= 4 && LT <= 20 && g_iir_occ3 >= 3) {
        iir_chain_warp_kernel<LT <= 20 ? LT : 20, 4, 3><<<grid, kIirWarps * 32, smem, st>>>(x, y, coef, nsec, nfilt, S, T, C, detrend,
                                                                                          round_decimals, carry_state);
    } else if (max_sections <= 4 && LT <= 20 && g_iir_occ3 == 2) {
        iir_chain_warp_kernel<LT <= 20 ? LT : 20, 4, 2><<<grid, kIirWarps * 32, smem, st>>>(x, y, coef, nsec, nfilt, S, T, C, detrend,
                                                                                          round_decimals, carry_state);
    } else if (max_sections <= 4) {
        auto kern = iir_chain_warp_kernel<LT, 4, 1>;
        if (const int rc = allow_dynamic_smem(kern, smem)) return rc;
        kern<<<grid, kIirWarps * 32, smem, st>>>(x, y, coef, nsec, nfilt, S, T, C, detrend, round_decimals, carry_state);
    } else {
        auto kern = iir_chain_warp_kernel<LT, kIirMaxS, 1>;
        if (const int rc = allow_dynamic_smem(kern, smem)) return rc;
        kern<<<grid, kIirWarps * 32, smem, st>>>(x, y, coef, nsec, nfilt, S, T, C, detrend, round_decimals, carry_state);
    }
    return 0;
}

}  // namespace na

extern "C" int na_iir_chain(const float* x, float* y, double* scratch, const double* coef, const int* nsec,
                            int64_t nfilt, int64_t B, int64_t T, int64_t C, int detrend, int round_decimals,
                            int carry_state, int64_t max_sections, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(B >= 1 && T >= 1 && T < (1 << 30) && C >= 1 && C < (1 << 20), NA_EINVAL,
               "na_iir_chain: bad shape B=%lld T=%lld C=%lld", (long long)B, (long long)T, (long long)C);
    NA_REQUIRE(nfilt >= 0 && nfilt <= kIirMaxF, NA_EUNSUPPORTED, "na_iir_chain: %lld filters (at most %d)", (long long)nfilt, kIirMaxF);
    NA_REQUIRE(round_decimals <= 22, NA_EINVAL, "na_iir_chain: round_decimals=%d", round_decimals);
    NA_REQUIRE_PTR(x); NA_REQUIRE_PTR(y);
    NA_REQUIRE(nfilt == 0 || (coef != nullptr && nsec != nullptr), NA_EINVAL, "na_iir_chain: null pointer");
    const int64_t S = B * C;
    NA_REQUIRE(max_sections >= 0 && max_sections <= kIirMaxS, NA_EUNSUPPORTED, "na_iir_chain: %lld sections per filter (at most %d)",
               (long long)max_sections, kIirMaxS);
    if (T <= 32 * 80) {               // warp-per-series, register-resident: no scratch
        const int L = (int)((T + 31) / 32), ms = (int)max_sections;
        int rc;
        if (L <= 20) rc = launch_iir_warp<20>(x, y, coef, nsec, (int)nfilt, ms, S, (int)T, (int)C, detrend, round_decimals, carry_state, as_stream(stream));
        else if (L <= 40) rc = launch_iir_warp<40>(x, y, coef, nsec, (int)nfilt, ms, S, (int)T, (int)C, detrend, round_decimals, carry_state, as_stream(stream));
        else rc = launch_iir_warp<80>(x, y, coef, nsec, (int)nfilt, ms, S, (int)T, (int)C, detrend, round_decimals, carry_state, as_stream(stream));
        if (rc) return rc;
        count_launch();
        return check_launch("na_iir_chain");
    }
    NA_REQUIRE(nfilt == 0 || scratch != nullptr, NA_EINVAL, "na_iir_chain: T > 2560 needs the scratch buffer");
    iir_chain_kernel<<<(unsigned)((S + 127) / 128), 128, 0, as_stream(stream)>>>(x, y, scratch, coef, nsec, (int)nfilt, S, (int)T,
                                                                              (int)C, detrend, round_decimals, carry_state);
    count_launch();
    return check_launch("na_iir_chain");
}
