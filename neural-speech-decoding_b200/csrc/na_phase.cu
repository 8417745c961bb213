// SURVEY 8(f) rank 1: the preprocessing step that sits in front of the decoder on every live window
// (Neuro-Alpha-App/Utilities/preprocessor.py:21-36 -> the vendored third-party phase-coupling filter,
// Utilities/MindsAI/mindsai_filter_python/core.py:14-48), on the GPU.  OPT-IN ONLY: the method is MindsApplied's
// (patent pending, reference implementation under the Polyform Noncommercial licence); this file is written from the
// published mathematics, shares no code with it, and is reached only through
// neural_speech_decoding_b200.preprocess_gpu.PhaseCouplingFilterGPU(accept_noncommercial_terms=True).
//
// Per window x [T][C] (C = 8 channels, fp32 in / out, all arithmetic in float64 like the reference):
//   1. analytic signal per channel: a = x + i H[x], H = Hilbert transform = IFFT(-i sgn(k) FFT(x))  (scipy.signal.hilbert)
//   2. phase unit vectors (cos phi, sin phi) = (x, H[x]) / |a|     (angle(0) = 0 -> (1, 0)); no atan2 / sin needed:
//      sin(phi_i - phi_j) = sin phi_i cos phi_j - cos phi_i sin phi_j
//   3. P[i][j] = sum_t sin^2(phi_i - phi_j) (i != j; the diagonal is 0), then P <- D^-1 P D^-1 with
//      D = sqrt(clip(diag P, 1e-12)) (= 1e-6: the diagonal is zero, so this scales P by 1e12 -- SURVEY 8(f) note)
//   4. M = (I + lambda P^T P)^-1  (8 x 8, Gauss-Jordan with partial pivoting),  y = M x
//
// One CTA per window.  T = 625 = 5^4: a radix-5 Stockham FFT in shared memory (4 stages, complex double).  Two real
// channels ride in one complex transform: H is a real linear operator, so IFFT(-i sgn(k) FFT(x_a + i x_b)) = H[x_a] + i H[x_b]
// -- 4 forward + 4 inverse transforms per window instead of 16, and no spectrum unpacking.  The pair's rounding leaks
// into each other's transform at eps times the larger channel, so every channel is first scaled by a power of two to
// [1, 2) (exact, and the phases do not depend on it), and an all-zero channel keeps H = 0 (phase 0, as in the
// reference) instead of taking the leak as its signal.  The twiddle table
// exp(-2 pi i k / 625) is computed on the host in float64 and passed in.  ~0.6 MFLOP (fp64) and 40 KB of DRAM traffic
// per window; the bound is the fp64 pipe / shared-memory latency, not HBM.
#include "na_common.cuh"

namespace na {

constexpr int kPhT = 625, kPhC = 8, kPhThreads = 256;

struct PhaseSmem {
    double2 buf[2][4][kPhT];          // ping-pong: 4 packed channel pairs
    double2 tw[kPhT];
    float x[kPhT * kPhC];
    double red[8][28];
    float cmax[8][8];                 // per warp, per channel: max |x|
    double cscale[kPhC];              // s = 2^-floor(log2 max|x|); 0 for an all-zero channel
    double2 hscale[4];                // per channel pair: (1 / (N s_{2p}), -1 / (N s_{2p+1})), 0 for an all-zero channel
    double P[8][8];
    double A[8][16];                  // [A | I] for the Gauss-Jordan inverse
};

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }

// in-place forward DFT of 5 points (w = exp(-2 pi i / 5))
__device__ __forceinline__ void dft5(double2 (&v)[5]) {
    constexpr double c1 = 0.30901699437494742410, c2 = -0.80901699437494742410;    // cos(2 pi / 5), cos(4 pi / 5)
    constexpr double s1 = 0.95105651629515357212, s2 = 0.58778525229247312917;     // sin(2 pi / 5), sin(4 pi / 5)
    const double2 t1 = cadd(v[1], v[4]), t2 = cadd(v[2], v[3]), t3 = csub(v[1], v[4]), t4 = csub(v[2], v[3]);
    const double2 a1 = make_double2(v[0].x + c1 * t1.x + c2 * t2.x, v[0].y + c1 * t1.y + c2 * t2.y);
    const double2 a2 = make_double2(v[0].x + c2 * t1.x + c1 * t2.x, v[0].y + c2 * t1.y + c1 * t2.y);
    const double2 b1 = make_double2(s1 * t3.x + s2 * t4.x, s1 * t3.y + s2 * t4.y);
    const double2 b2 = make_double2(s2 * t3.x - s1 * t4.x, s2 * t3.y - s1 * t4.y);
    v[0] = make_double2(v[0].x + t1.x + t2.x, v[0].y + t1.y + t2.y);
    v[1] = make_double2(a1.x + b1.y, a1.y - b1.x);          // a1 - i b1
    v[4] = make_double2(a1.x - b1.y, a1.y + b1.x);          // a1 + i b1
    v[2] = make_double2(a2.x + b2.y, a2.y - b2.x);
    v[3] = make_double2(a2.x - b2.y, a2.y + b2.x);
}

// Forward FFT of the 4 series in S.buf[0] (Stockham autosort, radix 5, 4 stages): the result is back in S.buf[0],
// with kScale: multiplied by S.hscale[p] component-wise.
template <bool kScale>
__device__ __forceinline__ void fft625x4(PhaseSmem& S, int tid) {
    int src = 0;
    for (int Ns = 1; Ns < kPhT; Ns *= 5) {
        const int tstep = kPhT / (Ns * 5);
        for (int w = tid; w < 4 * 125; w += kPhThreads) {
            const int p = w / 125, j = w % 125;
            const double2* in = S.buf[src][p];
            double2* out = S.buf[src ^ 1][p];
            const int k = j % Ns;
            double2 v[5];
            v[0] = in[j];
#pragma unroll
            for (int r = 1; r < 5; ++r) v[r] = cmul(in[j + r * 125], S.tw[k * r * tstep]);
            dft5(v);
            const int j0 = (j / Ns) * Ns * 5 + k;
            if (kScale && Ns * 5 == kPhT) {
                const double2 sc = S.hscale[p];
#pragma unroll
                for (int r = 0; r < 5; ++r) v[r] = make_double2(v[r].x * sc.x, v[r].y * sc.y);
            }
#pragma unroll
            for (int r = 0; r < 5; ++r) out[j0 + r * Ns] = v[r];
        }
        __syncthreads();
        src ^= 1;
    }
}

__global__ void __launch_bounds__(kPhThreads)
phase_coupling_filter_kernel(const float* __restrict__ x, float* __restrict__ y, const double* __restrict__ twiddle,
                             double lambd, int64_t B, int* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PhaseSmem& S = *reinterpret_cast<PhaseSmem*>(smem_raw);
    const int tid = threadIdx.x;
    const int64_t b = blockIdx.x;
    for (int i = tid; i < kPhT; i += kPhThreads) S.tw[i] = make_double2(twiddle[2 * i], twiddle[2 * i + 1]);
    {   // the window, coalesced 16-byte loads; thread tid only sees channels 4 (tid & 1) .. 4 (tid & 1) + 3
        const float4* src = reinterpret_cast<const float4*>(x + b * kPhT * kPhC);
        float4* dst = reinterpret_cast<float4*>(S.x);
        float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f;
        for (int i = tid; i < kPhT * kPhC / 4; i += kPhThreads) {
            const float4 q = src[i];
            dst[i] = q;
            m0 = fmaxf(m0, fabsf(q.x)); m1 = fmaxf(m1, fabsf(q.y)); m2 = fmaxf(m2, fabsf(q.z)); m3 = fmaxf(m3, fabsf(q.w));
        }
#pragma unroll
        for (int o = 2; o < 32; o <<= 1) {
            m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, o)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o));
            m2 = fmaxf(m2, __shfl_xor_sync(0xffffffffu, m2, o)); m3 = fmaxf(m3, __shfl_xor_sync(0xffffffffu, m3, o));
        }
        const int lane = tid & 31;
        if (lane < 2) {
            float* cm = &S.cmax[tid >> 5][4 * lane];
            cm[0] = m0; cm[1] = m1; cm[2] = m2; cm[3] = m3;
        }
    }
    __syncthreads();
    if (tid < kPhC) {       // fmaxf skips NaN; an Inf keeps scale 1 so that it reaches the output like in the reference
        float m = 0.f;
#pragma unroll
        for (int w = 0; w < kPhThreads / 32; ++w) m = fmaxf(m, S.cmax[w][tid]);
        const long long e = isfinite(m) ? ((__double_as_longlong((double)m) >> 52) & 0x7ff) - 1023 : 0;   // floor(log2 m)
        S.cscale[tid] = m == 0.f ? 0.0 : __longlong_as_double((1023 - e) << 52);
        // 1 / s is a power of two, so scaling by (1 / N) / s rounds like the unscaled (1 / N)
        const double h = m == 0.f ? 0.0 : (1.0 / kPhT) * __longlong_as_double((1023 + e) << 52);
        if (tid & 1) S.hscale[tid >> 1].y = -h;
        else S.hscale[tid >> 1].x = h;
    }
    __syncthreads();
    // ---- 1. z_p = x_{2p} + i x_{2p+1} (scaled);  FFT;  W = -i sgn(k) Z;  inverse FFT by conjugation --------------------
    for (int i = tid; i < 4 * kPhT; i += kPhThreads) {
        const int p = i / kPhT, t = i % kPhT;
        S.buf[0][p][t] = make_double2((double)S.x[t * kPhC + 2 * p] * S.cscale[2 * p],
                                      (double)S.x[t * kPhC + 2 * p + 1] * S.cscale[2 * p + 1]);
    }
    __syncthreads();
    fft625x4<false>(S, tid);
    for (int i = tid; i < 4 * kPhT; i += kPhThreads) {
        const int p = i / kPhT, k = i % kPhT;
        const double2 z = S.buf[0][p][k];
        // -i sgn(k) z, then conjugate (inverse transform = conj(FFT(conj(W))) / N):  k in 1..312: -i z = (z.y, -z.x) -> conj (z.y, z.x)
        double2 wv = make_double2(0.0, 0.0);
        if (k >= 1 && k <= (kPhT - 1) / 2) wv = make_double2(z.y, z.x);
        else if (k > (kPhT - 1) / 2) wv = make_double2(-z.y, -z.x);          // +i z = (-z.y, z.x) -> conj (-z.y, -z.x)
        S.buf[0][p][k] = wv;
    }
    __syncthreads();
    // H[s x_{2p}] = Re / N, H[s x_{2p+1}] = -Im / N: the last stage writes buf = (H[x_{2p}], H[x_{2p+1}]), and H = 0 for
    // an all-zero channel instead of the leak of its pair partner
    fft625x4<true>(S, tid);
    // ---- 2./3. phase unit vectors and the pairwise sums: angle(0) = 0 like np.angle, a NaN phase stays NaN ---------------
    double acc[28];
#pragma unroll
    for (int q = 0; q < 28; ++q) acc[q] = 0.0;
    for (int t = tid; t < kPhT; t += kPhThreads) {
        double cs[8], sn[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const double2 hv = S.buf[0][c >> 1][t];
            const double re = (double)S.x[t * kPhC + c];
            const double im = (c & 1) ? hv.y : hv.x;
            const double r = sqrt(re * re + im * im);
            cs[c] = r == 0.0 ? 1.0 : re / r;
            sn[c] = r == 0.0 ? 0.0 : im / r;
        }
        int q = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = i + 1; j < 8; ++j, ++q) {
                const double d = sn[i] * cs[j] - cs[i] * sn[j];
                acc[q] = fma(d, d, acc[q]);
            }
    }
#pragma unroll
    for (int q = 0; q < 28; ++q) {
        double v = acc[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((tid & 31) == 0) S.red[tid >> 5][q] = v;
    }
    __syncthreads();
    if (tid < 64) {
        const int i = tid >> 3, j = tid & 7;
        double v = 0.0;
        if (i != j) {
            const int a = i < j ? i : j, bb = i < j ? j : i;
            const int q = a * 8 - a * (a + 1) / 2 + (bb - a - 1);             // index of pair (a, bb), a < bb
#pragma unroll
            for (int w = 0; w < kPhThreads / 32; ++w) v += S.red[w][q];       // fixed order
        }
        const double dinv = 1.0 / sqrt(1e-12);                               // D^-1: the diagonal of P is zero -> clip(0, 1e-12)
        S.P[i][j] = (dinv * v) * dinv;
    }
    __syncthreads();
    // ---- 4. A = I + lambda P^T P;  M = A^-1 (Gauss-Jordan, partial pivoting; one warp) ---------------------------------
    if (tid < 64) {
        const int i = tid >> 3, j = tid & 7;
        double v = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) v = fma(S.P[k][i], S.P[k][j], v);
        S.A[i][j] = (i == j ? 1.0 : 0.0) + lambd * v;
        S.A[i][8 + j] = i == j ? 1.0 : 0.0;
    }
    __syncthreads();
    if (tid < 32) {
        bool singular = false;
        for (int col = 0; col < 8; ++col) {
            int piv = col;
            double best = fabs(S.A[col][col]);
            for (int r = col + 1; r < 8; ++r) {
                const double a = fabs(S.A[r][col]);
                if (a > best) { best = a; piv = r; }
            }
            if (best == 0.0) singular = true;           // an exactly zero pivot, as LAPACK's getrf reports; NaN is not singular
            __syncwarp();
            if (piv != col && tid < 16) { const double tmp = S.A[col][tid]; S.A[col][tid] = S.A[piv][tid]; S.A[piv][tid] = tmp; }
            __syncwarp();
            const double pinv = 1.0 / S.A[col][col];
            __syncwarp();
            if (tid < 16) S.A[col][tid] *= pinv;
            __syncwarp();
            for (int r = 0; r < 8; ++r) {
                if (r == col) continue;
                const double f = S.A[r][col];
                __syncwarp();
                if (tid < 16) S.A[r][tid] = fma(-f, S.A[col][tid], S.A[r][tid]);
                __syncwarp();
            }
        }
        if (tid == 0 && singular) atomicExch(status, 1);
    }
    __syncthreads();
    // ---- y = M x (float64 accumulate, fp32 out), coalesced stores -------------------------------------------------------
    for (int i = tid; i < kPhT * kPhC; i += kPhThreads) {
        const int t = i >> 3, c = i & 7;
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < 8; ++j) v = fma(S.A[c][8 + j], (double)S.x[t * kPhC + j], v);
        y[b * kPhT * kPhC + i] = (float)v;
    }
}

}  // namespace na

extern "C" int na_phase_coupling_filter(const float* x, float* y, const double* twiddle, double lambd, int* status,
                                        int64_t B, int64_t T, int64_t C, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(B >= 1 && B < ((int64_t)1 << 31), NA_EINVAL, "na_phase_coupling_filter: bad batch B=%lld", (long long)B);
    NA_REQUIRE(T == kPhT && C == kPhC, NA_EUNSUPPORTED,
               "na_phase_coupling_filter: implemented for windows of T=625 samples x C=8 channels (got T=%lld C=%lld)", (long long)T, (long long)C);
    NA_REQUIRE_PTR(x); NA_REQUIRE_PTR(y); NA_REQUIRE_PTR(twiddle);
    NA_REQUIRE(status != nullptr, NA_EINVAL, "na_phase_coupling_filter: null status");
    const size_t smem = sizeof(PhaseSmem);
    cudaError_t e = cudaFuncSetAttribute(phase_coupling_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "na_phase_coupling_filter: shared memory opt-in failed (%s)", cudaGetErrorString(e));
    phase_coupling_filter_kernel<<<(unsigned)B, kPhThreads, smem, as_stream(stream)>>>(x, y, twiddle, lambd, B, status);
    count_launch();
    return check_launch("na_phase_coupling_filter");
}
