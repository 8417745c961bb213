// Time-parallel gradient reductions: out[M][N] = sum_r G[r][m] * A[r][n] over a very tall
// row range (rows = T*Bp), tiny outputs.  Split over row chunks, partials reduced in a fixed
// order -> bit-reproducible run to run (no float atomics).
#include "na_common.cuh"

namespace na {

constexpr int kTnTile = 64;     // output tile 64 x 64
constexpr int kTnRows = 16;     // rows staged per iteration
constexpr int kTnThreads = 256; // 16 x 16 threads, 4 x 4 outputs each

template <bool TWO>      // TWO: second A operand (compile-time, so the single-operand loads stay branch-free)
__global__ void __launch_bounds__(kTnThreads)
gemm_tn_partial_kernel(const float* __restrict__ G, int64_t ldg, const float* __restrict__ A, int64_t lda,
                       int64_t R, int M, int N, float* __restrict__ partial, int64_t rows_per_chunk,
                       // optional second A operand: columns [N1, N) come from A2 at row r - shift (zero for r < shift);
                       // one pass over G then yields dW_ih AND dW_hh (h_{t-1} = the h rows shifted down by Bp)
                       int N1, const float* __restrict__ A2, int64_t lda2, int64_t shift) {
    __shared__ float Gs[kTnRows][kTnTile + 4];
    __shared__ float As[kTnRows][kTnTile + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * kTnTile, n0 = blockIdx.z * kTnTile;
    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_chunk;
    const int64_t r_end = min(R, r_begin + rows_per_chunk);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jn = 0; jn < 4; ++jn) acc[i][jn] = 0.f;

    // register double buffer: the global loads of the next 16 rows are in flight while the current 16 are multiplied
    // (the first version loaded, synchronised and multiplied in sequence and was latency-bound at 16 TFLOP/s)
    constexpr int kPer = (kTnRows * kTnTile) / kTnThreads;        // elements of each operand per thread and stage
    float gn[kPer], an[kPer];
    auto fetch = [&](int64_t r0) {
#pragma unroll
        for (int e = 0; e < kPer; ++e) {
            const int idx = tid + e * kTnThreads;
            const int rr = idx / kTnTile, cc = idx % kTnTile;
            const int64_t r = r0 + rr;
            gn[e] = (r < r_end && m0 + cc < M) ? __ldg(G + r * ldg + m0 + cc) : 0.f;
            const int n = n0 + cc;
            float av = 0.f;
            if (r < r_end && n < N) {
                if (!TWO || n < N1) av = __ldg(A + r * lda + n);
                else if (r >= shift) av = __ldg(A2 + (r - shift) * lda2 + (n - N1));
            }
            an[e] = av;
        }
    };
    fetch(r_begin);
    for (int64_t r0 = r_begin; r0 < r_end; r0 += kTnRows) {
#pragma unroll
        for (int e = 0; e < kPer; ++e) {
            const int idx = tid + e * kTnThreads;
            Gs[idx / kTnTile][idx % kTnTile] = gn[e];
            As[idx / kTnTile][idx % kTnTile] = an[e];
        }
        __syncthreads();
        if (r0 + kTnRows < r_end) fetch(r0 + kTnRows);
#pragma unroll
        for (int rr = 0; rr < kTnRows; ++rr) {
            const float4 g = *reinterpret_cast<const float4*>(&Gs[rr][ty * 4]);
            const float4 a = *reinterpret_cast<const float4*>(&As[rr][tx * 4]);
            const float gv[4] = {g.x, g.y, g.z, g.w}, av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int jn = 0; jn < 4; ++jn) acc[i][jn] = fmaf(gv[i], av[jn], acc[i][jn]);
        }
        __syncthreads();
    }
    float* out = partial + (size_t)blockIdx.x * M * N;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
#pragma unroll
        for (int jn = 0; jn < 4; ++jn) {
            const int n = n0 + tx * 4 + jn;
            if (m < M && n < N) out[(size_t)m * N + n] = acc[i][jn];
        }
    }
}

__global__ void colsum_partial_kernel(const float* __restrict__ G, int64_t ldg, int64_t R, int M,
                                      float* __restrict__ partial, int64_t rows_per_chunk) {
    const int m = blockIdx.y * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_chunk;
    const int64_t r_end = min(R, r_begin + rows_per_chunk);
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int64_t r = r_begin;
    for (; r + 3 < r_end; r += 4) {
        s0 += G[r * ldg + m];
        s1 += G[(r + 1) * ldg + m];
        s2 += G[(r + 2) * ldg + m];
        s3 += G[(r + 3) * ldg + m];
    }
    for (; r < r_end; ++r) s0 += G[r * ldg + m];
    partial[(size_t)blockIdx.x * M + m] = (s0 + s1) + (s2 + s3);
}

// out[i] = sum_c partial[c][i], c ascending (fixed order); kAdd: out[i] += that sum.
template <bool kAdd = false>
__global__ void reduce_partials_kernel(const float* __restrict__ partial, float* __restrict__ out,
                                       int nchunks, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = 0.f;
    for (int c = 0; c < nchunks; ++c) s += partial[(size_t)c * n + i];
    out[i] = kAdd ? out[i] + s : s;
}

int wgrad_nchunks(int64_t M, int64_t N, int64_t R) {
    const int64_t tiles = ((M + kTnTile - 1) / kTnTile) * ((N + kTnTile - 1) / kTnTile);
    int64_t n = 592 / (tiles > 0 ? tiles : 1);
    if (n < 4) n = 4;
    if (n > 296) n = 296;
    const int64_t max_by_rows = (R + kTnRows - 1) / kTnRows;
    if (n > max_by_rows) n = max_by_rows > 0 ? max_by_rows : 1;
    return (int)n;
}

// out[M][N] = G^T A over R rows (add: out += G^T A).  `partial` must hold wgrad_nchunks(M,N,R)*M*N floats.
static int gemm_tn_impl(const float* G, int64_t ldg, const float* A, int64_t lda, int64_t R, int64_t M, int64_t N,
                        float* out, float* partial, bool add, cudaStream_t st) {
    const int nch = wgrad_nchunks(M, N, R);
    int64_t rpc = (R + nch - 1) / nch;
    rpc = (rpc + kTnRows - 1) / kTnRows * kTnRows;
    const dim3 grid(nch, (unsigned)((M + kTnTile - 1) / kTnTile), (unsigned)((N + kTnTile - 1) / kTnTile));
    gemm_tn_partial_kernel<false><<<grid, kTnThreads, 0, st>>>(G, ldg, A, lda, R, (int)M, (int)N, partial, rpc, (int)N, nullptr, 0, 0);
    const int64_t n = M * N;
    if (add) reduce_partials_kernel<true><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partial, out, nch, n);
    else reduce_partials_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partial, out, nch, n);
    count_launch(2);
    return check_launch("gemm_tn");
}

int gemm_tn(const float* G, int64_t ldg, const float* A, int64_t lda, int64_t R, int64_t M, int64_t N,
            float* out, float* partial, cudaStream_t st) {
    return gemm_tn_impl(G, ldg, A, lda, R, M, N, out, partial, false, st);
}

// out1[M][N1] = G^T A1 over rows [0, R),  out2[M][N2] = G[shift:]^T A2[:R-shift]  in ONE pass over G.
__global__ void reduce_partials_split_kernel(const float* __restrict__ partial, float* __restrict__ out1, float* __restrict__ out2,
                                             int nchunks, int M, int N1, int N2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int N = N1 + N2;
    if (i >= (int64_t)M * N) return;
    float s = 0.f;
    for (int c = 0; c < nchunks; ++c) s += partial[(size_t)c * M * N + i];      // fixed order
    const int m = (int)(i / N), n = (int)(i % N);
    if (n < N1) out1[(size_t)m * N1 + n] = s;
    else out2[(size_t)m * N2 + (n - N1)] = s;
}

int gemm_tn2(const float* G, int64_t ldg, const float* A1, int64_t lda1, int64_t N1, const float* A2, int64_t lda2, int64_t N2,
             int64_t shift, int64_t R, int64_t M, float* out1, float* out2, float* partial, cudaStream_t st) {
    const int64_t N = N1 + N2;
    const int nch = wgrad_nchunks(M, N, R);
    int64_t rpc = (R + nch - 1) / nch;
    rpc = (rpc + kTnRows - 1) / kTnRows * kTnRows;
    const dim3 grid(nch, (unsigned)((M + kTnTile - 1) / kTnTile), (unsigned)((N + kTnTile - 1) / kTnTile));
    gemm_tn_partial_kernel<true><<<grid, kTnThreads, 0, st>>>(G, ldg, A1, lda1, R, (int)M, (int)N, partial, rpc, (int)N1, A2, lda2, shift);
    const int64_t n = M * N;
    reduce_partials_split_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partial, out1, out2, nch, (int)M, (int)N1, (int)N2);
    count_launch(2);
    return check_launch("gemm_tn2");
}

int reduce_partials(const float* partial, float* out, int nchunks, int64_t n, cudaStream_t st) {
    reduce_partials_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partial, out, nchunks, n);
    count_launch();
    return check_launch("reduce_partials");
}

int colsum(const float* G, int64_t ldg, int64_t R, int64_t M, float* out, float* partial, cudaStream_t st) {
    const int nch = wgrad_nchunks(M, 1, R);
    const int64_t rpc = (R + nch - 1) / nch;
    const dim3 grid(nch, (unsigned)((M + 127) / 128));
    colsum_partial_kernel<<<grid, 128, 0, st>>>(G, ldg, R, (int)M, partial, rpc);
    reduce_partials_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(partial, out, nch, M);
    count_launch(2);
    return check_launch("colsum");
}

}  // namespace na

extern "C" int64_t na_wgrad_partial_floats(int64_t K, int64_t H) {
    // worst case over the three reductions of one layer (row count unbounded)
    const int64_t M = 4 * H, big = (int64_t)1 << 40;
    const int64_t a = (int64_t)na::wgrad_nchunks(M, K + H, big) * M * (K + H);
    const int64_t b = (int64_t)na::wgrad_nchunks(M, H, big) * M * H;
    const int64_t c = (int64_t)na::wgrad_nchunks(M, 1, big) * M;
    return (a > b ? (a > c ? a : c) : (b > c ? b : c)) + 64;
}

extern "C" int na_lstm_layer_wgrad_f32_hx(const float* dgates, const float* in, const float* h, float* dw_ih,
                                          float* dw_hh, float* db, float* partials, int64_t T, int64_t Bp,
                                          int64_t K, int64_t H, const float* h_init, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(T >= 1 && Bp >= 1 && K >= 1 && H >= 1, NA_EINVAL, "na_lstm_layer_wgrad_f32: bad shape");
    NA_REQUIRE_PTR(dgates); NA_REQUIRE_PTR(in); NA_REQUIRE_PTR(h);
    NA_REQUIRE_PTR(dw_ih); NA_REQUIRE_PTR(dw_hh); NA_REQUIRE_PTR(db); NA_REQUIRE_PTR(partials);
    NA_OPTIONAL_PTR(h_init);
    cudaStream_t st = as_stream(stream);
    const int64_t R = T * Bp, G = 4 * H;
    int rc;
    if (K + H <= kTnTile) {
        // [in | h_{t-1}] fits one 64-column tile (layer 0 of the flagship: 8 + 48): dW_ih (all rows) and dW_hh (rows t >= 1
        // paired with h_{t-1} = the h rows shifted down by Bp) in ONE pass over dgates (10.2 -> 6.7 ms per 8,192 windows)
        rc = gemm_tn2(dgates, G, in, K, K, h, H, H, Bp, R, G, dw_ih, dw_hh, partials, st);
    } else {
        rc = gemm_tn(dgates, G, in, K, R, G, K, dw_ih, partials, st);
        if (rc) return rc;
        if (T > 1) rc = gemm_tn(dgates + Bp * G, G, h, H, R - Bp, G, H, dw_hh, partials, st);
        else rc = (int)cudaMemsetAsync(dw_hh, 0, sizeof(float) * G * H, st);
    }
    if (rc) return rc;
    // step 0 pairs with h_{-1} = h_init (zero without it): dW_hh += dgates_0^T h_init
    if (h_init && (rc = gemm_tn_impl(dgates, G, h_init, H, Bp, G, H, dw_hh, partials, true, st))) return rc;
    return colsum(dgates, G, R, G, db, partials, st);
}

extern "C" int na_lstm_layer_wgrad_f32(const float* dgates, const float* in, const float* h, float* dw_ih,
                                       float* dw_hh, float* db, float* partials, int64_t T, int64_t Bp,
                                       int64_t K, int64_t H, na_stream_t stream) {
    return na_lstm_layer_wgrad_f32_hx(dgates, in, h, dw_ih, dw_hh, db, partials, T, Bp, K, H, nullptr, stream);
}
