// K3 (generic tier): one LSTM layer forward / fused BPTT for ANY (K <= 4096, H <= 1024).
// This is the always-correct CUDA path behind the drop-in module for sizes the specialised
// kernels (na_lstm_h48.cu) do not cover.  Exact fp32: FFMA accumulation, libm activations.
//
// Layouts are time-major padded (TMP): row (t, b) = t*Bp + b.
#include "na_common.cuh"
#include <algorithm>

namespace na {

constexpr int kGenTile = 8;   // windows per CTA (the BPTT kernel's transposed d(gates) tile assumes 8)
static_assert(kGenTile == 8, "lstm_bwd_generic_kernel packs the 8 windows of a gate column into two float4");
// Threads per CTA at most.  Both kernels need 95-128 registers a thread, so 512 threads is what one CTA can get from the
// 64 K-register file; beyond it a thread owns UPT = 2 hidden units (H <= 1024) and the backward's threads loop over the
// K + H columns of its contraction.
constexpr int kGenMaxThreads = 512;

__global__ void pack_lstm_layer_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                                       const float* __restrict__ b_ih, const float* __restrict__ b_hh,
                                       float* __restrict__ wt, float* __restrict__ bias, int K, int H) {
    const int G = 4 * H;
    const int n = (K + H) * G;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += gridDim.x * blockDim.x) {
        const int k = idx / G, col = idx % G;
        wt[idx] = (k < K) ? w_ih[col * K + k] : w_hh[col * H + (k - K)];
    }
    for (int col = blockIdx.x * blockDim.x + threadIdx.x; col < G; col += gridDim.x * blockDim.x)
        bias[col] = b_ih[col] + b_hh[col];
}

// Thread j owns hidden units j + u * blockDim.x (u < UPT) for all kGenTile windows of the tile: the four weight columns of
// a k-step are loaded once (coalesced over j) and reused for every window; [x_t | h_{t-1}] is broadcast from shared memory.
// h_init / c_init [Bp][H] (optional) are h_{-1} / c_{-1}; zeros without them.
template <int UPT>
__global__ void __launch_bounds__(kGenMaxThreads)
lstm_fwd_generic_kernel(const float* __restrict__ in, const float* __restrict__ wt, const float* __restrict__ bias,
                        float* __restrict__ hout, float* __restrict__ cout, float* __restrict__ gates,
                        const float* __restrict__ drop_mask, float drop_scale, float* __restrict__ hout_drop,
                        int T, int64_t Bp, int K, int H,
                        const float* __restrict__ h_init, const float* __restrict__ c_init) {
    extern __shared__ float smem[];
    const int KH = K + H, G = 4 * H;
    float* a_s = smem;                       // [kGenTile][KH]
    const int64_t b0 = (int64_t)blockIdx.x * kGenTile;

    float c[UPT][kGenTile];
#pragma unroll
    for (int u = 0; u < UPT; ++u) {
        const int j = threadIdx.x + u * blockDim.x;
#pragma unroll
        for (int b = 0; b < kGenTile; ++b) c[u][b] = (c_init && j < H) ? c_init[(b0 + b) * H + j] : 0.f;
    }
    for (int idx = threadIdx.x; idx < kGenTile * KH; idx += blockDim.x) {
        const int b = idx / KH, k = idx % KH;
        a_s[idx] = (h_init && k >= K) ? h_init[(b0 + b) * H + (k - K)] : 0.f;
    }
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        const int64_t row0 = (int64_t)t * Bp + b0;
        for (int idx = threadIdx.x; idx < kGenTile * K; idx += blockDim.x) {
            const int b = idx / K, k = idx % K;
            a_s[b * KH + k] = in[(row0 + b) * K + k];
        }
        __syncthreads();
        float hn[UPT][kGenTile];             // h_t, written to a_s once every thread has read h_{t-1}
#pragma unroll
        for (int u = 0; u < UPT; ++u) {
            const int j = threadIdx.x + u * blockDim.x;
            if (j >= H) continue;
            float ai[kGenTile], af[kGenTile], ag[kGenTile], ao[kGenTile];
            const float bi = bias[j], bf = bias[H + j], bg = bias[2 * H + j], bo = bias[3 * H + j];
#pragma unroll
            for (int b = 0; b < kGenTile; ++b) { ai[b] = bi; af[b] = bf; ag[b] = bg; ao[b] = bo; }
            for (int k = 0; k < KH; ++k) {
                const float* wrow = wt + (size_t)k * G + j;
                const float wi = __ldg(wrow), wf = __ldg(wrow + H), wg = __ldg(wrow + 2 * H), wo = __ldg(wrow + 3 * H);
#pragma unroll
                for (int b = 0; b < kGenTile; ++b) {
                    const float a = a_s[b * KH + k];
                    ai[b] = fmaf(a, wi, ai[b]);
                    af[b] = fmaf(a, wf, af[b]);
                    ag[b] = fmaf(a, wg, ag[b]);
                    ao[b] = fmaf(a, wo, ao[b]);
                }
            }
#pragma unroll
            for (int b = 0; b < kGenTile; ++b) {
                const float i = sigmoid_acc(ai[b]), f = sigmoid_acc(af[b]);
                const float g = tanh_acc(ag[b]), o = sigmoid_acc(ao[b]);
                c[u][b] = fmaf(f, c[u][b], i * g);
                const float h = o * tanh_acc(c[u][b]);
                hn[u][b] = h;
                const int64_t row = row0 + b;
                hout[row * H + j] = h;
                if (hout_drop) hout_drop[row * H + j] = h * drop_mask[row * H + j] * drop_scale;
                if (cout) cout[row * H + j] = c[u][b];
                if (gates) {
                    float* gr = gates + row * G + j;
                    gr[0] = i; gr[H] = f; gr[2 * H] = g; gr[3 * H] = o;
                }
            }
        }
        __syncthreads();   // everyone is done reading h_{t-1}
#pragma unroll
        for (int u = 0; u < UPT; ++u) {
            const int j = threadIdx.x + u * blockDim.x;
            if (j < H) {
#pragma unroll
                for (int b = 0; b < kGenTile; ++b) a_s[b * KH + K + j] = hn[u][b];
            }
        }
        // the barrier at the top of the next step orders these h writes before the next reads
    }
}

// Reverse-time pass.  Threads do the elementwise gate backward of units j + u * blockDim.x (u < UPT); then they produce
// columns jj = threadIdx.x, threadIdx.x + blockDim.x, ... < K+H of dgates . [W_ih | W_hh]  (din for jj < K, recurrent dh
// otherwise).  Optional, [Bp][H] each: c_init = c_{-1} (zeros without it); dh_last / dc_last = the gradients w.r.t. this
// layer's final h / c, which enter at t = T-1; dh_init / dc_init receive the gradients w.r.t. h_{-1} / c_{-1}.
template <int UPT>
__global__ void __launch_bounds__(kGenMaxThreads)
lstm_bwd_generic_kernel(const float* __restrict__ dh_out, const float* __restrict__ gates, const float* __restrict__ cstate,
                        const float* __restrict__ w_ih, const float* __restrict__ w_hh, float* __restrict__ dgates,
                        float* __restrict__ din, const float* __restrict__ in_drop_mask, float drop_scale, int T,
                        int64_t Bp, int K, int H, const float* __restrict__ c_init, const float* __restrict__ dh_last,
                        const float* __restrict__ dc_last, float* __restrict__ dh_init, float* __restrict__ dc_init) {
    extern __shared__ float smem[];
    const int G = 4 * H;
    float* dg_s = smem;                         // [kGenTile][G]
    float* dhrec_s = smem + kGenTile * G;       // [kGenTile][H]
    const int64_t b0 = (int64_t)blockIdx.x * kGenTile;

    float dc[UPT][kGenTile];
#pragma unroll
    for (int u = 0; u < UPT; ++u) {
        const int j = threadIdx.x + u * blockDim.x;
#pragma unroll
        for (int b = 0; b < kGenTile; ++b) dc[u][b] = (dc_last && j < H) ? dc_last[(b0 + b) * H + j] : 0.f;
    }
    for (int idx = threadIdx.x; idx < kGenTile * H; idx += blockDim.x)
        dhrec_s[idx] = dh_last ? dh_last[(b0 + idx / H) * H + idx % H] : 0.f;
    __syncthreads();

    for (int t = T - 1; t >= 0; --t) {
        const int64_t row0 = (int64_t)t * Bp + b0;
#pragma unroll
        for (int u = 0; u < UPT; ++u) {
            const int j = threadIdx.x + u * blockDim.x;
            if (j >= H) continue;
            float pi_[kGenTile], pf_[kGenTile], pg_[kGenTile], po_[kGenTile];
#pragma unroll
            for (int b = 0; b < kGenTile; ++b) {
                const int64_t row = row0 + b;
                const float* gr = gates + row * G + j;
                const float i = gr[0], f = gr[H], g = gr[2 * H], o = gr[3 * H];
                const float ct = cstate[row * H + j];
                const float cp = (t > 0) ? cstate[(row - Bp) * H + j] : (c_init ? c_init[(b0 + b) * H + j] : 0.f);
                const float tc = tanh_acc(ct);
                const float dh = dh_out[row * H + j] + dhrec_s[b * H + j];
                const float d_o = dh * tc;
                const float dct = fmaf(dh * o, 1.0f - tc * tc, dc[u][b]);
                const float d_i = dct * g, d_g = dct * i, d_f = dct * cp;
                dc[u][b] = dct * f;
                const float pi = d_i * i * (1.0f - i);
                const float pf = d_f * f * (1.0f - f);
                const float pg = d_g * (1.0f - g * g);
                const float po = d_o * o * (1.0f - o);
                float* dgr = dgates + row * G + j;
                dgr[0] = pi; dgr[H] = pf; dgr[2 * H] = pg; dgr[3 * H] = po;
                pi_[b] = pi; pf_[b] = pf; pg_[b] = pg; po_[b] = po;
            }
            // d(gates) of this step in shared memory, TRANSPOSED: [gate column][window], so that the contraction below reads
            // the 8 windows of a column with two 16-byte broadcast loads instead of eight 4-byte ones
            float4* d4 = reinterpret_cast<float4*>(dg_s);
            d4[(j) * 2] = make_float4(pi_[0], pi_[1], pi_[2], pi_[3]);             d4[(j) * 2 + 1] = make_float4(pi_[4], pi_[5], pi_[6], pi_[7]);
            d4[(H + j) * 2] = make_float4(pf_[0], pf_[1], pf_[2], pf_[3]);         d4[(H + j) * 2 + 1] = make_float4(pf_[4], pf_[5], pf_[6], pf_[7]);
            d4[(2 * H + j) * 2] = make_float4(pg_[0], pg_[1], pg_[2], pg_[3]);     d4[(2 * H + j) * 2 + 1] = make_float4(pg_[4], pg_[5], pg_[6], pg_[7]);
            d4[(3 * H + j) * 2] = make_float4(po_[0], po_[1], po_[2], po_[3]);     d4[(3 * H + j) * 2 + 1] = make_float4(po_[4], po_[5], po_[6], po_[7]);
        }
        __syncthreads();
        for (int jj = (din != nullptr) ? threadIdx.x : K + threadIdx.x; jj < K + H; jj += blockDim.x) {
            const bool is_in = jj < K;
            float acc[kGenTile];
#pragma unroll
            for (int b = 0; b < kGenTile; ++b) acc[b] = 0.f;
            const float* wcol = is_in ? (w_ih + jj) : (w_hh + (jj - K));
            const int ld = is_in ? K : H;
            const float4* d4 = reinterpret_cast<const float4*>(dg_s);
#pragma unroll 4
            for (int col = 0; col < G; ++col) {
                const float w = __ldg(wcol + (size_t)col * ld);
                const float4 a = d4[col * 2], b4 = d4[col * 2 + 1];
                acc[0] = fmaf(a.x, w, acc[0]); acc[1] = fmaf(a.y, w, acc[1]); acc[2] = fmaf(a.z, w, acc[2]); acc[3] = fmaf(a.w, w, acc[3]);
                acc[4] = fmaf(b4.x, w, acc[4]); acc[5] = fmaf(b4.y, w, acc[5]); acc[6] = fmaf(b4.z, w, acc[6]); acc[7] = fmaf(b4.w, w, acc[7]);
            }
            if (is_in) {
#pragma unroll
                for (int b = 0; b < kGenTile; ++b) {
                    const int64_t o = (row0 + b) * K + jj;
                    din[o] = in_drop_mask ? acc[b] * in_drop_mask[o] * drop_scale : acc[b];
                }
            } else {
#pragma unroll
                for (int b = 0; b < kGenTile; ++b) dhrec_s[b * H + (jj - K)] = acc[b];
            }
        }
        __syncthreads();
    }
    if (dh_init)
        for (int idx = threadIdx.x; idx < kGenTile * H; idx += blockDim.x) dh_init[(b0 + idx / H) * H + idx % H] = dhrec_s[idx];
    if (dc_init) {
#pragma unroll
        for (int u = 0; u < UPT; ++u) {
            const int j = threadIdx.x + u * blockDim.x;
            if (j < H) {
#pragma unroll
                for (int b = 0; b < kGenTile; ++b) dc_init[(b0 + b) * H + j] = dc[u][b];
            }
        }
    }
}

}  // namespace na

extern "C" int na_pack_lstm_layer(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                                  float* wt, float* bias, int64_t K, int64_t H, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(K >= 1 && H >= 1 && K <= 4096 && H <= 1024, NA_EUNSUPPORTED,
               "na_pack_lstm_layer: unsupported K=%lld H=%lld", (long long)K, (long long)H);
    NA_REQUIRE_PTR(w_ih); NA_REQUIRE_PTR(w_hh); NA_REQUIRE_PTR(b_ih); NA_REQUIRE_PTR(b_hh);
    NA_REQUIRE_PTR(wt); NA_REQUIRE_PTR(bias);
    const int n = (int)((K + H) * 4 * H);
    pack_lstm_layer_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(w_ih, w_hh, b_ih, b_hh, wt, bias, (int)K, (int)H);
    count_launch();
    return check_launch("na_pack_lstm_layer");
}

namespace na {
int lstm_layer_fwd_generic(const float* in, const float* wt, const float* bias, float* hout, float* cout,
                           float* gates, const float* drop_mask, float drop_scale, float* hout_drop,
                           int64_t T, int64_t Bp, int64_t K, int64_t H, const float* h_init, const float* c_init,
                           cudaStream_t st) {
    const int threads = (int)std::min<int64_t>((H + 31) / 32 * 32, kGenMaxThreads);
    const size_t smem = sizeof(float) * kGenTile * (K + H);      // 160 KB at K = 4096, H = 1024
    auto kern = (H > kGenMaxThreads) ? lstm_fwd_generic_kernel<2> : lstm_fwd_generic_kernel<1>;
    if (int rc = prepare_launch(kern, threads, smem, "na_lstm_layer_fwd_f32(generic)")) return rc;
    kern<<<(unsigned)(Bp / kGenTile), threads, smem, st>>>(
        in, wt, bias, hout, cout, gates, drop_mask, drop_scale, hout_drop, (int)T, Bp, (int)K, (int)H, h_init, c_init);
    count_launch();
    return check_launch("na_lstm_layer_fwd_f32(generic)");
}

int lstm_layer_bwd_generic(const float* dh_out, const float* gates, const float* cstate, const float* w_ih,
                           const float* w_hh, float* dgates, float* din, const float* in_drop_mask,
                           float drop_scale, int64_t T, int64_t Bp, int64_t K, int64_t H, const float* c_init,
                           const float* dh_last, const float* dc_last, float* dh_init, float* dc_init, cudaStream_t st) {
    const int threads = (int)std::min<int64_t>((K + H + 31) / 32 * 32, kGenMaxThreads);
    const size_t smem = sizeof(float) * kGenTile * (4 * H + H);  // 160 KB at H = 1024
    auto kern = (H > kGenMaxThreads) ? lstm_bwd_generic_kernel<2> : lstm_bwd_generic_kernel<1>;
    if (int rc = prepare_launch(kern, threads, smem, "na_lstm_layer_bwd_f32(generic)")) return rc;
    kern<<<(unsigned)(Bp / kGenTile), threads, smem, st>>>(
        dh_out, gates, cstate, w_ih, w_hh, dgates, din, in_drop_mask, drop_scale, (int)T, Bp, (int)K, (int)H, c_init, dh_last,
        dc_last, dh_init, dc_init);
    count_launch();
    return check_launch("na_lstm_layer_bwd_f32(generic)");
}
}  // namespace na
