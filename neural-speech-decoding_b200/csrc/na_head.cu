// K4: attention pool over time (online softmax) + LayerNorm + Linear(H,32) + RReLU + Dropout
// + Linear(32,NC) (+ class softmax).  Replaces lstm_eeg_model.py:35-39 (+ :97).
// One warp per window; h is read exactly once from HBM (T*H*4 bytes per window), the
// [B,T,H] weighted temporary of the reference (:37) is never materialised.
#include "na_common.cuh"

namespace na {

int gemm_tn(const float* G, int64_t ldg, const float* A, int64_t lda, int64_t R, int64_t M, int64_t N,
            float* out, float* partial, cudaStream_t st);
int colsum(const float* G, int64_t ldg, int64_t R, int64_t M, float* out, float* partial, cudaStream_t st);
int reduce_partials(const float* partial, float* out, int nchunks, int64_t n, cudaStream_t st);

constexpr int kHeadWarps = 8;
constexpr int kFc = NA_FC_HIDDEN;

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

struct HeadParams {
    const float *attn_w, *attn_b, *ln_w, *ln_b, *fc0_w, *fc0_b, *fc3_w, *fc3_b;
    const float *rrelu_slope, *drop_mask;
    float drop_scale;
};

// Shared by forward and backward: LN -> fc0 -> RReLU -> dropout for one window held by a warp.
// zp[i] = pooled value of unit j = lane + 32 i.  Returns a_pre / a_post of fc unit `lane`.
template <int JPL>
__device__ __forceinline__ void head_tail(const float (&zp)[JPL], const HeadParams& p, const float* w0t,
                                          float* zs_warp, int64_t b, int H, int lane, float (&xhat)[JPL],
                                          float& rstd, float& a_pre, float& a_post, float& act_grad) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < JPL; ++i) s += (lane + 32 * i < H) ? zp[i] : 0.f;
    const float mean = warp_sum(s) / (float)H;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < JPL; ++i) {
        const float d = (lane + 32 * i < H) ? zp[i] - mean : 0.f;
        q = fmaf(d, d, q);
    }
    const float var = warp_sum(q) / (float)H;      // biased variance (nn.LayerNorm)
    rstd = 1.0f / sqrtf(var + kLnEps);
#pragma unroll
    for (int i = 0; i < JPL; ++i) {
        const int j = lane + 32 * i;
        xhat[i] = 0.f;
        if (j < H) {
            xhat[i] = (zp[i] - mean) * rstd;
            zs_warp[j] = fmaf(xhat[i], p.ln_w[j], p.ln_b[j]);
        }
    }
    __syncwarp();
    float a = p.fc0_b[lane];
    for (int j = 0; j < H; ++j) a = fmaf(w0t[j * (kFc + 1) + lane], zs_warp[j], a);
    const float slope = p.rrelu_slope ? p.rrelu_slope[b * kFc + lane] : kRReluEvalSlope;
    const float keep = p.drop_mask ? p.drop_mask[b * kFc + lane] * p.drop_scale : 1.0f;
    a_pre = a;
    act_grad = (a >= 0.f ? 1.0f : slope) * keep;
    a_post = (a >= 0.f ? a : a * slope) * keep;
}

// kEx: also store the attention scores (time-major [T][B], lane 0), the pooled vector and the LayerNorm output ([B][H]).
template <int JPL, int CH, bool kEx = false>
__global__ void __launch_bounds__(kHeadWarps * 32)
head_fwd_kernel(const float* __restrict__ h, HeadParams p, float* __restrict__ logits,
                float* __restrict__ probs, float* __restrict__ stats, float* __restrict__ zpool,
                const float* __restrict__ zpool_in,      // != NULL: tail only (pooling was done upstream)
                int T, int64_t B, int64_t Bp, int H, int NC,
                float* __restrict__ scores_tm, float* __restrict__ pooled, float* __restrict__ embedding) {
    extern __shared__ float smem[];
    float* w0t = smem;                               // [H][33]  fc0_w transposed
    float* zs = smem + H * (kFc + 1);                // [warps][H]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int idx = threadIdx.x; idx < kFc * H; idx += blockDim.x) {
        const int o = idx / H, j = idx % H;
        w0t[j * (kFc + 1) + o] = p.fc0_w[idx];
    }
    __syncthreads();
    const int64_t b = (int64_t)blockIdx.x * kHeadWarps + warp;
    if (b >= B) return;

    float wa[JPL], z[JPL];
#pragma unroll
    for (int i = 0; i < JPL; ++i) {
        const int j = lane + 32 * i;
        wa[i] = (j < H) ? p.attn_w[j] : 0.f;
        z[i] = 0.f;
    }
    const float ba = p.attn_b[0];
    float m = -INFINITY, l = 0.f;
    if (zpool_in != nullptr) {
        T = 0;                                    // skip the time loop below
        l = 1.0f;
#pragma unroll
        for (int i = 0; i < JPL; ++i) {
            const int j = lane + 32 * i;
            z[i] = (j < H) ? zpool_in[b * H + j] : 0.f;
        }
    }
    for (int t0 = 0; t0 < T; t0 += CH) {
        float hv[CH][JPL];
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const int t = t0 + u;
            const float* row = h + ((int64_t)t * Bp + b) * H;
#pragma unroll
            for (int i = 0; i < JPL; ++i) {
                const int j = lane + 32 * i;
                hv[u][i] = (t < T && j < H) ? __ldg(row + j) : 0.f;
            }
        }
        float s[CH];
        float cm = -INFINITY;
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            float d = 0.f;
#pragma unroll
            for (int i = 0; i < JPL; ++i) d = fmaf(hv[u][i], wa[i], d);
            s[u] = (t0 + u < T) ? warp_sum(d) + ba : -INFINITY;
            cm = fmaxf(cm, s[u]);
            if constexpr (kEx)
                if (scores_tm && lane == 0 && t0 + u < T) scores_tm[(int64_t)(t0 + u) * B + b] = s[u];
        }
        const float mn = fmaxf(m, cm);
        const float sc = expf(m - mn);     // first chunk: exp(-inf) = 0
        l *= sc;
#pragma unroll
        for (int i = 0; i < JPL; ++i) z[i] *= sc;
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const float e = expf(s[u] - mn);
            l += e;
#pragma unroll
            for (int i = 0; i < JPL; ++i) z[i] = fmaf(e, hv[u][i], z[i]);
        }
        m = mn;
    }
    float zp[JPL], xhat[JPL];
#pragma unroll
    for (int i = 0; i < JPL; ++i) {
        zp[i] = z[i] / l;
        const int j = lane + 32 * i;
        if (zpool && j < H) zpool[b * H + j] = zp[i];
        if constexpr (kEx)
            if (pooled && j < H) pooled[b * H + j] = zp[i];
    }
    if (stats && lane == 0) { stats[2 * b] = m; stats[2 * b + 1] = l; }

    float rstd, a_pre, a_post, act_grad;
    head_tail<JPL>(zp, p, w0t, zs + warp * H, b, H, lane, xhat, rstd, a_pre, a_post, act_grad);
    if constexpr (kEx)
        if (embedding)
            for (int j = lane; j < H; j += 32) embedding[b * H + j] = zs[warp * H + j];
    float lg = -INFINITY;
    for (int k = 0; k < NC; ++k) {
        const float v = warp_sum(a_post * p.fc3_w[k * kFc + lane]) + p.fc3_b[k];
        if (lane == k) lg = v;
    }
    if (lane < NC) logits[b * NC + lane] = lg;
    if (probs) {
        const float mx = warp_max(lg);
        const float e = (lane < NC) ? expf(lg - mx) : 0.f;
        const float sum = warp_sum(e);
        if (lane < NC) probs[b * NC + lane] = e / sum;
    }
}

// Backward.  scratch row b: [a_post 32 | da_pre 32 | zn H | dzn*xhat H | dzn H]; the parameter
// gradients are then plain column sums / G^T A products over the batch (na_reduce.cu).
template <int JPL, int CH>
__global__ void __launch_bounds__(kHeadWarps * 32)
head_bwd_kernel(const float* __restrict__ dlogits, const float* __restrict__ h, const float* __restrict__ stats,
                const float* __restrict__ zpool, HeadParams p, float* __restrict__ dh,
                float* __restrict__ scratch, float* __restrict__ wa_partial,
                float* __restrict__ dz_out,              // != NULL: tail only -> dz [B,H]; no time loop, dh untouched
                int T, int64_t B, int64_t Bp, int H, int NC) {
    extern __shared__ float smem[];
    float* w0t = smem;                               // [H][33]
    float* zs = w0t + H * (kFc + 1);                 // [warps][H]
    float* red = zs + kHeadWarps * H;                // [warps][H+1]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int S = 2 * kFc + 3 * H;
    for (int idx = threadIdx.x; idx < kFc * H; idx += blockDim.x) {
        const int o = idx / H, j = idx % H;
        w0t[j * (kFc + 1) + o] = p.fc0_w[idx];
    }
    __syncthreads();
    const int64_t b = (int64_t)blockIdx.x * kHeadWarps + warp;   // < Bp by construction of the grid

    float dwa[JPL];
    float dba = 0.f;
#pragma unroll
    for (int i = 0; i < JPL; ++i) dwa[i] = 0.f;

    if (b >= B) {
        if (b < Bp && dz_out == nullptr)
            for (int t = 0; t < T; ++t) {
                float* row = dh + ((int64_t)t * Bp + b) * H;
                for (int j = lane; j < H; j += 32) row[j] = 0.f;
            }
    } else {
        float wa[JPL], zp[JPL], xhat[JPL];
#pragma unroll
        for (int i = 0; i < JPL; ++i) {
            const int j = lane + 32 * i;
            wa[i] = (j < H) ? p.attn_w[j] : 0.f;
            zp[i] = (j < H) ? zpool[b * H + j] : 0.f;
        }
        const float ba = p.attn_b[0];
        const float m = dz_out ? 0.f : stats[2 * b], l = dz_out ? 1.f : stats[2 * b + 1];
        float rstd, a_pre, a_post, act_grad;
        head_tail<JPL>(zp, p, w0t, zs + warp * H, b, H, lane, xhat, rstd, a_pre, a_post, act_grad);

        const float dl = (lane < NC) ? dlogits[b * NC + lane] : 0.f;
        float da = 0.f;
        for (int k = 0; k < NC; ++k) da = fmaf(p.fc3_w[k * kFc + lane], __shfl_sync(0xffffffffu, dl, k), da);
        const float da_pre = da * act_grad;
        float* srow = scratch + b * S;
        srow[lane] = a_post;
        srow[kFc + lane] = da_pre;

        float dzn[JPL];
#pragma unroll
        for (int i = 0; i < JPL; ++i) dzn[i] = 0.f;
        for (int o = 0; o < kFc; ++o) {
            const float d = __shfl_sync(0xffffffffu, da_pre, o);
#pragma unroll
            for (int i = 0; i < JPL; ++i) {
                const int j = lane + 32 * i;
                if (j < H) dzn[i] = fmaf(w0t[j * (kFc + 1) + o], d, dzn[i]);
            }
        }
        float s1 = 0.f, s2 = 0.f, dxh[JPL];
#pragma unroll
        for (int i = 0; i < JPL; ++i) {
            const int j = lane + 32 * i;
            dxh[i] = 0.f;
            if (j < H) {
                srow[2 * kFc + j] = zs[warp * H + j];
                srow[2 * kFc + H + j] = dzn[i] * xhat[i];
                srow[2 * kFc + 2 * H + j] = dzn[i];
                dxh[i] = dzn[i] * p.ln_w[j];
                s1 += dxh[i];
                s2 = fmaf(dxh[i], xhat[i], s2);
            }
        }
        const float m1 = warp_sum(s1) / (float)H, m2 = warp_sum(s2) / (float)H;
        float dz[JPL];
#pragma unroll
        for (int i = 0; i < JPL; ++i) {
            const int j = lane + 32 * i;
            dz[i] = (j < H) ? rstd * (dxh[i] - m1 - xhat[i] * m2) : 0.f;
        }
        const float inv_l = 1.0f / l;
        if (dz_out != nullptr) {
            T = 0;                                // tail only: hand dz to the fused BPTT kernel
#pragma unroll
            for (int i = 0; i < JPL; ++i) {
                const int j = lane + 32 * i;
                if (j < H) dz_out[b * H + j] = dz[i];
            }
        }
        // Softmax-over-time backward in CENTRED form: with z = sum_t alpha_t h_t,
        //   ds_t = alpha_t (dz.h_t - dz.z) = alpha_t dz.(h_t - z),   sum_t ds_t = 0  =>
        //   d attn_w = sum_t ds_t h_t = sum_t ds_t (h_t - z).
        // Subtracting z element-wise first removes the cancellation between two large dot products
        // (attention is near-uniform, h_t ~ z) that costs ~2 digits in fp32.

        for (int t0 = 0; t0 < T; t0 += CH) {
            float hv[CH][JPL];
#pragma unroll
            for (int u = 0; u < CH; ++u) {
                const int t = t0 + u;
                const float* row = h + ((int64_t)t * Bp + b) * H;
#pragma unroll
                for (int i = 0; i < JPL; ++i) {
                    const int j = lane + 32 * i;
                    hv[u][i] = (t < T && j < H) ? __ldg(row + j) : 0.f;
                }
            }
#pragma unroll
            for (int u = 0; u < CH; ++u) {
                const int t = t0 + u;
                float d = 0.f, g = 0.f, hc[JPL];
#pragma unroll
                for (int i = 0; i < JPL; ++i) {
                    d = fmaf(hv[u][i], wa[i], d);
                    hc[i] = hv[u][i] - zp[i];
                    g = fmaf(hc[i], dz[i], g);
                }
                d = warp_sum(d) + ba;
                g = warp_sum(g);
                if (t < T) {
                    const float alpha = expf(d - m) * inv_l;
                    const float ds = alpha * g;
                    float* orow = dh + ((int64_t)t * Bp + b) * H;
#pragma unroll
                    for (int i = 0; i < JPL; ++i) {
                        const int j = lane + 32 * i;
                        if (j < H) orow[j] = fmaf(alpha, dz[i], ds * wa[i]);
                        dwa[i] = fmaf(ds, hc[i], dwa[i]);
                    }
                    dba += ds;
                }
            }
        }
    }
    // per-CTA partial of (d attn_w, d attn_b), warps summed in a fixed order
#pragma unroll
    for (int i = 0; i < JPL; ++i) {
        const int j = lane + 32 * i;
        if (j < H) red[warp * (H + 1) + j] = dwa[i];
    }
    if (lane == 0) red[warp * (H + 1) + H] = dba;
    __syncthreads();
    for (int j = threadIdx.x; j < H + 1; j += blockDim.x) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kHeadWarps; ++w) s += red[w * (H + 1) + j];
        wa_partial[(size_t)blockIdx.x * (H + 1) + j] = s;
    }
}

template <int JPL, int CH, bool kEx = false>
int launch_head_fwd(const float* h, const HeadParams& p, float* logits, float* probs, float* stats, float* zpool,
                    int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC, cudaStream_t st,
                    const float* zpool_in = nullptr, float* scores_tm = nullptr, float* pooled = nullptr,
                    float* embedding = nullptr) {
    const size_t smem = sizeof(float) * (H * (kFc + 1) + kHeadWarps * H);      // 164 KB at H = 1024
    if (int rc = prepare_launch(head_fwd_kernel<JPL, CH, kEx>, kHeadWarps * 32, smem, "na_head_fwd_f32")) return rc;
    const unsigned grid = (unsigned)((B + kHeadWarps - 1) / kHeadWarps);
    head_fwd_kernel<JPL, CH, kEx><<<grid, kHeadWarps * 32, smem, st>>>(h, p, logits, probs, stats, zpool, zpool_in, (int)T, B, Bp,
                                                                     (int)H, (int)NC, scores_tm, pooled, embedding);
    count_launch();
    return check_launch("na_head_fwd_f32");
}

template <int JPL, int CH>
int launch_head_bwd(const float* dlogits, const float* h, const float* stats, const float* zpool,
                    const HeadParams& p, float* dh, float* scratch, float* wa_partial, int64_t T, int64_t B,
                    int64_t Bp, int64_t H, int64_t NC, cudaStream_t st, float* dz_out = nullptr) {
    const size_t smem = sizeof(float) * (H * (kFc + 1) + kHeadWarps * H + kHeadWarps * (H + 1));   // 196 KB at H = 1024
    if (int rc = prepare_launch(head_bwd_kernel<JPL, CH>, kHeadWarps * 32, smem, "na_head_bwd_f32")) return rc;
    const unsigned grid = (unsigned)(Bp / kHeadWarps);
    head_bwd_kernel<JPL, CH><<<grid, kHeadWarps * 32, smem, st>>>(dlogits, h, stats, zpool, p, dh, scratch,
                                                                wa_partial, dz_out, (int)T, B, Bp, (int)H, (int)NC);
    count_launch();
    return check_launch("na_head_bwd_f32");
}

static int check_head_shape(const char* fn, int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC) {
    NA_REQUIRE(T >= 1 && B >= 1 && Bp >= B && Bp % NA_BATCH_ALIGN == 0, NA_EINVAL,
               "%s: bad shape T=%lld B=%lld Bp=%lld", fn, (long long)T, (long long)B, (long long)Bp);
    NA_REQUIRE(H >= 1 && H <= 1024, NA_EUNSUPPORTED, "%s: H=%lld outside [1,1024]", fn, (long long)H);
    NA_REQUIRE(NC >= 1 && NC <= NA_MAX_CLASSES, NA_EUNSUPPORTED, "%s: num_classes=%lld outside [1,%d]", fn,
               (long long)NC, NA_MAX_CLASSES);
    return NA_OK;
}

}  // namespace na

extern "C" int na_head_fwd_f32_ex(const float* h, const float* attn_w, const float* attn_b, const float* ln_w,
                                  const float* ln_b, const float* fc0_w, const float* fc0_b, const float* fc3_w,
                                  const float* fc3_b, const float* rrelu_slope, const float* drop_mask,
                                  float drop_scale, float* logits, float* probs, float* scores_tm, float* pooled,
                                  float* embedding, float* stats, float* zpool, int64_t T, int64_t B, int64_t Bp, int64_t H,
                                  int64_t NC, na_stream_t stream) {
    using namespace na;
    if (int rc = check_head_shape("na_head_fwd_f32", T, B, Bp, H, NC)) return rc;
    NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(logits);
    NA_OPTIONAL_PTR(scores_tm); NA_OPTIONAL_PTR(pooled); NA_OPTIONAL_PTR(embedding);
    NA_REQUIRE(attn_w && attn_b && ln_w && ln_b && fc0_w && fc0_b && fc3_w && fc3_b, NA_EINVAL,
               "na_head_fwd_f32: null parameter pointer");
    HeadParams p{attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, rrelu_slope, drop_mask, drop_scale};
    cudaStream_t st = as_stream(stream);
    if (scores_tm || pooled || embedding) {
#define NA_HEAD_EX(JPL, CH) \
        launch_head_fwd<JPL, CH, true>(h, p, logits, probs, stats, zpool, T, B, Bp, H, NC, st, nullptr, scores_tm, pooled, embedding)
        if (H <= 64) return NA_HEAD_EX(2, 8);
        if (H <= 128) return NA_HEAD_EX(4, 4);
        if (H <= 256) return NA_HEAD_EX(8, 2);
        if (H <= 512) return NA_HEAD_EX(16, 1);
        return NA_HEAD_EX(32, 1);
#undef NA_HEAD_EX
    }
    if (H <= 64) return launch_head_fwd<2, 8>(h, p, logits, probs, stats, zpool, T, B, Bp, H, NC, st);
    if (H <= 128) return launch_head_fwd<4, 4>(h, p, logits, probs, stats, zpool, T, B, Bp, H, NC, st);
    if (H <= 256) return launch_head_fwd<8, 2>(h, p, logits, probs, stats, zpool, T, B, Bp, H, NC, st);
    if (H <= 512) return launch_head_fwd<16, 1>(h, p, logits, probs, stats, zpool, T, B, Bp, H, NC, st);
    return launch_head_fwd<32, 1>(h, p, logits, probs, stats, zpool, T, B, Bp, H, NC, st);
}

extern "C" int na_head_fwd_f32(const float* h, const float* attn_w, const float* attn_b, const float* ln_w,
                               const float* ln_b, const float* fc0_w, const float* fc0_b, const float* fc3_w,
                               const float* fc3_b, const float* rrelu_slope, const float* drop_mask,
                               float drop_scale, float* logits, float* probs, float* stats, float* zpool,
                               int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC, na_stream_t stream) {
    return na_head_fwd_f32_ex(h, attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, rrelu_slope, drop_mask, drop_scale,
                              logits, probs, nullptr, nullptr, nullptr, stats, zpool, T, B, Bp, H, NC, stream);
}

namespace na {
// Attention pool of every prefix of the windows (EEG_LSTM.decode_prefixes on the FFMA path): h TMP [T][Bp][H] -> pooled
// [B][P][H], row j = the softmax-over-time pool of steps [0, t_j), t_j = min((j + 1) stride, T), P = ceil(T / stride).  One
// warp per window, h read once (rows of CH steps in flight, as in head_fwd_kernel).  The online softmax takes one step at a
// time -- score attn_w . h_t + attn_b, the running max raised with the rescale exp(m_old - m_new) -- so that z / l is the
// pooled vector of the prefix that ends at the step just taken in; it is stored at every prefix end.
// kState (EEG_LSTM.decode_stream, with stride = T: one pooled row): the online softmax starts from the state (m, l, z)
// the earlier chunks of the stream left, when m_in / l_in / z_in are given, and its state after the last step is stored
// to m_out / l_out [B] and z_out [B][H].
// kRagged (with kState; EEG_LSTM.decode_stream with lengths): window b takes in steps t < lengths[b] (clamped to [0, T])
// only, and its pooled row z / l is stored after them: the pool state it came with when it takes in none.
template <int JPL, int CH, bool kState = false, bool kRagged = false>
__global__ void __launch_bounds__(kHeadWarps * 32)
attention_pool_prefix_kernel(const float* __restrict__ h, const float* __restrict__ attn_w, const float* __restrict__ attn_b,
                             float* __restrict__ pooled, int T, int64_t B, int64_t Bp, int H, int stride,
                             const float* __restrict__ m_in = nullptr, const float* __restrict__ l_in = nullptr,
                             const float* __restrict__ z_in = nullptr, float* __restrict__ m_out = nullptr,
                             float* __restrict__ l_out = nullptr, float* __restrict__ z_out = nullptr,
                             const int32_t* __restrict__ lengths = nullptr) {
    static_assert(!kRagged || kState, "per-row lengths are a variant of the stream pool");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t b = (int64_t)blockIdx.x * kHeadWarps + warp;
    if (b >= B) return;
    const int Tb = kRagged ? min(max(lengths[b], 0), T) : T;    // the steps window b takes in
    float wa[JPL], z[JPL];
#pragma unroll
    for (int i = 0; i < JPL; ++i) {
        const int j = lane + 32 * i;
        wa[i] = (j < H) ? attn_w[j] : 0.f;
        z[i] = 0.f;
    }
    const float ba = attn_b[0];
    float* out = pooled + b * ((T + stride - 1) / stride) * H;
    float m = -INFINITY, l = 0.f;
    if constexpr (kState)
        if (z_in) {
            m = m_in[b];
            l = l_in[b];
#pragma unroll
            for (int i = 0; i < JPL; ++i) {
                const int j = lane + 32 * i;
                if (j < H) z[i] = z_in[b * H + j];
            }
        }
    int left = stride;                            // steps until the next prefix end
    for (int t0 = 0; t0 < Tb; t0 += CH) {
        float hv[CH][JPL];
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const int t = t0 + u;
            const float* row = h + ((int64_t)t * Bp + b) * H;
#pragma unroll
            for (int i = 0; i < JPL; ++i) {
                const int j = lane + 32 * i;
                hv[u][i] = (t < Tb && j < H) ? __ldg(row + j) : 0.f;
            }
        }
        float s[CH];
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            float d = 0.f;
#pragma unroll
            for (int i = 0; i < JPL; ++i) d = fmaf(hv[u][i], wa[i], d);
            s[u] = warp_sum(d) + ba;
        }
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const int t = t0 + u;
            if (t >= Tb) break;
            if (s[u] > m) {                       // first step: exp(-inf) = 0
                const float sc = expf(m - s[u]);
                l *= sc;
#pragma unroll
                for (int i = 0; i < JPL; ++i) z[i] *= sc;
                m = s[u];
            }
            const float e = expf(s[u] - m);
            l += e;
#pragma unroll
            for (int i = 0; i < JPL; ++i) z[i] = fmaf(e, hv[u][i], z[i]);
            if (!kRagged && (--left == 0 || t == T - 1)) {
                const float inv = 1.0f / l;
#pragma unroll
                for (int i = 0; i < JPL; ++i) {
                    const int j = lane + 32 * i;
                    if (j < H) out[j] = z[i] * inv;
                }
                out += H;
                left = stride;
            }
        }
    }
    if constexpr (kRagged) {                      // the one pooled row (stride T), after the row's last step
        const float inv = 1.0f / l;
#pragma unroll
        for (int i = 0; i < JPL; ++i) {
            const int j = lane + 32 * i;
            if (j < H) out[j] = z[i] * inv;
        }
    }
    if constexpr (kState) {
#pragma unroll
        for (int i = 0; i < JPL; ++i) {
            const int j = lane + 32 * i;
            if (j < H) z_out[b * H + j] = z[i];
        }
        if (lane == 0) {
            m_out[b] = m;
            l_out[b] = l;
        }
    }
}

template <int JPL, int CH>
int launch_attention_pool_prefix(const float* h, const float* attn_w, const float* attn_b, float* pooled, int64_t T, int64_t B,
                                 int64_t Bp, int64_t H, int stride, cudaStream_t st) {
    if (int rc = prepare_launch(attention_pool_prefix_kernel<JPL, CH>, kHeadWarps * 32, 0, "na_attention_pool_prefix_f32"))
        return rc;
    const unsigned grid = (unsigned)((B + kHeadWarps - 1) / kHeadWarps);
    attention_pool_prefix_kernel<JPL, CH><<<grid, kHeadWarps * 32, 0, st>>>(h, attn_w, attn_b, pooled, (int)T, B, Bp, (int)H,
                                                                           stride);
    count_launch();
    return check_launch("na_attention_pool_prefix_f32");
}
}  // namespace na

namespace na {
template <int JPL, int CH>
int launch_attention_pool_stream(const float* h, const float* attn_w, const float* attn_b, const float* m_in, const float* l_in,
                                 const float* z_in, float* pooled, float* m_out, float* l_out, float* z_out, int64_t T,
                                 int64_t B, int64_t Bp, int64_t H, cudaStream_t st) {
    if (int rc = prepare_launch(attention_pool_prefix_kernel<JPL, CH, true>, kHeadWarps * 32, 0, "na_attention_pool_stream_f32"))
        return rc;
    const unsigned grid = (unsigned)((B + kHeadWarps - 1) / kHeadWarps);
    attention_pool_prefix_kernel<JPL, CH, true><<<grid, kHeadWarps * 32, 0, st>>>(
        h, attn_w, attn_b, pooled, (int)T, B, Bp, (int)H, (int)T, m_in, l_in, z_in, m_out, l_out, z_out);
    count_launch();
    return check_launch("na_attention_pool_stream_f32");
}
}  // namespace na

namespace na {
template <int JPL, int CH>
int launch_attention_pool_stream_ragged(const float* h, const float* attn_w, const float* attn_b, const float* m_in,
                                        const float* l_in, const float* z_in, const int32_t* lengths, float* pooled,
                                        float* m_out, float* l_out, float* z_out, int64_t T, int64_t B, int64_t Bp,
                                        int64_t H, cudaStream_t st) {
    if (int rc = prepare_launch(attention_pool_prefix_kernel<JPL, CH, true, true>, kHeadWarps * 32, 0,
                                "na_attention_pool_stream_ragged_f32"))
        return rc;
    const unsigned grid = (unsigned)((B + kHeadWarps - 1) / kHeadWarps);
    attention_pool_prefix_kernel<JPL, CH, true, true><<<grid, kHeadWarps * 32, 0, st>>>(
        h, attn_w, attn_b, pooled, (int)T, B, Bp, (int)H, (int)T, m_in, l_in, z_in, m_out, l_out, z_out, lengths);
    count_launch();
    return check_launch("na_attention_pool_stream_ragged_f32");
}
}  // namespace na

extern "C" int na_attention_pool_stream_ragged_f32(const float* h, const float* attn_w, const float* attn_b,
                                                   const float* m_in, const float* l_in, const float* z_in,
                                                   const int32_t* lengths, float* pooled, float* m_out, float* l_out,
                                                   float* z_out, int64_t T, int64_t B, int64_t Bp, int64_t H,
                                                   na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(T >= 1 && T <= INT32_MAX && B >= 1 && Bp >= B && Bp % NA_BATCH_ALIGN == 0, NA_EINVAL,
               "na_attention_pool_stream_ragged_f32: bad shape T=%lld B=%lld Bp=%lld", (long long)T, (long long)B,
               (long long)Bp);
    NA_REQUIRE(H >= 1 && H <= 1024, NA_EUNSUPPORTED, "na_attention_pool_stream_ragged_f32: H=%lld outside [1,1024]",
               (long long)H);
    NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(lengths);
    NA_REQUIRE_PTR(pooled); NA_REQUIRE_PTR(m_out); NA_REQUIRE_PTR(l_out); NA_REQUIRE_PTR(z_out);
    NA_REQUIRE(attn_w && attn_b, NA_EINVAL, "na_attention_pool_stream_ragged_f32: null parameter pointer");
    const int given = (m_in != nullptr) + (l_in != nullptr) + (z_in != nullptr);
    NA_REQUIRE(given == 0 || given == 3, NA_EINVAL,
               "na_attention_pool_stream_ragged_f32: m_in, l_in and z_in must be given together (or all NULL)");
    NA_OPTIONAL_PTR(m_in); NA_OPTIONAL_PTR(l_in); NA_OPTIONAL_PTR(z_in);
    cudaStream_t st = as_stream(stream);
#define NA_POOL_RAGGED(JPL, CH)                                                                                        \
    launch_attention_pool_stream_ragged<JPL, CH>(h, attn_w, attn_b, m_in, l_in, z_in, lengths, pooled, m_out, l_out, \
                                                 z_out, T, B, Bp, H, st)
    if (H <= 64) return NA_POOL_RAGGED(2, 8);
    if (H <= 128) return NA_POOL_RAGGED(4, 4);
    if (H <= 256) return NA_POOL_RAGGED(8, 2);
    if (H <= 512) return NA_POOL_RAGGED(16, 1);
    return NA_POOL_RAGGED(32, 1);
#undef NA_POOL_RAGGED
}

extern "C" int na_attention_pool_stream_f32(const float* h, const float* attn_w, const float* attn_b, const float* m_in,
                                            const float* l_in, const float* z_in, float* pooled, float* m_out, float* l_out,
                                            float* z_out, int64_t T, int64_t B, int64_t Bp, int64_t H, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(T >= 1 && T <= INT32_MAX && B >= 1 && Bp >= B && Bp % NA_BATCH_ALIGN == 0, NA_EINVAL,
               "na_attention_pool_stream_f32: bad shape T=%lld B=%lld Bp=%lld", (long long)T, (long long)B, (long long)Bp);
    NA_REQUIRE(H >= 1 && H <= 1024, NA_EUNSUPPORTED, "na_attention_pool_stream_f32: H=%lld outside [1,1024]", (long long)H);
    NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(pooled); NA_REQUIRE_PTR(m_out); NA_REQUIRE_PTR(l_out); NA_REQUIRE_PTR(z_out);
    NA_REQUIRE(attn_w && attn_b, NA_EINVAL, "na_attention_pool_stream_f32: null parameter pointer");
    const int given = (m_in != nullptr) + (l_in != nullptr) + (z_in != nullptr);
    NA_REQUIRE(given == 0 || given == 3, NA_EINVAL,
               "na_attention_pool_stream_f32: m_in, l_in and z_in must be given together (or all NULL)");
    NA_OPTIONAL_PTR(m_in); NA_OPTIONAL_PTR(l_in); NA_OPTIONAL_PTR(z_in);
    cudaStream_t st = as_stream(stream);
#define NA_POOL_STREAM(JPL, CH) \
    launch_attention_pool_stream<JPL, CH>(h, attn_w, attn_b, m_in, l_in, z_in, pooled, m_out, l_out, z_out, T, B, Bp, H, st)
    if (H <= 64) return NA_POOL_STREAM(2, 8);
    if (H <= 128) return NA_POOL_STREAM(4, 4);
    if (H <= 256) return NA_POOL_STREAM(8, 2);
    if (H <= 512) return NA_POOL_STREAM(16, 1);
    return NA_POOL_STREAM(32, 1);
#undef NA_POOL_STREAM
}

extern "C" int na_attention_pool_prefix_f32(const float* h, const float* attn_w, const float* attn_b, float* pooled, int64_t T,
                                            int64_t B, int64_t Bp, int64_t H, int64_t stride, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(T >= 1 && T <= INT32_MAX && B >= 1 && Bp >= B && Bp % NA_BATCH_ALIGN == 0, NA_EINVAL,
               "na_attention_pool_prefix_f32: bad shape T=%lld B=%lld Bp=%lld", (long long)T, (long long)B, (long long)Bp);
    NA_REQUIRE(H >= 1 && H <= 1024, NA_EUNSUPPORTED, "na_attention_pool_prefix_f32: H=%lld outside [1,1024]", (long long)H);
    NA_REQUIRE(stride >= 1, NA_EINVAL, "na_attention_pool_prefix_f32: stride=%lld < 1", (long long)stride);
    NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(pooled);
    NA_REQUIRE(attn_w && attn_b, NA_EINVAL, "na_attention_pool_prefix_f32: null parameter pointer");
    const int sd = (int)(stride < T ? stride : T);          // a stride past the window: one prefix, the whole window
    cudaStream_t st = as_stream(stream);
    if (H <= 64) return launch_attention_pool_prefix<2, 8>(h, attn_w, attn_b, pooled, T, B, Bp, H, sd, st);
    if (H <= 128) return launch_attention_pool_prefix<4, 4>(h, attn_w, attn_b, pooled, T, B, Bp, H, sd, st);
    if (H <= 256) return launch_attention_pool_prefix<8, 2>(h, attn_w, attn_b, pooled, T, B, Bp, H, sd, st);
    if (H <= 512) return launch_attention_pool_prefix<16, 1>(h, attn_w, attn_b, pooled, T, B, Bp, H, sd, st);
    return launch_attention_pool_prefix<32, 1>(h, attn_w, attn_b, pooled, T, B, Bp, H, sd, st);
}

namespace na {
// Attention weights from the time-major scores the inference kernels wrote: scores [T][B] -> attn [B][T], per window
// alpha_t = exp(s_t - max_t s) / sum_t exp(s_t - max_t s) in fp32 (torch.softmax's two passes; a NaN score makes the
// window's whole row NaN, as in torch).  A CTA owns 32 windows: lane = window for the reads (one 128-byte run per step),
// the 8 warps stride over time, partial maxima / sums are combined in a fixed order; the write pass transposes 32 x 32
// blocks through shared memory so that lane = step for the stores.
constexpr int kSmWarps = 8;
__global__ void __launch_bounds__(kSmWarps * 32) attention_softmax_kernel(const float* __restrict__ s, float* __restrict__ a,
                                                                          int64_t T, int64_t B) {
    __shared__ float red[kSmWarps][32];
    __shared__ float tile[kSmWarps][32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t b0 = (int64_t)blockIdx.x * 32, b = b0 + lane;
    const bool live = b < B;
    auto nan_max = [](float m, float v) { return (v > m || v != v) ? v : m; };     // NaN wins, as torch.max
    float m = -INFINITY;
    if (live)
        for (int64_t t = warp; t < T; t += kSmWarps) m = nan_max(m, __ldg(s + t * B + b));
    red[warp][lane] = m;
    __syncthreads();
    m = red[0][lane];
#pragma unroll
    for (int w = 1; w < kSmWarps; ++w) m = nan_max(m, red[w][lane]);
    __syncthreads();
    float l = 0.f;
    if (live)
        for (int64_t t = warp; t < T; t += kSmWarps) l += expf(__ldg(s + t * B + b) - m);
    red[warp][lane] = l;
    __syncthreads();
    l = 0.f;
#pragma unroll
    for (int w = 0; w < kSmWarps; ++w) l += red[w][lane];
    // write pass: warp w handles steps [32 k, 32 k + 32) for k = w, w + 8, ...
    __shared__ float mrow[32], lrow[32];
    if (warp == 0) { mrow[lane] = m; lrow[lane] = l; }
    __syncthreads();
    const int nb = B - b0 < 32 ? (int)(B - b0) : 32;
    for (int64_t t0 = (int64_t)warp * 32; t0 < T; t0 += kSmWarps * 32) {
        const int nt = T - t0 < 32 ? (int)(T - t0) : 32;
        for (int i = 0; i < nt; ++i)                       // row i = step t0 + i, lane = window
            if (live) tile[warp][i][lane] = __ldg(s + (t0 + i) * B + b);
        __syncwarp();
        for (int r = 0; r < nb; ++r)                       // row r = window b0 + r, lane = step
            if (lane < nt) a[(b0 + r) * T + t0 + lane] = expf(tile[warp][lane][r] - mrow[r]) / lrow[r];
        __syncwarp();
    }
}
}  // namespace na

extern "C" int na_attention_softmax_f32(const float* scores_tm, float* attn, int64_t T, int64_t B, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(T >= 1 && T <= INT32_MAX && B >= 1, NA_EINVAL, "na_attention_softmax_f32: bad shape T=%lld B=%lld", (long long)T,
               (long long)B);
    NA_REQUIRE_PTR(scores_tm); NA_REQUIRE_PTR(attn);
    attention_softmax_kernel<<<(unsigned)((B + 31) / 32), kSmWarps * 32, 0, as_stream(stream)>>>(scores_tm, attn, T, B);
    count_launch();
    return check_launch("na_attention_softmax_f32");
}

extern "C" int64_t na_head_param_floats(int64_t H, int64_t NC) {
    return H + 1 + H + H + NA_FC_HIDDEN * H + NA_FC_HIDDEN + NA_FC_HIDDEN * NC + NC;
}

extern "C" int64_t na_head_partial_floats(int64_t B, int64_t H, int64_t NC) {
    const int64_t S = 2 * NA_FC_HIDDEN + 3 * H;
    const int64_t Bp = (B + NA_BATCH_ALIGN - 1) / NA_BATCH_ALIGN * NA_BATCH_ALIGN;
    const int64_t widest = (H > NC ? H : NC);
    return B * S + (Bp / na::kHeadWarps) * (H + 1) + 296 * NA_FC_HIDDEN * (widest > 64 ? widest : 64) + 256;
}

extern "C" int na_head_bwd_f32(const float* dlogits, const float* h, const float* stats, const float* zpool,
                               const float* attn_w, const float* attn_b, const float* ln_w, const float* ln_b,
                               const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                               const float* rrelu_slope, const float* drop_mask, float drop_scale, float* dh,
                               float* dparams, float* partials, int64_t T, int64_t B, int64_t Bp, int64_t H,
                               int64_t NC, na_stream_t stream) {
    using namespace na;
    if (int rc = check_head_shape("na_head_bwd_f32", T, B, Bp, H, NC)) return rc;
    NA_REQUIRE_PTR(dlogits); NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(stats); NA_REQUIRE_PTR(zpool);
    NA_REQUIRE_PTR(dh); NA_REQUIRE_PTR(dparams); NA_REQUIRE_PTR(partials);
    NA_REQUIRE(attn_w && attn_b && ln_w && ln_b && fc0_w && fc0_b && fc3_w && fc3_b, NA_EINVAL,
               "na_head_bwd_f32: null parameter pointer");
    HeadParams p{attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, rrelu_slope, drop_mask, drop_scale};
    cudaStream_t st = as_stream(stream);
    const int64_t S = 2 * kFc + 3 * H;
    const int64_t nblk = Bp / kHeadWarps;
    float* scratch = partials;
    float* wa_partial = scratch + B * S;
    float* gpart = wa_partial + nblk * (H + 1);
    gpart += (4 - ((gpart - partials) & 3)) & 3;   // keep 16-byte alignment of the sub-buffer
    int rc;
    if (H <= 64) rc = launch_head_bwd<2, 8>(dlogits, h, stats, zpool, p, dh, scratch, wa_partial, T, B, Bp, H, NC, st);
    else if (H <= 128) rc = launch_head_bwd<4, 4>(dlogits, h, stats, zpool, p, dh, scratch, wa_partial, T, B, Bp, H, NC, st);
    else if (H <= 256) rc = launch_head_bwd<8, 2>(dlogits, h, stats, zpool, p, dh, scratch, wa_partial, T, B, Bp, H, NC, st);
    else if (H <= 512) rc = launch_head_bwd<16, 1>(dlogits, h, stats, zpool, p, dh, scratch, wa_partial, T, B, Bp, H, NC, st);
    else rc = launch_head_bwd<32, 1>(dlogits, h, stats, zpool, p, dh, scratch, wa_partial, T, B, Bp, H, NC, st);
    if (rc) return rc;
    // dparams: [attn_w H | attn_b 1 | ln_w H | ln_b H | fc0_w 32H | fc0_b 32 | fc3_w 32NC | fc3_b NC]
    float* d_attn = dparams;
    float* d_lnw = d_attn + H + 1;
    float* d_lnb = d_lnw + H;
    float* d_fc0w = d_lnb + H;
    float* d_fc0b = d_fc0w + kFc * H;
    float* d_fc3w = d_fc0b + kFc;
    float* d_fc3b = d_fc3w + kFc * NC;
    if ((rc = reduce_partials(wa_partial, d_attn, (int)nblk, H + 1, st))) return rc;
    if ((rc = colsum(scratch + 2 * kFc + H, S, B, H, d_lnw, gpart, st))) return rc;
    if ((rc = colsum(scratch + 2 * kFc + 2 * H, S, B, H, d_lnb, gpart, st))) return rc;
    if ((rc = gemm_tn(scratch + kFc, S, scratch + 2 * kFc, S, B, kFc, H, d_fc0w, gpart, st))) return rc;
    if ((rc = colsum(scratch + kFc, S, B, kFc, d_fc0b, gpart, st))) return rc;
    if ((rc = gemm_tn(dlogits, NC, scratch, S, B, NC, kFc, d_fc3w, gpart, st))) return rc;
    return colsum(dlogits, NC, B, NC, d_fc3b, gpart, st);
}


// ---- tail-only forms (pooling fused upstream / time loop fused downstream: tensor-core training tier) ----
extern "C" int na_head_tail_fwd_f32(const float* zpool, const float* attn_w, const float* attn_b, const float* ln_w,
                                    const float* ln_b, const float* fc0_w, const float* fc0_b, const float* fc3_w,
                                    const float* fc3_b, const float* rrelu_slope, const float* drop_mask,
                                    float drop_scale, float* logits, float* probs, int64_t B, int64_t H, int64_t NC,
                                    na_stream_t stream) {
    using namespace na;
    const int64_t Bp = (B + NA_BATCH_ALIGN - 1) / NA_BATCH_ALIGN * NA_BATCH_ALIGN;
    if (int rc = check_head_shape("na_head_tail_fwd_f32", 1, B, Bp, H, NC)) return rc;
    NA_REQUIRE_PTR(zpool); NA_REQUIRE_PTR(logits);
    NA_REQUIRE(attn_w && attn_b && ln_w && ln_b && fc0_w && fc0_b && fc3_w && fc3_b, NA_EINVAL,
               "na_head_tail_fwd_f32: null parameter pointer");
    HeadParams p{attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, rrelu_slope, drop_mask, drop_scale};
    cudaStream_t st = as_stream(stream);
    if (H <= 64) return launch_head_fwd<2, 8>(nullptr, p, logits, probs, nullptr, nullptr, 1, B, Bp, H, NC, st, zpool);
    if (H <= 128) return launch_head_fwd<4, 4>(nullptr, p, logits, probs, nullptr, nullptr, 1, B, Bp, H, NC, st, zpool);
    if (H <= 256) return launch_head_fwd<8, 2>(nullptr, p, logits, probs, nullptr, nullptr, 1, B, Bp, H, NC, st, zpool);
    if (H <= 512) return launch_head_fwd<16, 1>(nullptr, p, logits, probs, nullptr, nullptr, 1, B, Bp, H, NC, st, zpool);
    return launch_head_fwd<32, 1>(nullptr, p, logits, probs, nullptr, nullptr, 1, B, Bp, H, NC, st, zpool);
}

// dlogits -> dz [B,H] (gradient w.r.t. the pooled vector) + the gradients of ln / fc0 / fc3 in `dparams`
// (same packing as na_head_bwd_f32; the attn_w / attn_b slots are zeroed -- the fused BPTT kernel owns them).
extern "C" int na_head_tail_bwd_f32(const float* dlogits, const float* zpool, const float* attn_w, const float* attn_b,
                                    const float* ln_w, const float* ln_b, const float* fc0_w, const float* fc0_b,
                                    const float* fc3_w, const float* fc3_b, const float* rrelu_slope,
                                    const float* drop_mask, float drop_scale, float* dz, float* dparams, float* partials,
                                    int64_t B, int64_t H, int64_t NC, na_stream_t stream) {
    using namespace na;
    const int64_t Bp = (B + NA_BATCH_ALIGN - 1) / NA_BATCH_ALIGN * NA_BATCH_ALIGN;
    if (int rc = check_head_shape("na_head_tail_bwd_f32", 1, B, Bp, H, NC)) return rc;
    NA_REQUIRE_PTR(dlogits); NA_REQUIRE_PTR(zpool); NA_REQUIRE_PTR(dz); NA_REQUIRE_PTR(dparams); NA_REQUIRE_PTR(partials);
    NA_REQUIRE(attn_w && attn_b && ln_w && ln_b && fc0_w && fc0_b && fc3_w && fc3_b, NA_EINVAL,
               "na_head_tail_bwd_f32: null parameter pointer");
    HeadParams p{attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, rrelu_slope, drop_mask, drop_scale};
    cudaStream_t st = as_stream(stream);
    const int64_t S = 2 * kFc + 3 * H;
    const int64_t nblk = Bp / kHeadWarps;
    float* scratch = partials;
    float* wa_partial = scratch + B * S;
    float* gpart = wa_partial + nblk * (H + 1);
    gpart += (4 - ((gpart - partials) & 3)) & 3;
    int rc;
    if (H <= 64) rc = launch_head_bwd<2, 8>(dlogits, nullptr, nullptr, zpool, p, nullptr, scratch, wa_partial, 1, B, Bp, H, NC, st, dz);
    else if (H <= 128) rc = launch_head_bwd<4, 4>(dlogits, nullptr, nullptr, zpool, p, nullptr, scratch, wa_partial, 1, B, Bp, H, NC, st, dz);
    else if (H <= 256) rc = launch_head_bwd<8, 2>(dlogits, nullptr, nullptr, zpool, p, nullptr, scratch, wa_partial, 1, B, Bp, H, NC, st, dz);
    else if (H <= 512) rc = launch_head_bwd<16, 1>(dlogits, nullptr, nullptr, zpool, p, nullptr, scratch, wa_partial, 1, B, Bp, H, NC, st, dz);
    else rc = launch_head_bwd<32, 1>(dlogits, nullptr, nullptr, zpool, p, nullptr, scratch, wa_partial, 1, B, Bp, H, NC, st, dz);
    if (rc) return rc;
    float* d_attn = dparams;
    float* d_lnw = d_attn + H + 1;
    float* d_lnb = d_lnw + H;
    float* d_fc0w = d_lnb + H;
    float* d_fc0b = d_fc0w + kFc * H;
    float* d_fc3w = d_fc0b + kFc;
    float* d_fc3b = d_fc3w + kFc * NC;
    if ((rc = (int)cudaMemsetAsync(d_attn, 0, sizeof(float) * (H + 1), st))) return fail(rc, "na_head_tail_bwd_f32: memset failed");
    if ((rc = colsum(scratch + 2 * kFc + H, S, B, H, d_lnw, gpart, st))) return rc;
    if ((rc = colsum(scratch + 2 * kFc + 2 * H, S, B, H, d_lnb, gpart, st))) return rc;
    if ((rc = gemm_tn(scratch + kFc, S, scratch + 2 * kFc, S, B, kFc, H, d_fc0w, gpart, st))) return rc;
    if ((rc = colsum(scratch + kFc, S, B, kFc, d_fc0b, gpart, st))) return rc;
    if ((rc = gemm_tn(dlogits, NC, scratch, S, B, NC, kFc, d_fc3w, gpart, st))) return rc;
    return colsum(dlogits, NC, B, NC, d_fc3b, gpart, st);
}
