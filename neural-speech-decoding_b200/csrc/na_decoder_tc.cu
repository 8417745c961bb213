// Tensor-core tier (bf16 operands, fp32 accumulate/state): the WHOLE 2-layer decoder forward
// (K2 input-gate contraction + K3 recurrence + K4 head + class softmax) as one persistent,
// warp-specialised sm_100a kernel built on tcgen05.mma / TMEM / TMA.
//
//   * CTA = one tile of 128 windows (UMMA M = 128, cta_group::1), one CTA per SM, persistent
//     over tiles.  Per layer and step ONE accumulator D[128 x 192] (all four gates of all 48
//     units) lives in TMEM: D0 at columns [0,192), D1 at [192,384).
//   * The time-parallel input contraction x_t.W_ih^T is not materialised (it would be HBM-write
//     bound, SURVEY 7.2): it is fused as extra K-steps of the per-step MMA,
//         layer 0:  A = [x_t (8) | 1 1 0.. (8) | h0_{t-1} (48)]            K = 64  (4 x K16)
//         layer 1:  A = [h0_t (48) | h1_{t-1} (48) | 1 1 0.. (8) | 0 (8)]  K = 112 (7 x K16)
//     and the bias rides on the constant-one columns as a bf16 hi+lo pair (fp32-accurate bias for
//     free).  B = [W_ih | bias | W_hh] is staged once per CTA in shared memory, K-major -- which
//     is exactly nn.LSTM's [4H, K] layout -- in the canonical no-swizzle core-matrix layout
//     ([K/8][rows][8] bf16: 8 rows x 16 B = one 128-B core matrix).
//   * A operands use the same layout, so (a) x_t of a tile is ONE contiguous 2 KB TMA bulk copy
//     from the time-major bf16 input and (b) the epilogue thread of window r writes the 8 bf16 of
//     a unit block with one conflict-free 16-B st.shared at row r.
//   * Gate columns are permuted to n = (j/8)*32 + gate*8 + j%8, so one tcgen05.ld.32x32b.x32
//     returns i,f,g,o of 8 units of the thread's window; c, the pooled sum and the softmax state
//     never leave registers.
//   * Warp roles (320 threads): warps 0-3 layer-0 epilogue, warps 4-7 layer-1 epilogue + attention
//     pooling + head, warp 8 MMA issuer (one lane), warp 9 TMA producer + TMEM allocator.
//     Layer 1 runs one step behind layer 0 (wavefront), so the two epilogue groups and the tensor
//     pipe overlap; all hand-offs are mbarriers (tcgen05.commit for MMA completion).
//   * Activations: tanh.approx.f32 (sigmoid = 0.5 tanh(x/2) + 0.5).  bf16 contract: logits within
//     2e-2 of the fp32 reference, argmax identical on the repo's windows.
#include "na_tc_common.cuh"

namespace na {
namespace tc {

constexpr int kXStages = 4;
constexpr int kK0Chunks = 8;                 // layer 0: x | ones | h0 x6
constexpr int kK1Chunks = 14;                // layer 1: h0 x6 | h1 x6 | ones | zero
constexpr int kThreads = 320;            // HS = 1; HS = 2 runs (16 + 2) warps = 576 threads
constexpr int kFc = NA_FC_HIDDEN;

struct HeadSmem {
    float wa[kH], lnw[kH], lnb[kH];
    float w0[kFc * kH];
    float b0[kFc];
    float w3[NA_MAX_CLASSES * kFc];
    float b3[NA_MAX_CLASSES];
    float ba;
};

struct Smem {
    alignas(128) unsigned char b0[kK0Chunks * kBChunk];          // 24,576
    alignas(128) unsigned char b1[kK1Chunks * kBChunk];          // 43,008
    alignas(128) unsigned char x[kXStages][2 * kAChunk];         // [x chunk | ones chunk] per stage
    alignas(128) unsigned char h0[2][6 * kAChunk];               // double-buffered h0_t
    alignas(128) unsigned char h1[6 * kAChunk];
    alignas(128) unsigned char onez[2 * kAChunk];                // [ones | zeros]
    HeadSmem head;
    alignas(8) uint64_t x_full[kXStages], x_empty[kXStages];
    uint64_t d0_full, d1_full, h0_ready[2], h0_free[2], h1_ready;
    uint32_t tmem_base;
    // HS == 2 only: the two half-row warps of a quarter exchange their partial attention scores every
    // step (double-buffered by step parity) and their pooled halves once per tile
    float score_part[2][2][kRows];
    float zx[kRows][kH / 2];
};

// ---- weight packing ----------------------------------------------------------------------------
// B0 [8 chunks][192][8] and B1 [14 chunks][192][8] bf16, row n = (j/8)*32 + gate*8 + j%8.
__global__ void pack_decoder_bf16_kernel(const float* __restrict__ w_ih0, const float* __restrict__ w_hh0,
                                         const float* __restrict__ b_ih0, const float* __restrict__ b_hh0,
                                         const float* __restrict__ w_ih1, const float* __restrict__ w_hh1,
                                         const float* __restrict__ b_ih1, const float* __restrict__ b_hh1,
                                         __nv_bfloat16* __restrict__ out) {
    const int total0 = kK0Chunks * 8 * kN, total1 = kK1Chunks * 8 * kN;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total0 + total1; idx += gridDim.x * blockDim.x) {
        const bool l1 = idx >= total0;
        const int e = l1 ? idx - total0 : idx;
        const int k = (e / (kN * 8)) * 8 + (e % 8);       // K index
        const int n = (e / 8) % kN;                       // permuted gate column
        const int j = (n / 32) * 8 + (n % 8), q = (n % 32) / 8;
        const int col = q * kH + j;                       // row of the torch weight tensors
        float v = 0.f;
        if (!l1) {
            const float b = b_ih0[col] + b_hh0[col];
            const float bh = val16_to_float(val16(b));
            if (k < 8) v = kF16InScaleInv * w_ih0[col * 8 + k];      // x is stored as x / 16 (na_common.cuh)
            else if (k == 8) v = bh;
            else if (k == 9) v = b - bh;
            else if (k >= 16) v = w_hh0[col * kH + (k - 16)];
        } else {
            const float b = b_ih1[col] + b_hh1[col];
            const float bh = val16_to_float(val16(b));
            if (k < 48) v = w_ih1[col * kH + k];
            else if (k < 96) v = w_hh1[col * kH + (k - 48)];
            else if (k == 96) v = bh;
            else if (k == 97) v = b - bh;
        }
        reinterpret_cast<uint16_t*>(out)[idx] = val16(v);
    }
}

// ---- the fused decoder kernel --------------------------------------------------------------------
// HS = number of epilogue warps per TMEM lane quarter and layer: each handles 6/HS unit blocks of its
// 32 windows.  HS = 2 doubles the warps per scheduler (4 instead of 2), which hides the
// tcgen05.ld / MUFU dependency latency that leaves the xu pipe at ~72 % with HS = 1.
template <int HS>
__global__ void __launch_bounds__((8 * HS + 2) * 32, 1)
decoder_infer_bf16_kernel(const __nv_bfloat16* __restrict__ x,        // TMP [T][Bp][8] bf16
                          const unsigned char* __restrict__ packed,   // B0 | B1 (pack_decoder_bf16_kernel)
                          const float* __restrict__ attn_w, const float* __restrict__ attn_b,
                          const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                          const float* __restrict__ fc0_w, const float* __restrict__ fc0_b,
                          const float* __restrict__ fc3_w, const float* __restrict__ fc3_b,
                          float* __restrict__ logits, float* __restrict__ probs,
                          int T, int64_t B, int64_t Bp, int NC, int nquarters) {
    constexpr int kThreads = (8 * HS + 2) * 32;       // shadows the namespace constant inside the kernel
    constexpr int kMmaWarp = 8 * HS, kTmaWarp = 8 * HS + 1, kNB = 6 / HS;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    Smem& S = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // ---- one-time setup --------------------------------------------------------------------------
    {
        const uint4* src = reinterpret_cast<const uint4*>(packed);
        uint4* dst = reinterpret_cast<uint4*>(S.b0);     // b0 and b1 are contiguous in Smem
        constexpr int n16 = (kK0Chunks + kK1Chunks) * kBChunk / 16;
        for (int i = tid; i < n16; i += kThreads) dst[i] = src[i];
        const uint4 ones = make_uint4(kValOnes2, 0u, 0u, 0u);     // bf16 {1,1,0,0,0,0,0,0}
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        for (int i = tid; i < kRows; i += kThreads) {
#pragma unroll
            for (int s = 0; s < kXStages; ++s) reinterpret_cast<uint4*>(S.x[s] + kAChunk)[i] = ones;
            reinterpret_cast<uint4*>(S.onez)[i] = ones;
            reinterpret_cast<uint4*>(S.onez + kAChunk)[i] = zero;
        }
        for (int i = tid; i < kH; i += kThreads) { S.head.wa[i] = attn_w[i]; S.head.lnw[i] = ln_w[i]; S.head.lnb[i] = ln_b[i]; }
        for (int i = tid; i < kFc * kH; i += kThreads) S.head.w0[i] = fc0_w[i];
        for (int i = tid; i < kFc; i += kThreads) S.head.b0[i] = fc0_b[i];
        for (int i = tid; i < NC * kFc; i += kThreads) S.head.w3[i] = fc3_w[i];
        for (int i = tid; i < NC; i += kThreads) S.head.b3[i] = fc3_b[i];
        if (tid == 0) {
            S.head.ba = attn_b[0];
            for (int s = 0; s < kXStages; ++s) { mbar_init(&S.x_full[s], 1); mbar_init(&S.x_empty[s], 1); }
            mbar_init(&S.d0_full, 1); mbar_init(&S.d1_full, 1);
            mbar_init(&S.h0_ready[0], 128 * HS); mbar_init(&S.h0_ready[1], 128 * HS);
            mbar_init(&S.h0_free[0], 1); mbar_init(&S.h0_free[1], 1);
            mbar_init(&S.h1_ready, 128 * HS);
            fence_mbar_init();
        }
        if (warp == kTmaWarp) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)),
                         "r"(kTmemCols)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        tc_fence_before();
        fence_proxy_async_smem();
        __syncthreads();
        tc_fence_after();
    }
    const uint32_t tmem = S.tmem_base;
    const uint32_t tmem_d0 = tmem, tmem_d1 = tmem + kN;

    // Work split: the batch is cut into 32-window quarters (one epilogue warp each); CTA i owns the
    // contiguous range [i*Q/G, (i+1)*Q/G) and walks it in tiles of up to 4 quarters.  A short last tile
    // keeps its idle epilogue warps out of the MUFU pipe, so the tail costs ~its share instead of a
    // whole extra 128-window round.
    const int q_begin = (int)(((int64_t)blockIdx.x * nquarters) / gridDim.x);
    const int q_end = (int)(((int64_t)(blockIdx.x + 1) * nquarters) / gridDim.x);
    int n0 = 0;                                            // running step index across tiles
    for (int q0 = q_begin; q0 < q_end; q0 += 4, n0 += T) {
        const int nq = min(4, q_end - q0);                 // active quarters of this tile
        const uint32_t x_bytes = (uint32_t)nq * 32u * 16u;
        const int64_t b0 = (int64_t)q0 * 32;
        // ---- zero h0_{-1}, h1_{-1} of this tile ----------------------------------------------------
        {
            uint4* z0 = reinterpret_cast<uint4*>(S.h0[(n0 + 1) & 1]);      // buffer of step n0-1
            uint4* z1 = reinterpret_cast<uint4*>(S.h1);
            for (int i = tid; i < 6 * kAChunk / 16; i += kThreads) { z0[i] = make_uint4(0, 0, 0, 0); z1[i] = make_uint4(0, 0, 0, 0); }
            fence_proxy_async_smem();
            __syncthreads();
        }

        if (warp == kTmaWarp) {
            // ================= TMA producer ==========================================================
            if (lane == 0) {
                for (int t = 0; t < T; ++t) {
                    const int n = n0 + t, s = n % kXStages, u = n / kXStages;
                    mbar_wait(&S.x_empty[s], (u & 1) ^ 1);
                    mbar_arrive_expect_tx(&S.x_full[s], x_bytes);
                    bulk_load(S.x[s], x + ((int64_t)t * Bp + b0) * 8, x_bytes, &S.x_full[s]);
                }
            }
        } else if (warp == kMmaWarp) {
            // ================= MMA issuer ============================================================
            if (lane == 0) {
                const uint64_t d_b0 = umma_desc(smem_u32(S.b0), kBChunk, 128), d_b1 = umma_desc(smem_u32(S.b1), kBChunk, 128);
                const uint64_t d_x0 = umma_desc(smem_u32(S.x[0]), kAChunk, 128);
                const uint64_t d_h0[2] = {umma_desc(smem_u32(S.h0[0]), kAChunk, 128), umma_desc(smem_u32(S.h0[1]), kAChunk, 128)};
                const uint64_t d_h1 = umma_desc(smem_u32(S.h1), kAChunk, 128), d_onez = umma_desc(smem_u32(S.onez), kAChunk, 128);
                for (int t = 0; t <= T; ++t) {
                    if (t < T) {                                   // layer 0, step n
                        const int n = n0 + t, s = n % kXStages, u = n / kXStages;
                        mbar_wait(&S.x_full[s], u & 1);
                        mbar_wait(&S.h0_ready[(n + 1) & 1], ((n - 1) >> 1) & 1);     // h0_{n-1} written, D0 drained
                        tc_fence_after();
                        const uint64_t hprev = d_h0[(n + 1) & 1];
                        umma_bf16(tmem_d0, desc_adv(d_x0, s * 2 * kAChunk), d_b0, 0u);
#pragma unroll
                        for (int i = 0; i < 3; ++i)
                            umma_bf16(tmem_d0, desc_adv(hprev, 2 * i * kAChunk), desc_adv(d_b0, (2 + 2 * i) * kBChunk), 1u);
                        umma_commit(&S.x_empty[s]);
                        umma_commit(&S.d0_full);
                    }
                    if (t >= 1) {                                  // layer 1, step m (one behind)
                        const int m = n0 + t - 1;
                        mbar_wait(&S.h0_ready[m & 1], (m >> 1) & 1);                 // h0_m written
                        mbar_wait(&S.h1_ready, (m - 1) & 1);                         // h1_{m-1} written, D1 drained
                        tc_fence_after();
                        const uint64_t hin = d_h0[m & 1];
#pragma unroll
                        for (int i = 0; i < 3; ++i)
                            umma_bf16(tmem_d1, desc_adv(hin, 2 * i * kAChunk), desc_adv(d_b1, 2 * i * kBChunk), i == 0 ? 0u : 1u);
#pragma unroll
                        for (int i = 0; i < 3; ++i)
                            umma_bf16(tmem_d1, desc_adv(d_h1, 2 * i * kAChunk), desc_adv(d_b1, (6 + 2 * i) * kBChunk), 1u);
                        umma_bf16(tmem_d1, d_onez, desc_adv(d_b1, 12 * kBChunk), 1u);
                        umma_commit(&S.d1_full);
                        umma_commit(&S.h0_free[m & 1]);
                    }
                }
            }
        } else if (warp < 4 * HS) {
            // ================= layer-0 epilogue: gates -> c, h0 (fp16) ================================
            const int q = warp & 3, hf = warp >> 2;
            const int row = q * 32 + lane;
            const uint32_t lane_base = (uint32_t)(q * 32) << 16;
            float c[8 * kNB];
#pragma unroll
            for (int j = 0; j < 8 * kNB; ++j) c[j] = 0.f;
            if (q >= nq) {                                 // idle quarter: keep the barrier protocol only
                for (int t = 0; t < T; ++t) {
                    const int n = n0 + t;
                    mbar_wait(&S.d0_full, n & 1);
                    mbar_arrive(&S.h0_ready[n & 1]);
                }
            } else
            for (int t = 0; t < T; ++t) {
                const int n = n0 + t;
                mbar_wait(&S.d0_full, n & 1);
                mbar_wait(&S.h0_free[n & 1], ((n >> 1) & 1) ^ 1);       // layer-1 MMA of step n-2 has read this buffer
                tc_fence_after();
                unsigned char* dst = S.h0[n & 1] + row * 16;
#pragma unroll
                for (int bb = 0; bb < kNB; ++bb) {
                    const int blk = hf * kNB + bb;
                    uint32_t v[32], hp[4];
                    tmem_ld32(tmem_d0 + lane_base + blk * 32, v);
                    cell_block(v, c + bb * 8, hp);
                    st_shared_v4(dst + blk * kAChunk, hp[0], hp[1], hp[2], hp[3]);
                }
                tc_fence_before();
                fence_proxy_async_smem();
                mbar_arrive(&S.h0_ready[n & 1]);
            }
        } else {
            // ================= layer-1 epilogue: gates -> c, h1; attention pooling; head ================
            const int q = (warp - 4 * HS) & 3, hf = (warp - 4 * HS) >> 2;
            const int row = q * 32 + lane;
            const uint32_t lane_base = (uint32_t)(q * 32) << 16;
            constexpr int kU = 8 * kNB;                    // units owned by this thread
            float c[kU], z[kU];
#pragma unroll
            for (int j = 0; j < kU; ++j) { c[j] = 0.f; z[j] = 0.f; }
            float mx = -INFINITY, l = 0.f;
            const float ba = S.head.ba;
            if (q >= nq) {                                 // idle quarter
                for (int t = 0; t < T; ++t) {
                    const int m = n0 + t;
                    mbar_wait(&S.d1_full, m & 1);
                    mbar_arrive(&S.h1_ready);
                }
            } else {
            for (int t = 0; t < T; ++t) {
                const int m = n0 + t;
                mbar_wait(&S.d1_full, m & 1);
                tc_fence_after();
                unsigned char* dst = S.h1 + row * 16;
                uint32_t hb[4 * kNB];
                float score = 0.f;
#pragma unroll
                for (int bb = 0; bb < kNB; ++bb) {
                    const int blk = hf * kNB + bb;
                    uint32_t v[32], hp[4];
                    tmem_ld32(tmem_d1 + lane_base + blk * 32, v);
                    cell_block(v, c + bb * 8, hp);
                    st_shared_v4(dst + blk * kAChunk, hp[0], hp[1], hp[2], hp[3]);
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        hb[bb * 4 + u] = hp[u];
                        score = fmaf(val_lo(hp[u]), S.head.wa[blk * 8 + 2 * u], score);
                        score = fmaf(val_hi(hp[u]), S.head.wa[blk * 8 + 2 * u + 1], score);
                    }
                }
                tc_fence_before();
                fence_proxy_async_smem();
                mbar_arrive(&S.h1_ready);
                if (HS == 2) {                             // total score = half 0 + half 1 (fixed order)
                    S.score_part[t & 1][hf][row] = score;
                    named_bar_sync(1 + q, 64);
                    score = S.score_part[t & 1][0][row] + S.score_part[t & 1][1][row];
                }
                score += ba;
                // online softmax over time (lstm_eeg_model.py:35-37), lazy rescale
                if (score > mx) {
                    const float sc = __expf(mx - score);
                    l *= sc;
#pragma unroll
                    for (int j = 0; j < kU; ++j) z[j] *= sc;
                    mx = score;
                }
                const float e = __expf(score - mx);
                l += e;
#pragma unroll
                for (int u = 0; u < 4 * kNB; ++u) {
                    z[2 * u] = fmaf(e, val_lo(hb[u]), z[2 * u]);
                    z[2 * u + 1] = fmaf(e, val_hi(hb[u]), z[2 * u + 1]);
                }
            }
            // ---- head for this window: LN -> fc0 -> RReLU(eval) -> fc3 -> softmax -------------------------
            float zf[kH];
            if (HS == 2) {                                 // half 1 hands its pooled half to half 0
                if (hf == 1) {
#pragma unroll
                    for (int j = 0; j < kU; ++j) S.zx[row][j] = z[j];
                }
                named_bar_sync(1 + q, 64);
#pragma unroll
                for (int j = 0; j < kU; ++j) { zf[j] = z[j]; zf[kU + j] = S.zx[row][j]; }
            } else {
#pragma unroll
                for (int j = 0; j < kU; ++j) zf[j] = z[j];
            }
            if (hf == 0) {
            const int64_t b = b0 + row;
            const float inv_l = 1.0f / l;
            float mean = 0.f;
#pragma unroll
            for (int j = 0; j < kH; ++j) { zf[j] *= inv_l; mean += zf[j]; }
            mean *= (1.0f / kH);
            float var = 0.f;
#pragma unroll
            for (int j = 0; j < kH; ++j) { const float d = zf[j] - mean; var = fmaf(d, d, var); }
            const float rstd = rsqrtf(var * (1.0f / kH) + kLnEps);
#pragma unroll
            for (int j = 0; j < kH; ++j) zf[j] = fmaf((zf[j] - mean) * rstd, S.head.lnw[j], S.head.lnb[j]);
            float lg[NA_MAX_CLASSES];
#pragma unroll
            for (int k = 0; k < NA_MAX_CLASSES; ++k) lg[k] = (k < NC) ? S.head.b3[k] : -INFINITY;
            for (int o = 0; o < kFc; ++o) {
                float a = S.head.b0[o];
#pragma unroll
                for (int j = 0; j < kH; ++j) a = fmaf(S.head.w0[o * kH + j], zf[j], a);
                a = a >= 0.f ? a : a * kRReluEvalSlope;
#pragma unroll
                for (int k = 0; k < NA_MAX_CLASSES; ++k)
                    if (k < NC) lg[k] = fmaf(S.head.w3[k * kFc + o], a, lg[k]);
            }
            if (b < B) {
                float mxl = -INFINITY;
#pragma unroll
                for (int k = 0; k < NA_MAX_CLASSES; ++k) mxl = fmaxf(mxl, lg[k]);
                float den = 0.f, pe[NA_MAX_CLASSES];
#pragma unroll
                for (int k = 0; k < NA_MAX_CLASSES; ++k) { pe[k] = (k < NC) ? __expf(lg[k] - mxl) : 0.f; den += pe[k]; }
#pragma unroll
                for (int k = 0; k < NA_MAX_CLASSES; ++k)
                    if (k < NC) {
                        logits[b * NC + k] = lg[k];
                        if (probs) probs[b * NC + k] = pe[k] / den;
                    }
            }
            }
            }
        }
        __syncthreads();       // tile done: every MMA has completed (layer-1 epilogue saw the last d1_full)
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kTmaWarp) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
    }
}

// Kernel selection (na_set_tuning("tc_infer_hs", v)): 3 = v2, the software-pipelined kernel of na_decoder_tc2.cu
// (default); 1 | 2 = the v1 kernel above with that many epilogue warps per quarter and layer (kept for A/B timing).
int g_infer_hs = 3;
void set_infer_hs(int hs) { g_infer_hs = (hs >= 1 && hs <= 3) ? hs : 3; }

// na_decoder_tc2.cu
int launch_pack_v2(const float*, const float*, const float*, const float*, const float*, const float*, const float*, const float*,
                   void*, cudaStream_t);
int launch_infer_v2(const void*, const unsigned char*, const float*, const float*, const float*, const float*, const float*,
                    const float*, const float*, const float*, float*, float*, int, int64_t, int64_t, int, int, cudaStream_t,
                    const float*, float*, float*, float*);
constexpr int64_t kPackedV1Bytes = (int64_t)(kK0Chunks + kK1Chunks) * kBChunk;

}  // namespace tc
}  // namespace na

extern "C" int64_t na_decoder_packed_bf16_bytes(void) {
    return 2 * na::tc::kPackedV1Bytes;      // [v1 section (training kernels, v1 inference) | v2 section (pre-scaled)]
}

extern "C" int na_decoder_pack_bf16(const float* w_ih0, const float* w_hh0, const float* b_ih0, const float* b_hh0,
                                    const float* w_ih1, const float* w_hh1, const float* b_ih1, const float* b_hh1,
                                    void* packed, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE_PTR(w_ih0); NA_REQUIRE_PTR(w_hh0); NA_REQUIRE_PTR(b_ih0); NA_REQUIRE_PTR(b_hh0);
    NA_REQUIRE_PTR(w_ih1); NA_REQUIRE_PTR(w_hh1); NA_REQUIRE_PTR(b_ih1); NA_REQUIRE_PTR(b_hh1);
    NA_REQUIRE_PTR(packed);
    tc::pack_decoder_bf16_kernel<<<64, 256, 0, as_stream(stream)>>>(w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1,
                                                                    reinterpret_cast<__nv_bfloat16*>(packed));
    count_launch();
    if (int rc = check_launch("na_decoder_pack_bf16")) return rc;
    return tc::launch_pack_v2(w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1,
                              reinterpret_cast<unsigned char*>(packed) + tc::kPackedV1Bytes, as_stream(stream));
}

extern "C" int na_decoder_infer_bf16_ex(const void* x_bf16_tmp, const void* packed, const float* attn_w,
                                        const float* attn_b, const float* ln_w, const float* ln_b, const float* fc0_w,
                                        const float* fc0_b, const float* fc3_w, const float* fc3_b, float* logits,
                                        float* probs, float* scores_tm, float* pooled, float* embedding, int64_t T, int64_t B,
                                        int64_t Bp, int64_t NC, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(T >= 1 && T < (1 << 20) && B >= 1 && Bp >= B && Bp % tc::kRows == 0, NA_EINVAL,
               "na_decoder_infer_bf16: bad shape T=%lld B=%lld Bp=%lld (Bp must be a multiple of %d)", (long long)T,
               (long long)B, (long long)Bp, tc::kRows);
    NA_REQUIRE(NC >= 1 && NC <= NA_MAX_CLASSES, NA_EUNSUPPORTED, "na_decoder_infer_bf16: num_classes=%lld", (long long)NC);
    NA_REQUIRE_PTR(x_bf16_tmp); NA_REQUIRE_PTR(packed); NA_REQUIRE_PTR(logits);
    NA_OPTIONAL_PTR(probs);
    NA_OPTIONAL_PTR(scores_tm); NA_OPTIONAL_PTR(pooled); NA_OPTIONAL_PTR(embedding);
    NA_REQUIRE(attn_w && attn_b && ln_w && ln_b && fc0_w && fc0_b && fc3_w && fc3_b, NA_EINVAL,
               "na_decoder_infer_bf16: null parameter pointer");
    NA_REQUIRE(tc::g_infer_hs == 3 || !(scores_tm || pooled || embedding), NA_EUNSUPPORTED,
               "na_decoder_infer_bf16_ex: the v1 kernel (tc_infer_hs = %d) does not write intermediates", tc::g_infer_hs);
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    const int hs = tc::g_infer_hs;
    if (hs == 3)
        return tc::launch_infer_v2(x_bf16_tmp, reinterpret_cast<const unsigned char*>(packed) + tc::kPackedV1Bytes, attn_w, attn_b,
                                   ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, (int)T, B, Bp, (int)NC, sms,
                                   as_stream(stream), nullptr, scores_tm, pooled, embedding);
    const size_t smem = sizeof(tc::Smem) + 1024;
    cudaError_t e = hs == 2 ? cudaFuncSetAttribute(tc::decoder_infer_bf16_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                            : cudaFuncSetAttribute(tc::decoder_infer_bf16_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "na_decoder_infer_bf16: shared memory opt-in failed (%s)", cudaGetErrorString(e));
    const int nquarters = (int)((B + 31) / 32);            // padding quarters beyond B are never scheduled
    const int ntiles = (nquarters + 3) / 4;
    const int grid = ntiles < sms ? ntiles : sms;
    if (hs == 2)
        tc::decoder_infer_bf16_kernel<2><<<grid, 18 * 32, smem, as_stream(stream)>>>(
            reinterpret_cast<const __nv_bfloat16*>(x_bf16_tmp), reinterpret_cast<const unsigned char*>(packed), attn_w, attn_b,
            ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, (int)T, B, Bp, (int)NC, nquarters);
    else
        tc::decoder_infer_bf16_kernel<1><<<grid, 10 * 32, smem, as_stream(stream)>>>(
            reinterpret_cast<const __nv_bfloat16*>(x_bf16_tmp), reinterpret_cast<const unsigned char*>(packed), attn_w, attn_b,
            ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, (int)T, B, Bp, (int)NC, nquarters);
    count_launch();
    return check_launch("na_decoder_infer_bf16");
}

extern "C" int na_decoder_infer_bf16(const void* x_bf16_tmp, const void* packed, const float* attn_w,
                                     const float* attn_b, const float* ln_w, const float* ln_b, const float* fc0_w,
                                     const float* fc0_b, const float* fc3_w, const float* fc3_b, float* logits,
                                     float* probs, int64_t T, int64_t B, int64_t Bp, int64_t NC, na_stream_t stream) {
    return na_decoder_infer_bf16_ex(x_bf16_tmp, packed, attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs,
                                    nullptr, nullptr, nullptr, T, B, Bp, NC, stream);
}

// The same forward straight from the caller's batch-first fp32 windows x [B][T][8] (lstm_eeg_model.py:32: `forward(x)`):
// the fp32 -> fp16 time-major pack of na_window_zscore is fused into the kernel's producer warp.
extern "C" int na_decoder_infer_bf16_x32_ex(const float* x, const void* packed, const float* attn_w, const float* attn_b,
                                            const float* ln_w, const float* ln_b, const float* fc0_w, const float* fc0_b,
                                            const float* fc3_w, const float* fc3_b, float* logits, float* probs,
                                            float* scores_tm, float* pooled, float* embedding, int64_t T, int64_t B, int64_t NC,
                                            na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(T >= 1 && T < (1 << 20) && B >= 1, NA_EINVAL, "na_decoder_infer_bf16_x32: bad shape T=%lld B=%lld", (long long)T, (long long)B);
    NA_REQUIRE(NC >= 1 && NC <= NA_MAX_CLASSES, NA_EUNSUPPORTED, "na_decoder_infer_bf16_x32: num_classes=%lld", (long long)NC);
    NA_REQUIRE_PTR(x); NA_REQUIRE_PTR(packed); NA_REQUIRE_PTR(logits);
    NA_OPTIONAL_PTR(probs);
    NA_OPTIONAL_PTR(scores_tm); NA_OPTIONAL_PTR(pooled); NA_OPTIONAL_PTR(embedding);
    NA_REQUIRE(attn_w && attn_b && ln_w && ln_b && fc0_w && fc0_b && fc3_w && fc3_b, NA_EINVAL,
               "na_decoder_infer_bf16_x32: null parameter pointer");
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return tc::launch_infer_v2(nullptr, reinterpret_cast<const unsigned char*>(packed) + tc::kPackedV1Bytes, attn_w, attn_b, ln_w, ln_b,
                               fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, (int)T, B, 0, (int)NC, sms, as_stream(stream), x,
                               scores_tm, pooled, embedding);
}

extern "C" int na_decoder_infer_bf16_x32(const float* x, const void* packed, const float* attn_w, const float* attn_b,
                                         const float* ln_w, const float* ln_b, const float* fc0_w, const float* fc0_b,
                                         const float* fc3_w, const float* fc3_b, float* logits, float* probs, int64_t T,
                                         int64_t B, int64_t NC, na_stream_t stream) {
    return na_decoder_infer_bf16_x32_ex(x, packed, attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, nullptr,
                                        nullptr, nullptr, T, B, NC, stream);
}
