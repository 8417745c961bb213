// Tensor-core tier, inference kernel v2: software-pipelined epilogue.
//
// Measured on B200 (scripts/time_tiles.py): a tile step of the v1 kernel (na_decoder_tc.cu) costs the same
// 2.67 us whether one or four TMEM lane quarters are active, i.e. the bound is the MUFU pipe of ONE SM
// sub-partition (a warp can only read the TMEM lanes of its own quarter, so the 32 windows of a quarter are
// always processed on one scheduler: 32 x 48 units x 2 layers x 5 tanh / 4 lanes per clock = 3,840 cycles),
// and v1 leaves that pipe idle ~26 % of the step: its layer-0 and layer-1 epilogue warps finish together,
// then both wait for the two MMAs (commit -> mbarrier -> tcgen05.ld round trips).
//
// v2 removes the bubble by construction.  Each epilogue warp owns (quarter q, unit group g: 16 units) of BOTH
// layers and alternates   layer-0 step t  ->  layer-1 step t-1  ->  layer-0 step t+1 ...
// The MMA of a layer is issued when that layer's epilogue phase ends and has the whole other phase
// (~1,900 cycles of MUFU work) to complete, so a warp never waits for the tensor pipe in steady state.
//   * 12 epilogue warps (4 quarters x 3 unit groups), warp 12 = MMA issuer, warp 13 = TMA producer + TMEM
//     allocator: 448 threads, 1 CTA / SM, persistent over 128-window tiles.
//   * No per-step cross-warp exchange: the attention score s_t = w_a.h1_t + b_a (lstm_eeg_model.py:35) is
//     computed BY THE TENSOR CORE as two extra accumulator columns of the next layer-1 MMA (h1_t is that
//     MMA's recurrent A operand anyway): B1 has N = 208 rows, row 192 = fp16(w_a) (+ b_a on the ones
//     column), row 193 = the fp16 rounding residual of w_a.  The online-softmax pooling of step t therefore
//     runs one step late, on the h1_t the thread kept in registers; one small N = 16 "flush" MMA after the
//     last step delivers s_{T-1}.
//   * Fewer CUDA-core instructions per cell: the 0.5 of sigmoid(x) = 0.5 tanh(x/2) + 0.5 is folded into the
//     packed weights (exact power-of-two scaling of the i, f, o rows), and the hidden state is carried as
//     H = 2h (the 0.5 folded into every weight column that multiplies h):
//         w = fma(Tf, c, c);  u = fma(Ti, Tg, Tg);  c = 0.5 (w + u);  H = fma(To, tanh c, tanh c)
//     5 MUFU + 5 FMA-pipe ops per cell.
//   * h_{-1} = 0 is handled by NOT issuing the recurrent MMAs of the first step (no buffer zeroing).
//   * Row replication for short tiles (template R): a tile step costs the same MUFU time whether a lane
//     quarter holds 32 windows or 1, so a remainder of <= 64 (<= 32) windows is laid out as R = 2 (4) copies
//     of the same rows (TMA loads x R times, epilogue threads store H to every copy) and every copy's warps
//     take a different 1/R of the hidden units: the tile then costs ~1/R of the MUFU work, i.e. the chain
//     latency (~0.35 of a full step) instead of a full step.  Small batches are spread over all SMs this way.
//     Gate columns are permuted in granules of 4 units, n = (j/4)*16 + gate*4 + j%4, so that 16 / 32
//     accumulator columns hold i,f,g,o of 4 / 8 units.
//   * Fused input (x32 != NULL, na_decoder_infer_bf16_x32): the producer warp reads the caller's batch-first fp32
//     [B][T][8] windows itself -- 32 B per window and step, staged three steps ahead by cp.async -- converts them to
//     fp16 and writes the x chunk, so the separate fp32 -> fp16 time-major pack (K1) and its intermediate are gone.
//   * One tcgen05.commit per layer and step: the x ring is released by a plain mbarrier.arrive of an epilogue thread
//     that has seen d0_full, and the h0 buffer written at step n is ordered after the layer-1 MMA of step n-2 by the
//     d1_full the writing thread already waited for.
#include "na_tc_common.cuh"

namespace na {
namespace tc {

constexpr int kV2XStages = 4;
constexpr int kV2K0Chunks = 8;                 // layer 0: x | ones | h0 x6
constexpr int kV2K1Chunks = 14;                // layer 1: h0 x6 | h1 x6 | ones | zero
constexpr int kN1 = 208;                       // layer-1 accumulator columns: 192 gates + 16 (score hi, lo, pad)
constexpr int kB1Chunk = kN1 * 16;             // bytes of one layer-1 B K-chunk in shared memory
constexpr int kV2Threads = 14 * 32;
constexpr int kV2Fc = NA_FC_HIDDEN;
constexpr uint32_t kIdescL1 = make_idesc(kN1, kFmtVal, kFmtVal);
constexpr uint32_t kIdescFlush = make_idesc(16, kFmtVal, kFmtVal);

struct HeadSmem2 {
    float lnw[kH], lnb[kH];
    float w0[kV2Fc * kH];
    float b0[kV2Fc];
    float w3[NA_MAX_CLASSES * kV2Fc];
    float b3[NA_MAX_CLASSES];
};

struct Smem2 {
    alignas(128) unsigned char b0[kV2K0Chunks * kBChunk];          // 24,576
    alignas(128) unsigned char b1[kV2K1Chunks * kB1Chunk];         // 46,592
    alignas(128) unsigned char x[kV2XStages][2 * kAChunk];         // [x chunk | ones chunk] per stage
    alignas(128) unsigned char h0[2][6 * kAChunk];                 // double-buffered H0_t (= 2 h0_t, fp16)
    alignas(128) unsigned char h1[6 * kAChunk];
    alignas(128) unsigned char onez[2 * kAChunk];                  // [ones | zeros]
    HeadSmem2 head;
    float zx[kRows][kH + 1];                                       // pooled vector exchange, once per tile
    alignas(16) float xf32[kV2XStages][kRows][8];                  // fused input: fp32 rows staged by cp.async
    alignas(8) uint64_t x_full[kV2XStages], x_empty[kV2XStages];
    uint64_t d0_full, d1_full, h0_ready[2], h1_ready;
    uint32_t tmem_base;
};

// ---- weight packing (v2 section of `packed`) ---------------------------------------------------------
// B0 [8 chunks][192][8] and B1 [14 chunks][192][8] fp16, row n = (j/4)*16 + gate*4 + j%4, pre-scaled:
// rows of the i, f, o gates by 0.5 (sigmoid via tanh), columns that multiply a hidden state by 0.5 (H = 2h).
__global__ void pack_decoder_v2_kernel(const float* __restrict__ w_ih0, const float* __restrict__ w_hh0,
                                       const float* __restrict__ b_ih0, const float* __restrict__ b_hh0,
                                       const float* __restrict__ w_ih1, const float* __restrict__ w_hh1,
                                       const float* __restrict__ b_ih1, const float* __restrict__ b_hh1,
                                       uint16_t* __restrict__ out) {
    const int total0 = kV2K0Chunks * 8 * kN, total1 = kV2K1Chunks * 8 * kN;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total0 + total1; idx += gridDim.x * blockDim.x) {
        const bool l1 = idx >= total0;
        const int e = l1 ? idx - total0 : idx;
        const int k = (e / (kN * 8)) * 8 + (e % 8);       // K index
        const int n = (e / 8) % kN;                       // permuted gate column
        const int j = (n / 16) * 4 + (n % 4), q = (n % 16) / 4;
        const int col = q * kH + j;                       // row of the torch weight tensors
        const float gs = (q == 2) ? 1.0f : 0.5f;          // gate pre-scale
        const float hs = 0.5f * gs;                       // ... times the H = 2h column scale
        float v = 0.f;
        if (!l1) {
            const float b = gs * (b_ih0[col] + b_hh0[col]);
            const float bh = val16_to_float(val16(b));
            if (k < 8) v = gs * kF16InScaleInv * w_ih0[col * 8 + k];      // x is stored as x / 16
            else if (k == 8) v = bh;
            else if (k == 9) v = b - bh;
            else if (k >= 16) v = hs * w_hh0[col * kH + (k - 16)];
        } else {
            const float b = gs * (b_ih1[col] + b_hh1[col]);
            const float bh = val16_to_float(val16(b));
            if (k < 48) v = hs * w_ih1[col * kH + k];
            else if (k < 96) v = hs * w_hh1[col * kH + (k - 48)];
            else if (k == 96) v = bh;
            else if (k == 97) v = b - bh;
        }
        out[idx] = val16(v);
    }
}

__device__ __forceinline__ void tmem_ld2(uint32_t taddr, uint32_t (&v)[2]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(v[0]), "=r"(v[1]) : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_shared_v2(void* p, uint32_t a, uint32_t b) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(smem_u32(p)), "r"(a), "r"(b) : "memory");
}

// tanh on the FMA pipe.  The MUFU pipe (16 results / clk / SM) bounds this kernel at 5 tanh.approx per cell while the FMA
// pipe is 15 % busy and two thirds of the issue slots are free (ncu, profiles/r1_tc2_infer_ncu_full.csv), so one of the five
// is evaluated as the [7/6] Pade approximant of tanh (Lambert's continued fraction)
//     tanh y ~ y (135135 + 17325 y^2 + 378 y^4 + y^6) / (135135 + 62370 y^2 + 3150 y^4 + 28 y^6),   |y| clamped to 5,
// absolute error < 1.1e-4 (tanh.approx: 5e-4); the reciprocal is an exponent-trick seed + one cubic + one quadratic
// Newton step (4e-6).  17 FMA-pipe / ALU instructions for one MUFU result.
// MEASURED (B200, round 2, scripts/time_offload.py): full round of 18,944 windows 1.575 ms without, 1.612 ms with the
// offload; short (row-replicated) round 0.701 -> 0.668 ms; 40,960 windows 3.79 -> 3.88 ms.  The xu pipe is 90 % busy but the
// three epilogue warps of a sub-partition are bound by their own dependent chains, so trading one MUFU for 17 dependent
// FMA-pipe instructions does not pay on full tiles.  Default: off (knob "tc_infer_tanh_fma").
__device__ __forceinline__ float tanh_fma(float y) {
    const float yc = fminf(fmaxf(y, -5.0f), 5.0f);
    const float y2 = yc * yc;
    const float num = yc * fmaf(fmaf(y2 + 378.0f, y2, 17325.0f), y2, 135135.0f);
    const float den = fmaf(fmaf(fmaf(28.0f, y2, 3150.0f), y2, 62370.0f), y2, 135135.0f);
    float r = __int_as_float(0x7EF311C7 - __float_as_int(den));
    float e = fmaf(-den, r, 1.0f);
    r = fmaf(r, fmaf(e, e, e), r);
    e = fmaf(-den, r, 1.0f);
    r = fmaf(r, e, r);
    return num * r;
}

// One cell update for the 4 units of a granule; v = [i x4 | f x4 | g x4 | o x4] pre-activations (i, f, o already
// halved by the packed weights).  Returns H = 2h packed as 2 x fp16x2.  NT = activations per cell on the FMA pipe (0 / 1).
template <int NT>
__device__ __forceinline__ void cell_granule(const uint32_t* v, float* c, uint32_t* hp) {
    float h[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float ti = tanh_apx(__uint_as_float(v[u]));
        const float tf = tanh_apx(__uint_as_float(v[4 + u]));
        const float tg = tanh_apx(__uint_as_float(v[8 + u]));
        const float to = NT >= 1 ? tanh_fma(__uint_as_float(v[12 + u])) : tanh_apx(__uint_as_float(v[12 + u]));
        const float w = fmaf(tf, c[u], c[u]);
        const float uu = fmaf(ti, tg, tg);
        c[u] = 0.5f * (w + uu);
        const float tcell = tanh_apx(c[u]);
        h[u] = fmaf(to, tcell, tcell);
    }
    hp[0] = pack_val(h[0], h[1]);
    hp[1] = pack_val(h[2], h[3]);
}

// Epilogue of one tile for one warp: both layers of (lane quarter q, unit group g).  R = row replication:
// the tile holds 128 / R distinct windows; copy rp = q / (4 / R) of source quarter qs = q % (4 / R) takes
// granules [4 g + rp * (4 / R), + 4 / R) of the 12 four-unit granules.
// kEx: also store the attention scores (time-major [T][B]) and the pooled vector / LayerNorm output ([B][48]) of every
// window b < B, in the reference's scale (h, not H = 2h): the scores and the LayerNorm output by the first row copy of
// the g == 0 warps (the one that runs the head), the pooled vector by every thread for the units it pooled.
template <int R, int NT, bool kEx>
__device__ __forceinline__ void epilogue_tile(Smem2& S, const int q, const int g, const int lane, const int nq, const int T,
                                              const int n0, uint32_t& k1, const uint32_t tmem_d0, const uint32_t tmem_d1,
                                              const int64_t b0, const int64_t B, const int NC, float* __restrict__ logits,
                                              float* __restrict__ probs, float* __restrict__ scores_tm,
                                              float* __restrict__ pooled, float* __restrict__ embedding) {
    constexpr int kQ = 4 / R;                      // distinct source quarters = granules per warp
    constexpr int kSlots = 4 / R, kU = 4 * kSlots; // granules / units owned by this thread
    const int qs = q % kQ, rp = q / kQ;
    const int wrow = qs * 32 + lane;               // window row of the tile (first copy)
    const bool ex_writer = kEx && g == 0 && rp == 0 && b0 + wrow < B;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const int gr0 = 4 * g + rp * kSlots;           // first granule
    if (qs >= nq) {                                // idle quarter: keep the barrier protocol only
        for (int t = 0; t <= T; ++t) {
            const int n = n0 + t;
            if (t < T) {
                mbar_wait(&S.d0_full, n & 1);
                if (q == 0 && g == 0 && lane == 0) mbar_arrive(&S.x_empty[n % kV2XStages]);
                mbar_arrive(&S.h0_ready[n & 1]);
            }
            if (t >= 1) { mbar_wait(&S.d1_full, k1 & 1); ++k1; mbar_arrive(&S.h1_ready); }
        }
        mbar_wait(&S.d1_full, k1 & 1); ++k1;
        return;
    }
    float c0[kU], c1[kU], z[kU];
#pragma unroll
    for (int j = 0; j < kU; ++j) { c0[j] = 0.f; c1[j] = 0.f; z[j] = 0.f; }
    uint32_t hprev[2 * kSlots];
#pragma unroll
    for (int j = 0; j < 2 * kSlots; ++j) hprev[j] = 0u;
    float mx = -INFINITY, l = 0.f;
    auto pool = [&](float score) {                 // online softmax over time (lstm_eeg_model.py:35-37), lazy rescale
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
        for (int u = 0; u < 2 * kSlots; ++u) {
            z[2 * u] = fmaf(e, val_lo(hprev[u]), z[2 * u]);
            z[2 * u + 1] = fmaf(e, val_hi(hprev[u]), z[2 * u + 1]);
        }
    };
    // gates of this thread's granules -> cell update -> H (fp16) stored to every row copy of the A operand `buf`
    auto layer_phase = [&](const uint32_t tmem_d, float* c, unsigned char* buf, uint32_t* hb) {
        if constexpr (R == 4) {
            uint32_t v[16];
            tmem_ld16(tmem_d + lane_base + gr0 * 16, v);
            cell_granule<NT>(v, c, hb);
            unsigned char* dst = buf + (gr0 >> 1) * kAChunk + wrow * 16 + (gr0 & 1) * 8;
#pragma unroll
            for (int rep = 0; rep < 4; ++rep) st_shared_v2(dst + rep * 32 * 16, hb[0], hb[1]);
        } else {
#pragma unroll
            for (int pr = 0; pr < kSlots / 2; ++pr) {       // pairs of granules = one 8-unit K chunk
                uint32_t v[32];
                tmem_ld32(tmem_d + lane_base + (gr0 + 2 * pr) * 16, v);
                cell_granule<NT>(v, c + pr * 8, hb + pr * 4);
                cell_granule<NT>(v + 16, c + pr * 8 + 4, hb + pr * 4 + 2);
                unsigned char* dst = buf + ((gr0 >> 1) + pr) * kAChunk + wrow * 16;
#pragma unroll
                for (int rep = 0; rep < R; ++rep)
                    st_shared_v4(dst + rep * (kRows / R) * 16, hb[pr * 4], hb[pr * 4 + 1], hb[pr * 4 + 2], hb[pr * 4 + 3]);
            }
        }
    };
    for (int t = 0; t <= T; ++t) {
        const int n = n0 + t;
        if (t < T) {                               // ---- layer 0, step t
            // d0_full: the layer-0 MMA of step n has completed -> its x stage is free (one thread tells the TMA producer;
            // a plain mbarrier.arrive instead of a second tcgen05.commit per step).  The h0 buffer written below was last
            // read by the layer-1 MMA of step n-2, whose d1_full this thread waited for in the previous iteration.
            mbar_wait(&S.d0_full, n & 1);
            if (q == 0 && g == 0 && lane == 0) mbar_arrive(&S.x_empty[n % kV2XStages]);
            tc_fence_after();
            uint32_t hb[2 * kSlots];
            layer_phase(tmem_d0, c0, S.h0[n & 1], hb);
            tc_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(&S.h0_ready[n & 1]);
        }
        if (t >= 1) {                              // ---- layer 1, step t-1 (+ pooling of step t-2)
            mbar_wait(&S.d1_full, k1 & 1); ++k1;
            tc_fence_after();
            uint32_t sc2[2];
            tmem_ld2(tmem_d1 + lane_base + kN, sc2);
            uint32_t hb[2 * kSlots];
            layer_phase(tmem_d1, c1, S.h1, hb);
            tc_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(&S.h1_ready);
            if (t >= 2) pool(__uint_as_float(sc2[0]) + __uint_as_float(sc2[1]));
            // the score columns hold w_a / 2 . H1 + b_a = w_a . h1 + b_a: no rescaling
            if constexpr (kEx)
                if (t >= 2 && ex_writer && scores_tm)
                    scores_tm[(int64_t)(t - 2) * B + b0 + wrow] = __uint_as_float(sc2[0]) + __uint_as_float(sc2[1]);
#pragma unroll
            for (int u = 0; u < 2 * kSlots; ++u) hprev[u] = hb[u];
        }
    }
    {                                              // flush: score of the last step
        mbar_wait(&S.d1_full, k1 & 1); ++k1;
        tc_fence_after();
        uint32_t sc2[2];
        tmem_ld2(tmem_d1 + lane_base + kN, sc2);
        tc_fence_before();
        pool(__uint_as_float(sc2[0]) + __uint_as_float(sc2[1]));
        if constexpr (kEx)
            if (ex_writer && scores_tm) scores_tm[(int64_t)(T - 1) * B + b0 + wrow] = __uint_as_float(sc2[0]) + __uint_as_float(sc2[1]);
    }
    // ---- head for this window: LN -> fc0 -> RReLU(eval) -> fc3 -> softmax ----------------------
#pragma unroll
    for (int j = 0; j < kU; ++j) S.zx[wrow][gr0 * 4 + j] = z[j];
    if constexpr (kEx)
        // every copy stores the units it pooled, from its own registers: a further use of the head's products would
        // change which of them the assembler contracts into FMAs, and the logits would no longer be the default's
        if (pooled && b0 + wrow < B) {
            float zp[kU];
            const float inv = 0.5f / l;            // z accumulated H = 2h
#pragma unroll
            for (int j = 0; j < kU; ++j) zp[j] = z[j] * inv;
            store_row<kU>(pooled + (b0 + wrow) * kH + gr0 * 4, zp);
        }
    named_bar_sync(1 + qs, 96 * R);                // the 3 R warps that share source quarter qs
    if (g == 0 && rp == 0) {
        const int64_t b = b0 + wrow;
        float zf[kH];
        const float inv_l = 0.5f / l;              // z accumulated H = 2h
        float mean = 0.f;
#pragma unroll
        for (int j = 0; j < kH; ++j) { zf[j] = S.zx[wrow][j] * inv_l; mean += zf[j]; }
        mean *= (1.0f / kH);
        float var = 0.f;
#pragma unroll
        for (int j = 0; j < kH; ++j) { const float d = zf[j] - mean; var = fmaf(d, d, var); }
        const float rstd = rsqrtf(var * (1.0f / kH) + kLnEps);
#pragma unroll
        for (int j = 0; j < kH; ++j) zf[j] = fmaf((zf[j] - mean) * rstd, S.head.lnw[j], S.head.lnb[j]);
        if constexpr (kEx)
            if (ex_writer && embedding) store_row<kH>(embedding + b * kH, zf);
        float lg[NA_MAX_CLASSES];
#pragma unroll
        for (int k = 0; k < NA_MAX_CLASSES; ++k) lg[k] = (k < NC) ? S.head.b3[k] : -INFINITY;
        for (int o = 0; o < kV2Fc; ++o) {
            float a = S.head.b0[o];
#pragma unroll
            for (int j = 0; j < kH; ++j) a = fmaf(S.head.w0[o * kH + j], zf[j], a);
            a = a >= 0.f ? a : a * kRReluEvalSlope;
#pragma unroll
            for (int k = 0; k < NA_MAX_CLASSES; ++k)
                if (k < NC) lg[k] = fmaf(S.head.w3[k * kV2Fc + o], a, lg[k]);
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

template <int NT, bool kEx = false>
__global__ void __launch_bounds__(kV2Threads, 1)
decoder_infer_v2_kernel(const __nv_bfloat16* __restrict__ x,        // TMP [T][Bp][8] fp16 bits
                        const unsigned char* __restrict__ packed,   // v2 section: B0 | B1 (pack_decoder_v2_kernel)
                        const float* __restrict__ attn_w, const float* __restrict__ attn_b,
                        const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                        const float* __restrict__ fc0_w, const float* __restrict__ fc0_b,
                        const float* __restrict__ fc3_w, const float* __restrict__ fc3_b,
                        float* __restrict__ logits, float* __restrict__ probs,
                        int T, int64_t B, int64_t Bp, int NC, int nquarters, int allow_rep,
                        const float* __restrict__ x32,         // != NULL: the caller's [B][T][8] fp32 windows, read directly (x unused)
                        float* __restrict__ scores_tm,         // kEx: [T][B] scores, [B][48] pooled / LayerNorm output
                        float* __restrict__ pooled, float* __restrict__ embedding) {
    constexpr int kMmaWarp = 12, kTmaWarp = 13;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    Smem2& S = *reinterpret_cast<Smem2*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);      // provably warp-uniform: role branches are uniform control flow

    // ---- one-time setup --------------------------------------------------------------------------
    {
        const uint4* src = reinterpret_cast<const uint4*>(packed);
        uint4* d0 = reinterpret_cast<uint4*>(S.b0);
        constexpr int n0_16 = kV2K0Chunks * kBChunk / 16;
        for (int i = tid; i < n0_16; i += kV2Threads) d0[i] = src[i];
        // layer 1: 192 packed rows per chunk -> 208-row chunks; rows 192..207 = attention score columns
        for (int i = tid; i < kV2K1Chunks * kN; i += kV2Threads) {
            const int ch = i / kN, r = i % kN;
            reinterpret_cast<uint4*>(S.b1 + ch * kB1Chunk)[r] = src[n0_16 + i];
        }
        for (int i = tid; i < kV2K1Chunks * 16; i += kV2Threads) {
            const int ch = i / 16, r = i % 16;
            uint16_t w[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int k = ch * 8 + e;
                float v = 0.f;
                if (r < 2) {
                    float full = 0.f;
                    if (k >= 48 && k < 96) full = 0.5f * attn_w[k - 48];      // multiplies H1 = 2 h1
                    else if (k == 96) full = attn_b[0];
                    const float hi = val16_to_float(val16(full));
                    v = (r == 0) ? hi : full - hi;
                }
                w[e] = val16(v);
            }
            uint4 pk;
            pk.x = w[0] | ((uint32_t)w[1] << 16); pk.y = w[2] | ((uint32_t)w[3] << 16);
            pk.z = w[4] | ((uint32_t)w[5] << 16); pk.w = w[6] | ((uint32_t)w[7] << 16);
            reinterpret_cast<uint4*>(S.b1 + ch * kB1Chunk)[kN + r] = pk;
        }
        const uint4 ones = make_uint4(kValOnes2, 0u, 0u, 0u);     // fp16 {1,1,0,0,0,0,0,0}
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        for (int i = tid; i < kRows; i += kV2Threads) {
#pragma unroll
            for (int s = 0; s < kV2XStages; ++s) reinterpret_cast<uint4*>(S.x[s] + kAChunk)[i] = ones;
            reinterpret_cast<uint4*>(S.onez)[i] = ones;
            reinterpret_cast<uint4*>(S.onez + kAChunk)[i] = zero;
        }
        for (int i = tid; i < kH; i += kV2Threads) { S.head.lnw[i] = ln_w[i]; S.head.lnb[i] = ln_b[i]; }
        for (int i = tid; i < kV2Fc * kH; i += kV2Threads) S.head.w0[i] = fc0_w[i];
        for (int i = tid; i < kV2Fc; i += kV2Threads) S.head.b0[i] = fc0_b[i];
        for (int i = tid; i < NC * kV2Fc; i += kV2Threads) S.head.w3[i] = fc3_w[i];
        for (int i = tid; i < NC; i += kV2Threads) S.head.b3[i] = fc3_b[i];
        if (tid == 0) {
            for (int s = 0; s < kV2XStages; ++s) { mbar_init(&S.x_full[s], 1); mbar_init(&S.x_empty[s], 1); }
            mbar_init(&S.d0_full, 1); mbar_init(&S.d1_full, 1);
            mbar_init(&S.h0_ready[0], 384); mbar_init(&S.h0_ready[1], 384);
            mbar_init(&S.h1_ready, 384);
            fence_mbar_init();
        }
        if (warp == kTmaWarp) tmem_alloc_all(&S.tmem_base);
        tc_fence_before();
        fence_proxy_async_smem();
        __syncthreads();
        tc_fence_after();
    }
    const uint32_t tmem = __shfl_sync(0xffffffffu, S.tmem_base, 0);
    const uint32_t tmem_d0 = tmem, tmem_d1 = tmem + kN;

    // Work split: 32-window quarters, CTA i owns a contiguous range and walks it in tiles of up to 4 quarters; a
    // remainder of 2 quarters runs as one R = 2 tile, a remainder of 1 as an R = 4 tile.
    const int q_begin = (int)(((int64_t)blockIdx.x * nquarters) / gridDim.x);
    const int q_end = (int)(((int64_t)(blockIdx.x + 1) * nquarters) / gridDim.x);
    int n0 = 0;                                            // running layer-0 step index across tiles
    uint32_t k1 = 0;                                       // running d1_full phase index (T + 1 per tile)
    for (int q0 = q_begin; q0 < q_end; n0 += T) {
        const int nq = min(4, q_end - q0);                 // active source quarters of this tile
        const int R = !allow_rep ? 1 : (nq == 1 ? 4 : (nq == 2 ? 2 : 1));
        const uint32_t x_bytes = (uint32_t)nq * 32u * 16u;
        const int64_t b0 = (int64_t)q0 * 32;

        if (warp == kTmaWarp) {
            // ================= producer of x_t ========================================================
            if (x32 != nullptr) {
                // Fused K1: the warp reads the caller's batch-first fp32 windows itself (32 B per window and step,
                // sector-sized; the neighbouring step is served from L2), converts to fp16 and writes the A chunk --
                // no time-major fp16 copy of the input exists.  Loads of step t+1 are in flight while step t is stored.
                // cp.async (LDGSTS) stages the fp32 rows kPre steps ahead in shared memory (no registers held across the
                // DRAM latency), so even a latency-bound short tile (~1 us per step) never waits for its input.
                const int nrows = nq * 32;
                constexpr int kPre = 3;
                auto issue = [&](int t) {                          // fp32 rows of step t -> S.xf32[t % 4]
                    if (t < T) {
#pragma unroll
                        for (int rr = 0; rr < 4; ++rr) {
                            const int row = rr * 32 + lane;
                            const int64_t b = b0 + row;
                            if (row < nrows && b < B) {
                                const float* src = x32 + (b * T + t) * 8;
                                const uint32_t dst = smem_u32(&S.xf32[t % kV2XStages][row][0]);
                                asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
                                asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 16), "l"(src + 4) : "memory");
                            }
                        }
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");      // one (possibly empty) group per step
                };
#pragma unroll
                for (int t = 0; t < kPre; ++t) issue(t);
                for (int t = 0; t < T; ++t) {
                    const int n = n0 + t, s = n % kV2XStages, u = n / kV2XStages;
                    asm volatile("cp.async.wait_group %0;" ::"n"(kPre - 1) : "memory");   // this step's rows have landed
                    mbar_wait(&S.x_empty[s], (u & 1) ^ 1);
#pragma unroll
                    for (int rr = 0; rr < 4; ++rr) {
                        const int row = rr * 32 + lane;
                        if (row < nrows) {
                            float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
                            if (b0 + row < B) {
                                v0 = *reinterpret_cast<const float4*>(&S.xf32[t % kV2XStages][row][0]);
                                v1 = *reinterpret_cast<const float4*>(&S.xf32[t % kV2XStages][row][4]);
                            }
                            const uint32_t p0 = pack_val(kF16InScale * v0.x, kF16InScale * v0.y), p1 = pack_val(kF16InScale * v0.z, kF16InScale * v0.w);
                            const uint32_t p2 = pack_val(kF16InScale * v1.x, kF16InScale * v1.y), p3 = pack_val(kF16InScale * v1.z, kF16InScale * v1.w);
                            for (int rep = 0; rep < R; ++rep) st_shared_v4(S.x[s] + (rep * (kRows / R) + row) * 16, p0, p1, p2, p3);
                        }
                    }
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&S.x_full[s]);
                    issue(t + kPre);                               // re-uses the staging slot read two steps ago (t + 3 = t - 1 mod 4)
                }
                asm volatile("cp.async.wait_group 0;" ::: "memory");
            } else if (lane == 0) {
                for (int t = 0; t < T; ++t) {
                    const int n = n0 + t, s = n % kV2XStages, u = n / kV2XStages;
                    mbar_wait(&S.x_empty[s], (u & 1) ^ 1);
                    mbar_arrive_expect_tx(&S.x_full[s], x_bytes * (uint32_t)R);
                    const __nv_bfloat16* src = x + ((int64_t)t * Bp + b0) * 8;
                    for (int rep = 0; rep < R; ++rep) bulk_load(S.x[s] + rep * (kRows / R) * 16, src, x_bytes, &S.x_full[s]);
                }
            }
        } else if (warp == kMmaWarp) {
            // ================= MMA issuer ============================================================
            {
                // whole warp, warp-uniform control flow; one elected lane issues (descriptors stay on the uniform datapath)
                const bool leader = elect_one();
                const uint64_t d_b0 = umma_desc(smem_u32(S.b0), kBChunk, 128), d_b1 = umma_desc(smem_u32(S.b1), kB1Chunk, 128);
                const uint64_t d_x0 = umma_desc(smem_u32(S.x[0]), kAChunk, 128);
                const uint64_t d_h0[2] = {umma_desc(smem_u32(S.h0[0]), kAChunk, 128), umma_desc(smem_u32(S.h0[1]), kAChunk, 128)};
                const uint64_t d_h1 = umma_desc(smem_u32(S.h1), kAChunk, 128), d_onez = umma_desc(smem_u32(S.onez), kAChunk, 128);
                for (int t = 0; t <= T; ++t) {
                    const int n = n0 + t;
                    if (t >= 1) {                                  // H0_{t-1} written, D0 drained
                        mbar_wait(&S.h0_ready[(n - 1) & 1], ((n - 1) >> 1) & 1);
                        tc_fence_after();
                    }
                    if (t < T) {                                   // layer 0, step t
                        const int s = n % kV2XStages, u = n / kV2XStages;
                        mbar_wait(&S.x_full[s], u & 1);
                        tc_fence_after();
                        if (leader) umma_bf16(tmem_d0, desc_adv(d_x0, s * 2 * kAChunk), d_b0, 0u);
                        if (t >= 1) {
                            const uint64_t hprev = d_h0[(n - 1) & 1];
#pragma unroll
                            for (int i = 0; i < 3; ++i)
                                if (leader) umma_bf16(tmem_d0, desc_adv(hprev, 2 * i * kAChunk), desc_adv(d_b0, (2 + 2 * i) * kBChunk), 1u);
                        }
                        if (leader) umma_commit(&S.d0_full);
                    }
                    if (t >= 1) {                                  // layer 1, step m = t - 1
                        const int m = n - 1;
                        if (t >= 2) {                              // H1_{m-1} written, D1 drained
                            mbar_wait(&S.h1_ready, (m - 1) & 1);
                            tc_fence_after();
                        }
                        const uint64_t hin = d_h0[m & 1];
#pragma unroll
                        for (int i = 0; i < 3; ++i)
                            if (leader) umma_bf16_i(tmem_d1, desc_adv(hin, 2 * i * kAChunk), desc_adv(d_b1, 2 * i * kB1Chunk), kIdescL1, i == 0 ? 0u : 1u);
                        if (t >= 2) {
#pragma unroll
                            for (int i = 0; i < 3; ++i)
                                if (leader) umma_bf16_i(tmem_d1, desc_adv(d_h1, 2 * i * kAChunk), desc_adv(d_b1, (6 + 2 * i) * kB1Chunk), kIdescL1, 1u);
                        }
                        if (leader) umma_bf16_i(tmem_d1, d_onez, desc_adv(d_b1, 12 * kB1Chunk), kIdescL1, 1u);
                        if (leader) umma_commit(&S.d1_full);
                    }
                }
                // flush: s_{T-1} = w_a . h1_{T-1} + b_a into the 16 score columns only
                {
                    const int m = n0 + T - 1;
                    mbar_wait(&S.h1_ready, m & 1);
                    tc_fence_after();
                    const uint64_t d_b1s = desc_adv(d_b1, kN * 16);          // rows 192..207 of every chunk
#pragma unroll
                    for (int i = 0; i < 3; ++i)
                        if (leader) umma_bf16_i(tmem_d1 + kN, desc_adv(d_h1, 2 * i * kAChunk), desc_adv(d_b1s, (6 + 2 * i) * kB1Chunk), kIdescFlush, i == 0 ? 0u : 1u);
                    if (leader) umma_bf16_i(tmem_d1 + kN, d_onez, desc_adv(d_b1s, 12 * kB1Chunk), kIdescFlush, 1u);
                    if (leader) umma_commit(&S.d1_full);
                }
            }
        } else {
            // ================= epilogue: both layers of (quarter q, unit group g) ========================
            const int q = warp & 3, g = warp >> 2;
            if (R == 1) epilogue_tile<1, NT, kEx>(S, q, g, lane, nq, T, n0, k1, tmem_d0, tmem_d1, b0, B, NC, logits, probs, scores_tm, pooled, embedding);
            else if (R == 2) epilogue_tile<2, NT, kEx>(S, q, g, lane, nq, T, n0, k1, tmem_d0, tmem_d1, b0, B, NC, logits, probs, scores_tm, pooled, embedding);
            else epilogue_tile<4, NT, kEx>(S, q, g, lane, nq, T, n0, k1, tmem_d0, tmem_d1, b0, B, NC, logits, probs, scores_tm, pooled, embedding);
        }
        __syncthreads();       // tile done: every MMA has completed (the epilogue saw the flush d1_full)
        q0 += nq;
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kTmaWarp) {
        tc_fence_after();
        tmem_free_all(tmem);
    }
}

int g_infer_tanh_fma = 0;  // na_set_tuning("tc_infer_tanh_fma", 0 / 1): activations per cell on the FMA pipe (A/B timing)
void set_infer_tanh_fma(int v) { g_infer_tanh_fma = v ? 1 : 0; }
int g_infer_rep = 1;       // na_set_tuning("tc_infer_rep", 0) disables row replication (A/B timing)
void set_infer_rep(int v) { g_infer_rep = v ? 1 : 0; }

size_t infer_v2_smem_bytes() { return sizeof(Smem2) + 1024; }

int launch_pack_v2(const float* w_ih0, const float* w_hh0, const float* b_ih0, const float* b_hh0, const float* w_ih1,
                   const float* w_hh1, const float* b_ih1, const float* b_hh1, void* out, cudaStream_t stream) {
    pack_decoder_v2_kernel<<<64, 256, 0, stream>>>(w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1,
                                                   reinterpret_cast<uint16_t*>(out));
    count_launch();
    return check_launch("na_decoder_pack_bf16 (v2 section)");
}

int launch_infer_v2(const void* x, const unsigned char* packed_v2, const float* attn_w, const float* attn_b, const float* ln_w,
                    const float* ln_b, const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                    float* logits, float* probs, int T, int64_t B, int64_t Bp, int NC, int sms, cudaStream_t stream,
                    const float* x32, float* scores_tm, float* pooled, float* embedding) {
    const size_t smem = infer_v2_smem_bytes();
    const bool ex = scores_tm || pooled || embedding;
    auto kern = g_infer_tanh_fma ? (ex ? decoder_infer_v2_kernel<1, true> : decoder_infer_v2_kernel<1>)
                                 : (ex ? decoder_infer_v2_kernel<0, true> : decoder_infer_v2_kernel<0>);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "na_decoder_infer_bf16: shared memory opt-in failed (%s)", cudaGetErrorString(e));
    const int nquarters = (int)((B + 31) / 32);            // padding quarters beyond B are never scheduled
    // one CTA per SM; fewer than 4 quarters per CTA run as row-replicated tiles (see epilogue_tile<R>)
    const int grid = nquarters < sms ? nquarters : sms;
    kern<<<grid, kV2Threads, smem, stream>>>(reinterpret_cast<const __nv_bfloat16*>(x), packed_v2, attn_w, attn_b,
                                             ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, T, B, Bp, NC,
                                             nquarters, g_infer_rep, x32, scores_tm, pooled, embedding);
    count_launch();
    return check_launch("na_decoder_infer_bf16 (v2)");
}

}  // namespace tc
}  // namespace na

// ---- training forward, generation 2 (shares this translation unit's helpers) ------------------------------------
namespace na {
namespace tc {
__device__ __forceinline__ void st_global_v4f(float* p, float a, float b, float c, float d) {
    *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
// TCL32 (see na_train_tc.cu): fp32 tile-chunk layout [T][Bp/128][12][128][4]
__device__ __forceinline__ int64_t tcl32_off(int t, int ntiles, int tile, int chunk, int row) {
    return (((((int64_t)t * ntiles + tile) * 12 + chunk) * kRows) + row) * 4;
}
}  // namespace tc
}  // namespace na
#include "na_train_fwd2.cuh"
