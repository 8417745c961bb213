// Exact tier on the tensor cores: the whole eval forward x -> logits/probs at fp32 accuracy (1e-5 contract) with
// tcgen05.mma, by SPLITTING every 32-bit operand into two fp16 halves.
//
// An fp32 value v (bounded: |h| < 1, trained weights, EEG samples of a few tens) is v = hi + lo + O(2^-22 |v|) with
// hi = fp16(v), lo = fp16(v - hi).  A product a.w is then a_hi w_hi + a_hi w_lo + a_lo w_hi + O(2^-22): three fp16 MMAs
// with fp32 accumulation in TMEM reproduce the fp32 dot product to ~2e-7 relative (numpy simulation of the whole
// 625-step decoder on the repo's windows: 2.3e-7 of max|logit| against 1.3e-7 for plain fp32; measured on B200: see
// tests/test_gpu_parity.py).  The exact FFMA kernels (na_lstm_h48.cu) reach 0.56 of the CUDA-core peak = 1.05 M
// windows/s; here the tensor pipe does the 3x contraction in ~3,100 cycles per 128-window step and the bound becomes
// the transcendental pipe again: accurate activations cost 2 MUFU each (ex2.approx + rcp.approx, ~2e-7 absolute -- the
// tanh.approx of the 16-bit tier is 5e-4 and cannot be used), 10 per cell update -> 7,680 MUFU cycles per step.
//
// Structure = decoder_infer_v2_kernel (na_decoder_tc2.cu): 12 epilogue warps own both layers of (lane quarter, 16-unit
// group) and alternate layer-0 step t / layer-1 step t-1; one elected MMA lane; the producer warp reads the caller's
// fp32 [B][T][8] windows directly and writes x_hi / x_lo; the attention score is an extra accumulator column of the
// next layer-1 MMA (3-term split as well); cell state, pooling, LayerNorm, MLP and softmax in fp32.
//   A chunks ([128 rows][8] fp16 = 2 KB):  x stage = [x_hi | ones | x_lo];  h0[2], h1 = 6 hi chunks + 6 lo chunks
//   B0 (15 chunks x 192 rows): Wih_hi | bias(hi,lo) | Whh_hi x6 | Wih_lo | Whh_lo x6
//   B1 (25 chunks x 208 rows): Wih_hi x6 | Whh_hi x6 | bias(hi,lo) | Wih_lo x6 | Whh_lo x6;  rows 192.. = attention
//   K16 MMAs pair two chunks through the descriptor's leading-byte-offset, so (x_lo | zeros), (x_hi | zeros) and
//   (ones | zeros) pairs need no copies.  220 KB of shared memory; head parameters are read from global memory.
#include "na_x3_common.cuh"

namespace na {
namespace tc {

struct SmemX3 {
    alignas(128) unsigned char b0[kX3B0Chunks * kBChunk];          // 46,080
    alignas(128) unsigned char b1[kX3B1Chunks * kX3B1Chunk];       // 83,200
    alignas(128) unsigned char x[kX3XStages][3 * kAChunk];         // [x_hi | ones | x_lo]
    alignas(128) unsigned char h0[2][12 * kAChunk];                // hi x6 | lo x6 ; also the head's z exchange (tile end)
    alignas(128) unsigned char h1[12 * kAChunk];
    alignas(128) unsigned char onez[2 * kAChunk];                  // [ones | zeros]
    alignas(8) uint64_t x_full[kX3XStages], x_empty[kX3XStages];
    uint64_t d0_full, d1_full, h0_ready[2], h1_ready;
    uint32_t tmem_base;
};

// ---- weight image: [B0 15 chunks][192][8] | [B1 25 chunks][192][8] fp16, row n = (j/4)*16 + gate*4 + j%4 ------------------
__global__ void pack_decoder_x3_kernel(const float* __restrict__ w_ih0, const float* __restrict__ w_hh0,
                                       const float* __restrict__ b_ih0, const float* __restrict__ b_hh0,
                                       const float* __restrict__ w_ih1, const float* __restrict__ w_hh1,
                                       const float* __restrict__ b_ih1, const float* __restrict__ b_hh1,
                                       uint16_t* __restrict__ out) {
    const int total0 = kX3B0Chunks * 8 * kN, total1 = kX3B1Chunks * 8 * kN;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total0 + total1; idx += gridDim.x * blockDim.x) {
        const bool l1 = idx >= total0;
        const int e = l1 ? idx - total0 : idx;
        const int ch = e / (kN * 8), kk = e % 8;
        const int n = (e / 8) % kN;
        const int j = (n / 16) * 4 + (n % 4), q = (n % 16) / 4;
        const int col = q * kH + j;                       // row of the torch weight tensors
        float v = 0.f;
        bool want_lo = false, is_bias = false;
        if (!l1) {
            if (ch == 0) v = kX3XScaleInv * w_ih0[col * 8 + kk];
            else if (ch == 1) { is_bias = true; v = b_ih0[col] + b_hh0[col]; }
            else if (ch <= 7) v = w_hh0[col * kH + (ch - 2) * 8 + kk];
            else if (ch == 8) { want_lo = true; v = kX3XScaleInv * w_ih0[col * 8 + kk]; }
            else { want_lo = true; v = w_hh0[col * kH + (ch - 9) * 8 + kk]; }
        } else {
            if (ch <= 5) v = w_ih1[col * kH + ch * 8 + kk];
            else if (ch <= 11) v = w_hh1[col * kH + (ch - 6) * 8 + kk];
            else if (ch == 12) { is_bias = true; v = b_ih1[col] + b_hh1[col]; }
            else if (ch <= 18) { want_lo = true; v = w_ih1[col * kH + (ch - 13) * 8 + kk]; }
            else { want_lo = true; v = w_hh1[col * kH + (ch - 19) * 8 + kk]; }
        }
        uint16_t hi, lo;
        split16(v, hi, lo);
        uint16_t r;
        if (is_bias) r = kk == 0 ? hi : (kk == 1 ? lo : (uint16_t)0);      // the ones chunk is {1, 1, 0, ...}
        else r = want_lo ? lo : hi;
        out[idx] = r;
    }
}

// Epilogue of one tile for one warp: both layers of (lane quarter q, unit group g).  R = row replication as in
// decoder_infer_v2_kernel: the tile holds 128 / R distinct windows, copy rp = q / (4 / R) of source quarter qs = q % (4 / R)
// takes granules [4 g + rp * (4 / R), + 4 / R) of the 12 four-unit granules and stores its h (hi and lo) to every copy.
// kEx: also store the attention scores (time-major [T][B]) and the pooled vector / LayerNorm output ([B][48]) of every
// window b < B: the scores and the LayerNorm output by the first row copy of the g == 0 warps (the one that runs the
// head), the pooled vector by every thread for the units it pooled.
template <int R, int NR, bool kEx>
__device__ __forceinline__ void x3_epilogue_tile(SmemX3& S, const int q, const int g, const int lane, const int nq, const int T,
                                                 const int n0, uint32_t& k1, const uint32_t tmem_d0, const uint32_t tmem_d1,
                                                 const int64_t b0, const int64_t B, const int NC,
                                                 const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                                                 const float* __restrict__ fc0_w, const float* __restrict__ fc0_b,
                                                 const float* __restrict__ fc3_w, const float* __restrict__ fc3_b,
                                                 float* __restrict__ logits, float* __restrict__ probs,
                                                 float* __restrict__ scores_tm, float* __restrict__ pooled,
                                                 float* __restrict__ embedding) {
    constexpr int kQ = 4 / R, kSlots = 4 / R, kU = 4 * kSlots;
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
                if (q == 0 && g == 0 && lane == 0) mbar_arrive(&S.x_empty[n % kX3XStages]);
                mbar_arrive(&S.h0_ready[n & 1]);
            }
            if (t >= 1) { mbar_wait(&S.d1_full, k1 & 1); ++k1; mbar_arrive(&S.h1_ready); }
        }
        mbar_wait(&S.d1_full, k1 & 1); ++k1;
        return;
    }
    float c0[kU], c1[kU], z[kU], hprev[kU];
#pragma unroll
    for (int j = 0; j < kU; ++j) { c0[j] = 0.f; c1[j] = 0.f; z[j] = 0.f; hprev[j] = 0.f; }
    float mx = -INFINITY, l = 0.f;
    auto pool = [&](float score) {                 // online softmax over time (lstm_eeg_model.py:35-37), fp32
        if (score > mx) {
            const float sc = expf(mx - score);
            l *= sc;
#pragma unroll
            for (int j = 0; j < kU; ++j) z[j] *= sc;
            mx = score;
        }
        const float e = expf(score - mx);
        l += e;
#pragma unroll
        for (int j = 0; j < kU; ++j) z[j] = fmaf(e, hprev[j], z[j]);
    };
    // gates of this thread's granules -> cell update -> h (fp32, kept in hout) -> hi / lo fp16 into every row copy of `buf`
    auto layer_phase = [&](const uint32_t tmem_d, float* c, unsigned char* buf, float* hout) {
        if constexpr (R == 4) {
            uint32_t v[16];
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                  "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                : "r"(tmem_d + lane_base + gr0 * 16)
                : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            cell_granule_exact<NR>(v, c, hout);
            const uint32_t hi0 = pack_val(hout[0], hout[1]), hi1 = pack_val(hout[2], hout[3]);
            const uint32_t lo0 = pack_val(hout[0] - val_lo(hi0), hout[1] - val_hi(hi0));
            const uint32_t lo1 = pack_val(hout[2] - val_lo(hi1), hout[3] - val_hi(hi1));
            unsigned char* dst = buf + (gr0 >> 1) * kAChunk + wrow * 16 + (gr0 & 1) * 8;
#pragma unroll
            for (int rep = 0; rep < 4; ++rep) {
                asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(smem_u32(dst + rep * 32 * 16)), "r"(hi0), "r"(hi1) : "memory");
                asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(smem_u32(dst + 6 * kAChunk + rep * 32 * 16)), "r"(lo0), "r"(lo1) : "memory");
            }
        } else {
#pragma unroll
            for (int pr = 0; pr < kSlots / 2; ++pr) {       // pairs of granules = one 8-unit K chunk
                uint32_t v[32], hi[4], lo[4];
                tmem_ld32(tmem_d + lane_base + (gr0 + 2 * pr) * 16, v);
                cell_granule_exact<NR>(v, c + pr * 8, hout + pr * 8);
                cell_granule_exact<NR>(v + 16, c + pr * 8 + 4, hout + pr * 8 + 4);
                split_pack8(hout + pr * 8, hi, lo);
                unsigned char* dst = buf + ((gr0 >> 1) + pr) * kAChunk + wrow * 16;
#pragma unroll
                for (int rep = 0; rep < R; ++rep) {
                    st_shared_v4(dst + rep * (kRows / R) * 16, hi[0], hi[1], hi[2], hi[3]);
                    st_shared_v4(dst + 6 * kAChunk + rep * (kRows / R) * 16, lo[0], lo[1], lo[2], lo[3]);
                }
            }
        }
    };
    for (int t = 0; t <= T; ++t) {
        const int n = n0 + t;
        if (t < T) {                               // ---- layer 0, step t
            mbar_wait(&S.d0_full, n & 1);
            if (q == 0 && g == 0 && lane == 0) mbar_arrive(&S.x_empty[n % kX3XStages]);
            tc_fence_after();
            float hdummy[kU];
            layer_phase(tmem_d0, c0, S.h0[n & 1], hdummy);
            tc_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(&S.h0_ready[n & 1]);
        }
        if (t >= 1) {                              // ---- layer 1, step t-1 (+ pooling of step t-2)
            mbar_wait(&S.d1_full, k1 & 1); ++k1;
            tc_fence_after();
            uint32_t sc2[2];
            x3_tmem_ld2(tmem_d1 + lane_base + kN, sc2);
            if (t >= 2) pool(__uint_as_float(sc2[0]));     // pooling of step t-2 (h_{t-2} in hprev) first: frees hprev
            if constexpr (kEx)
                if (t >= 2 && ex_writer && scores_tm) scores_tm[(int64_t)(t - 2) * B + b0 + wrow] = __uint_as_float(sc2[0]);
            layer_phase(tmem_d1, c1, S.h1, hprev);
            tc_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(&S.h1_ready);
        }
    }
    {                                              // flush: score of the last step
        mbar_wait(&S.d1_full, k1 & 1); ++k1;
        tc_fence_after();
        uint32_t sc2[2];
        x3_tmem_ld2(tmem_d1 + lane_base + kN, sc2);
        tc_fence_before();
        pool(__uint_as_float(sc2[0]));
        if constexpr (kEx)
            if (ex_writer && scores_tm) scores_tm[(int64_t)(T - 1) * B + b0 + wrow] = __uint_as_float(sc2[0]);
    }
    // ---- head: LN -> fc0 -> RReLU(eval) -> fc3 -> softmax (fp32; parameters from global memory) ------
    float* zx = reinterpret_cast<float*>(S.h0[0]);             // [128][49] floats <= the two h0 buffers
#pragma unroll
    for (int j = 0; j < kU; ++j) zx[wrow * (kH + 1) + gr0 * 4 + j] = z[j];
    if constexpr (kEx)
        // every copy stores the units it pooled, from its own registers: a further use of the head's products would
        // change which of them the assembler contracts into FMAs, and the logits would no longer be the default's
        if (pooled && b0 + wrow < B) {
            float zp[kU];
            const float inv = 1.0f / l;
#pragma unroll
            for (int j = 0; j < kU; ++j) zp[j] = z[j] * inv;
            store_row<kU>(pooled + (b0 + wrow) * kH + gr0 * 4, zp);
        }
    named_bar_sync(1 + qs, 96 * R);                // the 3 R warps that share source quarter qs
    if (g == 0 && rp == 0) {
        const int64_t b = b0 + wrow;
        float zf[kH];
        const float inv_l = 1.0f / l;
        float mean = 0.f;
#pragma unroll
        for (int j = 0; j < kH; ++j) { zf[j] = zx[wrow * (kH + 1) + j] * inv_l; mean += zf[j]; }
        mean *= (1.0f / kH);
        float var = 0.f;
#pragma unroll
        for (int j = 0; j < kH; ++j) { const float d = zf[j] - mean; var = fmaf(d, d, var); }
        const float rstd = 1.0f / sqrtf(var * (1.0f / kH) + kLnEps);
#pragma unroll
        for (int j = 0; j < kH; ++j) zf[j] = fmaf((zf[j] - mean) * rstd, __ldg(ln_w + j), __ldg(ln_b + j));
        if constexpr (kEx)
            if (ex_writer && embedding) store_row<kH>(embedding + b * kH, zf);
        float lg[NA_MAX_CLASSES];
#pragma unroll
        for (int k = 0; k < NA_MAX_CLASSES; ++k) lg[k] = (k < NC) ? __ldg(fc3_b + k) : -INFINITY;
        for (int o = 0; o < kX3Fc; ++o) {
            float a = __ldg(fc0_b + o);
#pragma unroll
            for (int j = 0; j < kH; ++j) a = fmaf(__ldg(fc0_w + o * kH + j), zf[j], a);
            a = a >= 0.f ? a : a * kRReluEvalSlope;
#pragma unroll
            for (int k = 0; k < NA_MAX_CLASSES; ++k)
                if (k < NC) lg[k] = fmaf(__ldg(fc3_w + k * kX3Fc + o), a, lg[k]);
        }
        if (b < B) {
            float mxl = -INFINITY;
#pragma unroll
            for (int k = 0; k < NA_MAX_CLASSES; ++k) mxl = fmaxf(mxl, lg[k]);
            float den = 0.f, pe[NA_MAX_CLASSES];
#pragma unroll
            for (int k = 0; k < NA_MAX_CLASSES; ++k) { pe[k] = (k < NC) ? expf(lg[k] - mxl) : 0.f; den += pe[k]; }
#pragma unroll
            for (int k = 0; k < NA_MAX_CLASSES; ++k)
                if (k < NC) {
                    logits[b * NC + k] = lg[k];
                    if (probs) probs[b * NC + k] = pe[k] / den;
                }
        }
    }
}

template <int NR, bool kEx = false>
__global__ void __launch_bounds__(kX3Threads, 1)
decoder_infer_x3_kernel(const float* __restrict__ x32,              // [B][T][8] fp32, batch-first
                        const unsigned char* __restrict__ packed,   // pack_decoder_x3_kernel image
                        const float* __restrict__ attn_w, const float* __restrict__ attn_b,
                        const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                        const float* __restrict__ fc0_w, const float* __restrict__ fc0_b,
                        const float* __restrict__ fc3_w, const float* __restrict__ fc3_b,
                        float* __restrict__ logits, float* __restrict__ probs,
                        int T, int64_t B, int NC, int nquarters,
                        float* __restrict__ scores_tm,              // kEx: [T][B] scores, [B][48] pooled / LayerNorm output
                        float* __restrict__ pooled, float* __restrict__ embedding) {
    constexpr int kMmaWarp = 12, kTmaWarp = 13;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SmemX3& S = *reinterpret_cast<SmemX3*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);

    // ---- one-time setup --------------------------------------------------------------------------
    {
        const uint4* src = reinterpret_cast<const uint4*>(packed);
        uint4* d0 = reinterpret_cast<uint4*>(S.b0);
        constexpr int n0_16 = kX3B0Chunks * kBChunk / 16;
        for (int i = tid; i < n0_16; i += kX3Threads) d0[i] = src[i];
        for (int i = tid; i < kX3B1Chunks * kN; i += kX3Threads) {
            const int ch = i / kN, r = i % kN;
            reinterpret_cast<uint4*>(S.b1 + ch * kX3B1Chunk)[r] = src[n0_16 + i];
        }
        // rows 192..207 of every layer-1 chunk: row 192 = the attention vector split like the weights (hi in the hi
        // chunks of the h1 part, lo in its lo chunks, the bias pair on the ones chunk); everything else zero
        for (int i = tid; i < kX3B1Chunks * 16; i += kX3Threads) {
            const int ch = i / 16, r = i % 16;
            uint16_t w[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                uint16_t val = 0;
                if (r == 0) {
                    uint16_t hi, lo;
                    if (ch >= 6 && ch <= 11) { split16(attn_w[(ch - 6) * 8 + e], hi, lo); val = hi; }
                    else if (ch >= 19) { split16(attn_w[(ch - 19) * 8 + e], hi, lo); val = lo; }
                    else if (ch == 12) { split16(attn_b[0], hi, lo); val = e == 0 ? hi : (e == 1 ? lo : (uint16_t)0); }
                }
                w[e] = val;
            }
            uint4 pk;
            pk.x = w[0] | ((uint32_t)w[1] << 16); pk.y = w[2] | ((uint32_t)w[3] << 16);
            pk.z = w[4] | ((uint32_t)w[5] << 16); pk.w = w[6] | ((uint32_t)w[7] << 16);
            reinterpret_cast<uint4*>(S.b1 + ch * kX3B1Chunk)[kN + r] = pk;
        }
        const uint4 ones = make_uint4(kValOnes2, 0u, 0u, 0u);     // fp16 {1,1,0,0,0,0,0,0}
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        for (int i = tid; i < kRows; i += kX3Threads) {
#pragma unroll
            for (int s = 0; s < kX3XStages; ++s) reinterpret_cast<uint4*>(S.x[s] + kAChunk)[i] = ones;
            reinterpret_cast<uint4*>(S.onez)[i] = ones;
            reinterpret_cast<uint4*>(S.onez + kAChunk)[i] = zero;
        }
        if (tid == 0) {
            for (int s = 0; s < kX3XStages; ++s) { mbar_init(&S.x_full[s], 1); mbar_init(&S.x_empty[s], 1); }
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

    const int q_begin = (int)(((int64_t)blockIdx.x * nquarters) / gridDim.x);
    const int q_end = (int)(((int64_t)(blockIdx.x + 1) * nquarters) / gridDim.x);
    int n0 = 0;
    uint32_t k1 = 0;
    for (int q0 = q_begin; q0 < q_end; n0 += T) {
        const int nq = min(4, q_end - q0);                 // active source quarters of this tile
        const int R = nq == 1 ? 4 : (nq == 2 ? 2 : 1);     // short tiles are row-replicated (see x3_epilogue_tile)
        const int64_t b0 = (int64_t)q0 * 32;

        if (warp == kTmaWarp) {
            // ================= producer: fp32 rows -> x_hi / x_lo chunks (rows of step t+1 are in flight) ========
            const int nrows = nq * 32;
            float4 cur[4][2], nxt[4][2];
            auto fetch = [&](int t, float4 (&v)[4][2]) {
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) {
                    const int row = rr * 32 + lane;
                    const int64_t b = b0 + row;
                    if (row < nrows && b < B) {
                        const float4* src = reinterpret_cast<const float4*>(x32 + (b * T + t) * 8);
                        v[rr][0] = __ldg(src);
                        v[rr][1] = __ldg(src + 1);
                    } else {
                        v[rr][0] = make_float4(0.f, 0.f, 0.f, 0.f);
                        v[rr][1] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
            };
            fetch(0, cur);
            for (int t = 0; t < T; ++t) {
                const int n = n0 + t, s = n % kX3XStages, u = n / kX3XStages;
                if (t + 1 < T) fetch(t + 1, nxt);
                mbar_wait(&S.x_empty[s], (u & 1) ^ 1);
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) {
                    const int row = rr * 32 + lane;
                    if (row < nrows) {
                        const float f[8] = {kX3XScale * cur[rr][0].x, kX3XScale * cur[rr][0].y, kX3XScale * cur[rr][0].z, kX3XScale * cur[rr][0].w,
                                            kX3XScale * cur[rr][1].x, kX3XScale * cur[rr][1].y, kX3XScale * cur[rr][1].z, kX3XScale * cur[rr][1].w};
                        uint32_t hi[4], lo[4];
                        split_pack8(f, hi, lo);
                        for (int rep = 0; rep < R; ++rep) {
                            const int rr2 = rep * (kRows / R) + row;
                            st_shared_v4(S.x[s] + rr2 * 16, hi[0], hi[1], hi[2], hi[3]);
                            st_shared_v4(S.x[s] + 2 * kAChunk + rr2 * 16, lo[0], lo[1], lo[2], lo[3]);
                        }
                    }
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.x_full[s]);
#pragma unroll
                for (int rr = 0; rr < 4; ++rr) { cur[rr][0] = nxt[rr][0]; cur[rr][1] = nxt[rr][1]; }
            }
        } else if (warp == kMmaWarp) {
            // ================= MMA issuer (whole warp, one elected lane) ========================================
            const bool leader = elect_one();
            // descriptors pair two K chunks through the leading byte offset (LBO): adjacent chunks, or chunk + zeros
            const uint32_t a_x0 = smem_u32(S.x[0]), a_zero = smem_u32(S.onez + kAChunk), a_ones = smem_u32(S.onez);
            const uint64_t d_b0 = umma_desc(smem_u32(S.b0), kBChunk, 128), d_b1 = umma_desc(smem_u32(S.b1), kX3B1Chunk, 128);
            const uint64_t d_h0[2] = {umma_desc(smem_u32(S.h0[0]), kAChunk, 128), umma_desc(smem_u32(S.h0[1]), kAChunk, 128)};
            const uint64_t d_h1 = umma_desc(smem_u32(S.h1), kAChunk, 128);
            const uint64_t d_bias = umma_desc(a_ones, kAChunk, 128);                                // (ones | zeros)
            for (int t = 0; t <= T; ++t) {
                const int n = n0 + t;
                if (t >= 1) {                                  // h0_{t-1} (hi and lo) written, D0 drained
                    mbar_wait(&S.h0_ready[(n - 1) & 1], ((n - 1) >> 1) & 1);
                    tc_fence_after();
                }
                if (t < T) {                                   // layer 0, step t
                    const int s = n % kX3XStages, u = n / kX3XStages;
                    mbar_wait(&S.x_full[s], u & 1);
                    tc_fence_after();
                    const uint32_t xs = a_x0 + s * 3 * kAChunk;
                    if (leader) {
                        // (x_hi | ones) . (Wih_hi | bias);  (x_hi | zeros) . (Wih_lo | *);  (x_lo | zeros) . (Wih_hi | *)
                        umma_bf16(tmem_d0, umma_desc(xs, kAChunk, 128), d_b0, 0u);
                        umma_bf16(tmem_d0, umma_desc(xs, a_zero - xs, 128), desc_adv(d_b0, 8 * kBChunk), 1u);
                        umma_bf16(tmem_d0, umma_desc(xs + 2 * kAChunk, a_zero - (xs + 2 * kAChunk), 128), d_b0, 1u);
                    }
                    if (t >= 1) {
                        const uint64_t hp = d_h0[(n - 1) & 1];
#pragma unroll
                        for (int i = 0; i < 3; ++i) {
                            if (leader) {
                                umma_bf16(tmem_d0, desc_adv(hp, 2 * i * kAChunk), desc_adv(d_b0, (2 + 2 * i) * kBChunk), 1u);        // hi . hi
                                umma_bf16(tmem_d0, desc_adv(hp, 2 * i * kAChunk), desc_adv(d_b0, (9 + 2 * i) * kBChunk), 1u);        // hi . lo
                                umma_bf16(tmem_d0, desc_adv(hp, (6 + 2 * i) * kAChunk), desc_adv(d_b0, (2 + 2 * i) * kBChunk), 1u);  // lo . hi
                            }
                        }
                    }
                    if (leader) umma_commit(&S.d0_full);
                }
                if (t >= 1) {                                  // layer 1, step m = t - 1
                    const int m = n - 1;
                    if (t >= 2) {
                        mbar_wait(&S.h1_ready, (m - 1) & 1);
                        tc_fence_after();
                    }
                    const uint64_t hin = d_h0[m & 1];
                    if (leader) umma_bf16_i(tmem_d1, d_bias, desc_adv(d_b1, 12 * kX3B1Chunk), kX3IdescL1, 0u);
#pragma unroll
                    for (int i = 0; i < 3; ++i) {
                        if (leader) {
                            umma_bf16_i(tmem_d1, desc_adv(hin, 2 * i * kAChunk), desc_adv(d_b1, 2 * i * kX3B1Chunk), kX3IdescL1, 1u);
                            umma_bf16_i(tmem_d1, desc_adv(hin, 2 * i * kAChunk), desc_adv(d_b1, (13 + 2 * i) * kX3B1Chunk), kX3IdescL1, 1u);
                            umma_bf16_i(tmem_d1, desc_adv(hin, (6 + 2 * i) * kAChunk), desc_adv(d_b1, 2 * i * kX3B1Chunk), kX3IdescL1, 1u);
                        }
                    }
                    if (t >= 2) {
#pragma unroll
                        for (int i = 0; i < 3; ++i) {
                            if (leader) {
                                umma_bf16_i(tmem_d1, desc_adv(d_h1, 2 * i * kAChunk), desc_adv(d_b1, (6 + 2 * i) * kX3B1Chunk), kX3IdescL1, 1u);
                                umma_bf16_i(tmem_d1, desc_adv(d_h1, 2 * i * kAChunk), desc_adv(d_b1, (19 + 2 * i) * kX3B1Chunk), kX3IdescL1, 1u);
                                umma_bf16_i(tmem_d1, desc_adv(d_h1, (6 + 2 * i) * kAChunk), desc_adv(d_b1, (6 + 2 * i) * kX3B1Chunk), kX3IdescL1, 1u);
                            }
                        }
                    }
                    if (leader) umma_commit(&S.d1_full);
                }
            }
            {   // flush: score of the last step into the 16 score columns (rows 192..207 of the h1-part chunks + bias)
                const int m = n0 + T - 1;
                mbar_wait(&S.h1_ready, m & 1);
                tc_fence_after();
                const uint64_t d_b1s = desc_adv(d_b1, kN * 16);
                if (leader) umma_bf16_i(tmem_d1 + kN, d_bias, desc_adv(d_b1s, 12 * kX3B1Chunk), kX3IdescFlush, 0u);
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    if (leader) {
                        umma_bf16_i(tmem_d1 + kN, desc_adv(d_h1, 2 * i * kAChunk), desc_adv(d_b1s, (6 + 2 * i) * kX3B1Chunk), kX3IdescFlush, 1u);
                        umma_bf16_i(tmem_d1 + kN, desc_adv(d_h1, 2 * i * kAChunk), desc_adv(d_b1s, (19 + 2 * i) * kX3B1Chunk), kX3IdescFlush, 1u);
                        umma_bf16_i(tmem_d1 + kN, desc_adv(d_h1, (6 + 2 * i) * kAChunk), desc_adv(d_b1s, (6 + 2 * i) * kX3B1Chunk), kX3IdescFlush, 1u);
                    }
                }
                if (leader) umma_commit(&S.d1_full);
            }
        } else {
            // ================= epilogue: both layers of (quarter q, unit group g) ================================
            const int q = warp & 3, g = warp >> 2;
            if (R == 1) x3_epilogue_tile<1, NR, kEx>(S, q, g, lane, nq, T, n0, k1, tmem_d0, tmem_d1, b0, B, NC, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, scores_tm, pooled, embedding);
            else if (R == 2) x3_epilogue_tile<2, NR, kEx>(S, q, g, lane, nq, T, n0, k1, tmem_d0, tmem_d1, b0, B, NC, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, scores_tm, pooled, embedding);
            else x3_epilogue_tile<4, NR, kEx>(S, q, g, lane, nq, T, n0, k1, tmem_d0, tmem_d1, b0, B, NC, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, scores_tm, pooled, embedding);
        }
        __syncthreads();       // tile done: every MMA has completed; the z exchange in h0 has been consumed
        q0 += nq;
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kTmaWarp) {
        tc_fence_after();
        tmem_free_all(tmem);
    }
}

}  // namespace tc
}  // namespace na

namespace na { namespace tc {
int g_x3_rcp_fma = kX3DefaultNR;
void set_x3_rcp_fma(int v) { g_x3_rcp_fma = v; }
} }

extern "C" int64_t na_decoder_packed_x3_bytes(void) {
    return (int64_t)(na::tc::kX3B0Chunks + na::tc::kX3B1Chunks) * na::tc::kBChunk;
}

extern "C" int na_decoder_pack_x3(const float* w_ih0, const float* w_hh0, const float* b_ih0, const float* b_hh0,
                                  const float* w_ih1, const float* w_hh1, const float* b_ih1, const float* b_hh1,
                                  void* packed, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE_PTR(w_ih0); NA_REQUIRE_PTR(w_hh0); NA_REQUIRE_PTR(b_ih0); NA_REQUIRE_PTR(b_hh0);
    NA_REQUIRE_PTR(w_ih1); NA_REQUIRE_PTR(w_hh1); NA_REQUIRE_PTR(b_ih1); NA_REQUIRE_PTR(b_hh1);
    NA_REQUIRE_PTR(packed);
    tc::pack_decoder_x3_kernel<<<128, 256, 0, as_stream(stream)>>>(w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1,
                                                                   reinterpret_cast<uint16_t*>(packed));
    count_launch();
    return check_launch("na_decoder_pack_x3");
}

extern "C" int na_decoder_infer_x3_ex(const float* x, const void* packed, const float* attn_w, const float* attn_b,
                                      const float* ln_w, const float* ln_b, const float* fc0_w, const float* fc0_b,
                                      const float* fc3_w, const float* fc3_b, float* logits, float* probs, float* scores_tm,
                                      float* pooled, float* embedding, int64_t T, int64_t B, int64_t NC, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(T >= 1 && T < (1 << 20) && B >= 1, NA_EINVAL, "na_decoder_infer_x3: bad shape T=%lld B=%lld", (long long)T, (long long)B);
    NA_REQUIRE(NC >= 1 && NC <= NA_MAX_CLASSES, NA_EUNSUPPORTED, "na_decoder_infer_x3: num_classes=%lld", (long long)NC);
    NA_REQUIRE_PTR(x); NA_REQUIRE_PTR(packed); NA_REQUIRE_PTR(logits);
    NA_OPTIONAL_PTR(probs);
    NA_OPTIONAL_PTR(scores_tm); NA_OPTIONAL_PTR(pooled); NA_OPTIONAL_PTR(embedding);
    NA_REQUIRE(attn_w && attn_b && ln_w && ln_b && fc0_w && fc0_b && fc3_w && fc3_b, NA_EINVAL,
               "na_decoder_infer_x3: null parameter pointer");
    const bool ex = scores_tm || pooled || embedding;
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    const size_t smem = sizeof(tc::SmemX3) + 1024;
    const int nquarters = (int)((B + 31) / 32);
    const int grid = nquarters < sms ? nquarters : sms;    // < 4 quarters per CTA run as row-replicated tiles
#define NA_X3_LAUNCH(NRV, EXV)                                                                                                       \
    {                                                                                                                                \
        cudaError_t e = cudaFuncSetAttribute(tc::decoder_infer_x3_kernel<NRV, EXV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e != cudaSuccess) return fail((int)e, "na_decoder_infer_x3: shared memory opt-in failed (%s)", cudaGetErrorString(e));    \
        tc::decoder_infer_x3_kernel<NRV, EXV><<<grid, tc::kX3Threads, smem, as_stream(stream)>>>(                                    \
            x, reinterpret_cast<const unsigned char*>(packed), attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, \
            (int)T, B, (int)NC, nquarters, scores_tm, pooled, embedding);                                                            \
    }
    switch (tc::g_x3_rcp_fma * 2 + (ex ? 1 : 0)) {
        case 0: NA_X3_LAUNCH(0, false) break;
        case 1: NA_X3_LAUNCH(0, true) break;
        case 4: NA_X3_LAUNCH(2, false) break;
        case 5: NA_X3_LAUNCH(2, true) break;
        case 6: NA_X3_LAUNCH(3, false) break;
        case 7: NA_X3_LAUNCH(3, true) break;
        default:
            if (ex) NA_X3_LAUNCH(1, true) else NA_X3_LAUNCH(1, false)
            break;
    }
#undef NA_X3_LAUNCH
    count_launch();
    return check_launch("na_decoder_infer_x3");
}

extern "C" int na_decoder_infer_x3(const float* x, const void* packed, const float* attn_w, const float* attn_b,
                                   const float* ln_w, const float* ln_b, const float* fc0_w, const float* fc0_b,
                                   const float* fc3_w, const float* fc3_b, float* logits, float* probs, int64_t T,
                                   int64_t B, int64_t NC, na_stream_t stream) {
    return na_decoder_infer_x3_ex(x, packed, attn_w, attn_b, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, logits, probs, nullptr,
                                  nullptr, nullptr, T, B, NC, stream);
}
