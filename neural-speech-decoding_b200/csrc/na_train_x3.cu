// Exact tier (fp32 contract, 1e-5 on logits AND gradients), TRAINING, on the tensor cores.
//
// Same idea as the exact inference kernel (na_decoder_x3.cu): every fp32 operand is split into two fp16 halves
// (v = hi + lo + O(2^-22 |v|)) and every product is three tcgen05 MMAs (hi.hi + hi.lo + lo.hi) with fp32 accumulation in
// TMEM; activations through ex2 / rcp (2e-7), never tanh.approx.  It replaces the FFMA recurrence / generic BPTT kernels
// (na_lstm_h48.cu, na_lstm_generic.cu: 0.16 M windows/s per train step) at the flagship shape (C = 8, H = 48, 2 layers).
//
// One kernel per layer and direction, 128-window tiles (UMMA M = 128), 12 epilogue warps (TMEM lane quarter x 16-unit
// group) + one MMA-issuing warp + one TMA producer lane, persistent over tiles:
//
//   lstm_fwd_x3_kernel<L>    gates_t = [in_t | 1 | h_{t-1}] . W (3-way split) -> cell update -> h_t, c_t saved
//                            L = 0: also h0 after dropout (the input of layer 1);  L = 1: attention score as an extra
//                            accumulator column of the NEXT step's MMA, online-softmax pooling -> z, (max, sum)
//   lstm_bwd_x3_kernel<L>    per step, descending: G = the same gate recompute; epilogue: activations, d(gates) from
//                            dh_t = dh_in_t + dh_rec, c_t, c_{t-1}; R: [din | dh_rec] = dG . [W_ih | W_hh] (the forward
//                            weight image re-used as an MN-major B operand: no transposed copy); d(gates) go to shared
//                            memory (A operand of R) and to HBM (hi / lo) for the weight-gradient kernel.
//                            L = 1 fuses the time loop of the head backward (dh_t = alpha_t dz + ds_t w_a, centred form).
//   lstm_wgrad_x3_kernel<L>  time-parallel dW = sum_{t, tile} [in_t | h_{t-1} | 1]^T . dG_t (3-way split, both operands
//                            MN-major straight from the saved tile-chunk slabs), fp32 accumulation in TMEM over all the
//                            work items of a CTA, per-CTA partials reduced in a fixed order (bit-reproducible).
//
// Step pipelines (round 2, second pass).  Forward: two gate accumulators; the input + bias MMAs of step t+1 are issued right
// behind the recurrent MMAs of step t (only 9 of a step's 12 / 19 MMAs wait for h_t), saves go to HBM after the release fence.
// BPTT: two gate accumulators as well (the recompute of step t-1 runs under the epilogue of step t); half tiles evaluate the
// activations under R.  Weight gradients, half tiles: d(gates) are stored compactly (64 rows per chunk) and the kernel runs
// four half-size stages.
//
// Layouts (tile = 128 consecutive windows, chunk = [128 rows][8 fp16] = 2 KB, the UMMA no-swizzle core-matrix layout):
//   XS    fp16 [T][NT][2][128][8]     x / 16 split: chunk 0 = hi, 1 = lo                      (na_x3_split_input)
//   TCLX  fp16 [T][NT][12][128][8]    h split: chunks 0-5 = hi (units 8c..8c+7), 6-11 = lo
//   TCL32 fp32 [T][NT][12][128][4]    c, din (thread = window reads / writes 16 B, coalesced)
//   DGX   fp16 [T][NT][48][128][8]    d(gates) split: chunks 0-23 = hi, 24-47 = lo; column n = (j/4)*16 + gate*4 + j%4
//         (half tiles: [T][NT][48][64][8] -- only the 64 real window rows of a tile are stored)
#include "na_x3_common.cuh"

namespace na {
int reduce_partials(const float* partial, float* out, int nchunks, int64_t n, cudaStream_t st);   // na_reduce.cu
namespace tc {

constexpr int kTxThreads = 14 * 32;
constexpr int kTxMmaWarp = 12, kTxTmaWarp = 13;
constexpr int kTxStages = 3;
constexpr uint32_t kTxAccCols = 256;      // forward: TMEM column stride of the two gate accumulators (192 gates + 16 score columns)

// kDx backward (layer 0): dx = dG . [W_ih | bias] as an N = 16 accumulator at TMEM column 2 x 192 + 64 (464 of 512 in use)
constexpr uint32_t kTxDxCol = 2 * kN + 64;
constexpr uint32_t kTxIdescDx = make_idesc(16, kFmtVal, kFmtVal, false, true);

__device__ __forceinline__ int64_t tclx_off(int t, int ntiles, int tile, int chunk, int row) {       // fp16 elements
    return ((((int64_t)t * ntiles + tile) * 12 + chunk) * kRows + row) * 8;
}
__device__ __forceinline__ int64_t tcl32x_off(int t, int ntiles, int tile, int chunk, int row) {     // fp32 elements
    return ((((int64_t)t * ntiles + tile) * 12 + chunk) * kRows + row) * 4;
}
__device__ __forceinline__ int64_t dgx_off(int t, int ntiles, int tile, int chunk, int row) {        // fp16 elements
    return ((((int64_t)t * ntiles + tile) * 48 + chunk) * kRows + row) * 8;
}
// half tiles: only the 64 real window rows are stored ([T][NT][48][64][8]), so the weight-gradient kernel fetches a whole
// column group with one bulk copy
__device__ __forceinline__ int64_t dgx_half_off(int t, int ntiles, int tile, int chunk, int row) {   // fp16 elements
    return ((((int64_t)t * ntiles + tile) * 48 + chunk) * 64 + row) * 8;
}
template <bool HALF>
__device__ __forceinline__ int64_t dgx_any(int t, int ntiles, int tile, int chunk, int row) {
    return HALF ? dgx_half_off(t, ntiles, tile, chunk, row) : dgx_off(t, ntiles, tile, chunk, row);
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// input split: fp32 [B][T][8] -> XS (x / 16 as fp16 hi + lo), padding rows zero
// ---------------------------------------------------------------------------------------------------------------
// half != 0 (half tiles): window b lives in row (b / 64) * 128 + b % 64 AND in the mirror row + 64 (see lstm_fwd_x3_kernel)
constexpr int kSplitTC = 16;     // timesteps per warp: 16 x 32 B = four 128-byte lines of a window, re-used out of L1
// warp = 32 consecutive window slots (lane = row of a tile), looping over kSplitTC timesteps: every store is a 512-byte
// contiguous run of a chunk (the first version mapped consecutive threads to consecutive t: 16-byte stores 4 KB apart, 0.35 ms
// per 8,192 windows), every 128-byte line of x is fetched from HBM once.
__global__ void __launch_bounds__(256) x3_split_input_kernel(const float* __restrict__ x, __half* __restrict__ xs, int64_t B, int T, int64_t Bp, int half) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t b = (int64_t)blockIdx.x * 32 + lane;                            // window slot
    const int t0 = (blockIdx.y * 8 + w) * kSplitTC;
    const int ntiles = (int)(Bp / kRows);
    const int per = half ? 64 : kRows;
    const int tile = (int)(b / per), row = (int)(b % per);
    const float* src = x + b * (int64_t)T * 8;
    for (int t = t0; t < t0 + kSplitTC && t < T; ++t) {
        float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (b < B) {
            const float4 a0 = *reinterpret_cast<const float4*>(src + (int64_t)t * 8), a1 = *reinterpret_cast<const float4*>(src + (int64_t)t * 8 + 4);
            f[0] = kX3XScale * a0.x; f[1] = kX3XScale * a0.y; f[2] = kX3XScale * a0.z; f[3] = kX3XScale * a0.w;
            f[4] = kX3XScale * a1.x; f[5] = kX3XScale * a1.y; f[6] = kX3XScale * a1.z; f[7] = kX3XScale * a1.w;
        }
        uint32_t hi[4], lo[4];
        split_pack8(f, hi, lo);
        __half* dst = xs + ((((int64_t)t * ntiles + tile) * 2) * kRows + row) * 8;
        *reinterpret_cast<uint4*>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(dst + kRows * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        if (half) {
            *reinterpret_cast<uint4*>(dst + 64 * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(dst + kRows * 8 + 64 * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// forward of one layer with saves
// ---------------------------------------------------------------------------------------------------------------
template <int LAYER>
struct TxFwdSmem {
    static constexpr int kBBytes = LAYER == 0 ? kX3B0Chunks * kBChunk : kX3B1Chunks * kX3B1Chunk;
    static constexpr int kInChunks = LAYER == 0 ? 2 : 12;
    alignas(128) unsigned char b[kBBytes];
    alignas(128) unsigned char in[kTxStages][kInChunks * kAChunk];
    alignas(128) unsigned char h[12 * kAChunk];                     // h_{t-1}: hi x6 | lo x6
    alignas(128) unsigned char onez[2 * kAChunk];                   // [ones | zeros]
    alignas(8) uint64_t in_full[kTxStages], in_empty[kTxStages];
    uint64_t d_full, h_ready;
    uint32_t tmem_base;
};

// HALF = half tiles (strong scaling / small batches, as in the 16-bit tier): 64 distinct windows per tile, rows 64..127 of
// every operand mirror rows 0..63; copy rp = q / 2 of a window takes K chunk 2 g + rp (8 units per thread instead of 16)
// and stores h to both row copies (shared memory and HBM), so every MMA row stays complete.
template <int LAYER, bool HALF>
__global__ void __launch_bounds__(kTxThreads, 1)
lstm_fwd_x3_kernel(const __half* __restrict__ in,                   // L0: XS;  L1: TCLX (h0, or h0 after dropout)
                   const unsigned char* __restrict__ packed,        // this layer's part of the pack_decoder_x3_kernel image
                   const float* __restrict__ attn_w, const float* __restrict__ attn_b,        // L1
                   const unsigned char* __restrict__ mask, uint64_t seed, uint32_t thresh16, float drop_scale,   // L0: dropout of h0
                   __half* __restrict__ h_out, __half* __restrict__ hd_out, float* __restrict__ c_out,
                   float* __restrict__ zpool, float* __restrict__ stats, int64_t B,          // L1
                   int T, int64_t Bp, int ntiles, int64_t drop_stride) {
    using SM = TxFwdSmem<LAYER>;
    constexpr int kInChunks = SM::kInChunks;
    constexpr int kNW = LAYER == 0 ? kN : kX3N1;                      // accumulator columns (L1: + 16 score columns)
    constexpr int kBStride = LAYER == 0 ? kBChunk : kX3B1Chunk;
    constexpr uint32_t kIdescG = make_idesc(kNW, kFmtVal, kFmtVal);
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SM& S = *reinterpret_cast<SM*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);

    // ---- one-time setup ---------------------------------------------------------------------------------------
    {
        const uint4* src = reinterpret_cast<const uint4*>(packed);
        if (LAYER == 0) {
            uint4* d0 = reinterpret_cast<uint4*>(S.b);
            for (int i = tid; i < kX3B0Chunks * kBChunk / 16; i += kTxThreads) d0[i] = src[i];
        } else {
            for (int i = tid; i < kX3B1Chunks * kN; i += kTxThreads) {
                const int ch = i / kN, r = i % kN;
                reinterpret_cast<uint4*>(S.b + ch * kX3B1Chunk)[r] = src[i];
            }
            // rows 192..207 of every chunk: row 192 = the attention vector split like the weights, the rest zero
            for (int i = tid; i < kX3B1Chunks * 16; i += kTxThreads) {
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
                reinterpret_cast<uint4*>(S.b + ch * kX3B1Chunk)[kN + r] = pk;
            }
        }
        const uint4 ones = make_uint4(kValOnes2, 0u, 0u, 0u), zero = make_uint4(0u, 0u, 0u, 0u);
        for (int i = tid; i < kRows; i += kTxThreads) {
            reinterpret_cast<uint4*>(S.onez)[i] = ones;
            reinterpret_cast<uint4*>(S.onez + kAChunk)[i] = zero;
        }
        if (tid == 0) {
            for (int s = 0; s < kTxStages; ++s) { mbar_init(&S.in_full[s], 1); mbar_init(&S.in_empty[s], 1); }
            mbar_init(&S.d_full, 1);
            mbar_init(&S.h_ready, 12 * 32);
            fence_mbar_init();
        }
        if (warp == kTxTmaWarp) tmem_alloc_all(&S.tmem_base);
        tc_fence_before();
        fence_proxy_async_smem();
        __syncthreads();
        tc_fence_after();
    }
    const uint32_t tmem_d = __shfl_sync(0xffffffffu, S.tmem_base, 0);
    const bool drop = LAYER == 0 && hd_out != nullptr;

    uint32_t in_cnt = 0;                         // producer / MMA: input stages produced / consumed
    uint32_t hr_cnt = 0;                         // MMA: h_ready phases consumed
    uint32_t df_cnt = 0;                         // epilogue: d_full phases consumed
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t b0 = (int64_t)tile * kRows;
        if (warp == kTxTmaWarp) {
            if (lane == 0)
                for (int t = 0; t < T; ++t, ++in_cnt) {
                    const uint32_t s = in_cnt % kTxStages, u = in_cnt / kTxStages;
                    mbar_wait(&S.in_empty[s], (u & 1) ^ 1);
                    mbar_arrive_expect_tx(&S.in_full[s], kInChunks * kAChunk);
                    bulk_load(S.in[s], in + (((int64_t)t * ntiles + tile) * kInChunks) * (kAChunk / 2), kInChunks * kAChunk, &S.in_full[s]);
                }
        } else if (warp == kTxMmaWarp) {
            const bool leader = elect_one();
            const uint32_t a_ones = smem_u32(S.onez), a_zero = a_ones + kAChunk;
            const uint64_t d_b = umma_desc(smem_u32(S.b), kBStride, 128);
            const uint64_t d_h = umma_desc(smem_u32(S.h), kAChunk, 128);
            const uint64_t d_bias = umma_desc(a_ones, kAChunk, 128);                              // (ones | zeros)
            // Two accumulators (2 x 256 TMEM columns): the input + bias part of step t+1 does not depend on h_t, so it is issued
            // right after the recurrent part of step t and runs under the epilogue of step t; only the 9 recurrent MMAs of a step
            // (of 12 / 19) stay on the critical path h_t -> gates -> h_{t+1}.  Accumulator (t+1) & 1 was last read by the epilogue of
            // step t-1, whose h_ready this warp has already consumed.
            auto issue_in = [&](const int t) {
                const uint32_t s = in_cnt % kTxStages, u = in_cnt / kTxStages;
                ++in_cnt;
                mbar_wait(&S.in_full[s], u & 1);
                tc_fence_after();
                const uint32_t acc = tmem_d + (uint32_t)(t & 1) * kTxAccCols;
                const uint32_t xs = smem_u32(S.in[s]);
                if (LAYER == 0) {
                    if (leader) {
                        // (x_hi | ones) . (Wih_hi | bias);  (x_hi | zeros) . (Wih_lo | *);  (x_lo | zeros) . (Wih_hi | *)
                        umma_bf16_i(acc, umma_desc(xs, a_ones - xs, 128), d_b, kIdescG, 0u);
                        umma_bf16_i(acc, umma_desc(xs, a_zero - xs, 128), desc_adv(d_b, 8 * kBStride), kIdescG, 1u);
                        umma_bf16_i(acc, umma_desc(xs + kAChunk, a_zero - (xs + kAChunk), 128), d_b, kIdescG, 1u);
                    }
                } else {
                    const uint64_t d_in = umma_desc(xs, kAChunk, 128);
                    if (leader) umma_bf16_i(acc, d_bias, desc_adv(d_b, 12 * kBStride), kIdescG, 0u);
#pragma unroll
                    for (int i = 0; i < 3; ++i)
                        if (leader) {
                            umma_bf16_i(acc, desc_adv(d_in, 2 * i * kAChunk), desc_adv(d_b, 2 * i * kBStride), kIdescG, 1u);
                            umma_bf16_i(acc, desc_adv(d_in, 2 * i * kAChunk), desc_adv(d_b, (13 + 2 * i) * kBStride), kIdescG, 1u);
                            umma_bf16_i(acc, desc_adv(d_in, (6 + 2 * i) * kAChunk), desc_adv(d_b, 2 * i * kBStride), kIdescG, 1u);
                        }
                }
                if (leader) umma_commit(&S.in_empty[s]);
            };
            issue_in(0);
            for (int t = 0; t < T; ++t) {
                const uint32_t acc = tmem_d + (uint32_t)(t & 1) * kTxAccCols;
                if (t >= 1) {
                    mbar_wait(&S.h_ready, hr_cnt & 1); ++hr_cnt;
                    tc_fence_after();
                    constexpr int kRecHi = LAYER == 0 ? 2 : 6, kRecLo = LAYER == 0 ? 9 : 19;      // first W_hh chunk (hi / lo) of the image
#pragma unroll
                    for (int i = 0; i < 3; ++i)
                        if (leader) {
                            umma_bf16_i(acc, desc_adv(d_h, 2 * i * kAChunk), desc_adv(d_b, (kRecHi + 2 * i) * kBStride), kIdescG, 1u);
                            umma_bf16_i(acc, desc_adv(d_h, 2 * i * kAChunk), desc_adv(d_b, (kRecLo + 2 * i) * kBStride), kIdescG, 1u);
                            umma_bf16_i(acc, desc_adv(d_h, (6 + 2 * i) * kAChunk), desc_adv(d_b, (kRecHi + 2 * i) * kBStride), kIdescG, 1u);
                        }
                }
                if (leader) umma_commit(&S.d_full);
                if (t + 1 < T) issue_in(t + 1);
            }
            // the last h of the tile has been written (and the accumulator drained)
            mbar_wait(&S.h_ready, hr_cnt & 1); ++hr_cnt;
            tc_fence_after();
            if (LAYER == 1) {   // flush: score of the last step into the 16 score columns
                const uint64_t d_bs = desc_adv(d_b, kN * 16);
                const uint32_t accf = tmem_d + (uint32_t)(T & 1) * kTxAccCols + kN;        // the "next" accumulator's score columns
                if (leader) umma_bf16_i(accf, d_bias, desc_adv(d_bs, 12 * kBStride), kX3IdescFlush, 0u);
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    if (leader) {
                        umma_bf16_i(accf, desc_adv(d_h, 2 * i * kAChunk), desc_adv(d_bs, (6 + 2 * i) * kBStride), kX3IdescFlush, 1u);
                        umma_bf16_i(accf, desc_adv(d_h, 2 * i * kAChunk), desc_adv(d_bs, (19 + 2 * i) * kBStride), kX3IdescFlush, 1u);
                        umma_bf16_i(accf, desc_adv(d_h, (6 + 2 * i) * kAChunk), desc_adv(d_bs, (6 + 2 * i) * kBStride), kX3IdescFlush, 1u);
                    }
                if (leader) umma_commit(&S.d_full);
            }
        } else {
            // ================= epilogue: (lane quarter q, 16-unit group g) =========================================
            const int q = warp & 3, g = warp >> 2;
            const int row = q * 32 + lane;
            const uint32_t lane_base = (uint32_t)(q * 32) << 16;
            constexpr int kNB = HALF ? 1 : 2;                        // 8-unit chunks per thread
            const int rp = HALF ? (q >> 1) : 0;
            const int crow = HALF ? (row & 63) : row;                // canonical row (first copy)
            const int chunk0 = HALF ? 2 * g + rp : 2 * g;            // first K chunk of this thread
            const int64_t bwin = HALF ? (int64_t)tile * 64 + crow : b0 + row;
            float c[8 * kNB], hprev[8 * kNB], z[8 * kNB];
#pragma unroll
            for (int j = 0; j < 8 * kNB; ++j) { c[j] = 0.f; hprev[j] = 0.f; z[j] = 0.f; }
            float mx = -INFINITY, l = 0.f;
            auto pool = [&](float score) {                           // online softmax over time (lstm_eeg_model.py:35-37), fp32
                if (score > mx) {
                    const float sc = expf(mx - score);
                    l *= sc;
#pragma unroll
                    for (int j = 0; j < 8 * kNB; ++j) z[j] *= sc;
                    mx = score;
                }
                const float e = expf(score - mx);
                l += e;
#pragma unroll
                for (int j = 0; j < 8 * kNB; ++j) z[j] = fmaf(e, hprev[j], z[j]);
            };
            for (int t = 0; t < T; ++t) {
                const int64_t grow = (int64_t)t * Bp + b0 + crow;                        // mask-tensor row
                const int64_t gkey = HALF ? (int64_t)t * drop_stride + bwin : grow;     // counter-based generator: layout-independent
                uint32_t keep[kNB];
#pragma unroll
                for (int pr = 0; pr < kNB; ++pr) keep[pr] = 0xFFu;
                if (drop) {
#pragma unroll
                    for (int pr = 0; pr < kNB; ++pr) {
                        const int blk = chunk0 + pr;
                        keep[pr] = mask ? mask_keep8(*reinterpret_cast<const uint2*>(mask + grow * kH + blk * 8))
                                        : dropout_keep8(seed, gkey, blk, thresh16);
                    }
                }
                mbar_wait(&S.d_full, df_cnt & 1); ++df_cnt;
                tc_fence_after();
                const uint32_t acc = tmem_d + (uint32_t)(t & 1) * kTxAccCols;
                if (LAYER == 1) {
                    uint32_t sc2[2];
                    x3_tmem_ld2(acc + lane_base + kN, sc2);
                    if (t >= 1) pool(__uint_as_float(sc2[0]));       // score of h_{t-1}, which is still in hprev
                }
                // h_t goes to shared memory first; the saves go to HBM only AFTER the fence + arrive that release h_t to the tensor
                // pipe (the fence otherwise waits for the global stores, on the step's critical path)
                uint32_t hi[4 * kNB], lo[4 * kNB];
#pragma unroll
                for (int pr = 0; pr < kNB; ++pr) {                    // pairs of granules = one 8-unit chunk
                    uint32_t v[32];
                    const int chunk = chunk0 + pr;
                    tmem_ld32(acc + lane_base + chunk * 32, v);
                    cell_granule_exact(v, c + pr * 8, hprev + pr * 8);
                    cell_granule_exact(v + 16, c + pr * 8 + 4, hprev + pr * 8 + 4);
                    split_pack8(hprev + pr * 8, reinterpret_cast<uint32_t(&)[4]>(hi[pr * 4]), reinterpret_cast<uint32_t(&)[4]>(lo[pr * 4]));
                    st_shared_v4(S.h + chunk * kAChunk + row * 16, hi[pr * 4], hi[pr * 4 + 1], hi[pr * 4 + 2], hi[pr * 4 + 3]);
                    st_shared_v4(S.h + (6 + chunk) * kAChunk + row * 16, lo[pr * 4], lo[pr * 4 + 1], lo[pr * 4 + 2], lo[pr * 4 + 3]);
                    if (HALF) {                                       // the other row copy
                        st_shared_v4(S.h + chunk * kAChunk + (row ^ 64) * 16, hi[pr * 4], hi[pr * 4 + 1], hi[pr * 4 + 2], hi[pr * 4 + 3]);
                        st_shared_v4(S.h + (6 + chunk) * kAChunk + (row ^ 64) * 16, lo[pr * 4], lo[pr * 4 + 1], lo[pr * 4 + 2], lo[pr * 4 + 3]);
                    }
                }
                tc_fence_before();
                fence_proxy_async_smem();
                mbar_arrive(&S.h_ready);
#pragma unroll
                for (int pr = 0; pr < kNB; ++pr) {
                    const int chunk = chunk0 + pr;
                    const uint4 vhi = make_uint4(hi[pr * 4], hi[pr * 4 + 1], hi[pr * 4 + 2], hi[pr * 4 + 3]);
                    const uint4 vlo = make_uint4(lo[pr * 4], lo[pr * 4 + 1], lo[pr * 4 + 2], lo[pr * 4 + 3]);
                    *reinterpret_cast<uint4*>(h_out + tclx_off(t, ntiles, tile, chunk, row)) = vhi;
                    *reinterpret_cast<uint4*>(h_out + tclx_off(t, ntiles, tile, 6 + chunk, row)) = vlo;
                    if (HALF) {
                        *reinterpret_cast<uint4*>(h_out + tclx_off(t, ntiles, tile, chunk, row ^ 64)) = vhi;
                        *reinterpret_cast<uint4*>(h_out + tclx_off(t, ntiles, tile, 6 + chunk, row ^ 64)) = vlo;
                    }
                    *reinterpret_cast<float4*>(c_out + tcl32x_off(t, ntiles, tile, 2 * chunk, row)) =
                        make_float4(c[pr * 8], c[pr * 8 + 1], c[pr * 8 + 2], c[pr * 8 + 3]);
                    *reinterpret_cast<float4*>(c_out + tcl32x_off(t, ntiles, tile, 2 * chunk + 1, row)) =
                        make_float4(c[pr * 8 + 4], c[pr * 8 + 5], c[pr * 8 + 6], c[pr * 8 + 7]);
                    if (drop) {
                        float hd[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) hd[u] = ((keep[pr] >> u) & 1u) ? hprev[pr * 8 + u] * drop_scale : 0.f;
                        uint32_t dhi[4], dlo[4];
                        split_pack8(hd, dhi, dlo);
                        const uint4 whi = make_uint4(dhi[0], dhi[1], dhi[2], dhi[3]), wlo = make_uint4(dlo[0], dlo[1], dlo[2], dlo[3]);
                        *reinterpret_cast<uint4*>(hd_out + tclx_off(t, ntiles, tile, chunk, row)) = whi;
                        *reinterpret_cast<uint4*>(hd_out + tclx_off(t, ntiles, tile, 6 + chunk, row)) = wlo;
                        if (HALF) {
                            *reinterpret_cast<uint4*>(hd_out + tclx_off(t, ntiles, tile, chunk, row ^ 64)) = whi;
                            *reinterpret_cast<uint4*>(hd_out + tclx_off(t, ntiles, tile, 6 + chunk, row ^ 64)) = wlo;
                        }
                    }
                }
            }
            if (LAYER == 1) {
                mbar_wait(&S.d_full, df_cnt & 1); ++df_cnt;              // flush: score of the last step
                tc_fence_after();
                uint32_t sc2[2];
                x3_tmem_ld2(tmem_d + (uint32_t)(T & 1) * kTxAccCols + lane_base + kN, sc2);
                tc_fence_before();
                pool(__uint_as_float(sc2[0]));
                if (bwin < B) {
                    const float inv_l = 1.0f / l;
                    float* zo = zpool + bwin * kH + chunk0 * 8;
#pragma unroll
                    for (int j = 0; j < 8 * kNB; j += 4)
                        *reinterpret_cast<float4*>(zo + j) = make_float4(z[j] * inv_l, z[j + 1] * inv_l, z[j + 2] * inv_l, z[j + 3] * inv_l);
                    if (g == 0 && rp == 0) { stats[2 * bwin] = mx; stats[2 * bwin + 1] = l; }
                }
            }
        }
        __syncthreads();       // tile done: every MMA of the tile has completed and its accumulator has been read
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kTxTmaWarp) { tc_fence_after(); tmem_free_all(tmem_d); }
}

// ---------------------------------------------------------------------------------------------------------------
// backward of one layer
// ---------------------------------------------------------------------------------------------------------------
template <int LAYER>
struct TxBwdSmem {
    static constexpr int kBChunks = LAYER == 0 ? kX3B0Chunks : kX3B1Chunks;
    static constexpr int kActChunks = LAYER == 0 ? 14 : 24;          // L0: [x_hi | x_lo | hp hi x6 | hp lo x6];  L1: [in hi x6 | lo x6 | hp hi x6 | lo x6]
    alignas(128) unsigned char b[kBChunks * kBChunk];                // forward weight image (192 rows per chunk)
    alignas(128) unsigned char act[kActChunks * kAChunk];
    alignas(128) unsigned char dg[48 * kAChunk];                     // d(gates): hi x24 | lo x24
    alignas(128) unsigned char onez[2 * kAChunk];
    alignas(8) uint64_t act_full, act_free;
    uint64_t g_full[2], r_full, dg_ready;     // g_full per gate accumulator: a barrier must never run two phases ahead of its waiter
    uint32_t tmem_base;
    float wa[kH];
    float ba;
    float2 xch[3][kRows];                                           // fused head backward: per-step exchange of the 3 unit-group warps
    alignas(8) uint64_t dx_full;                                    // kDx, layer 0: the dx MMAs of a step have completed (last, so
                                                                    // the other members keep their offsets in every instantiation)
};

// gates of one cell at fp32 accuracy: 5 ex2 + 2 rcp (the reciprocals of each group are combined)
__device__ __forceinline__ void gates_exact(float vi, float vf, float vg, float vo, float ct,
                                            float& gi, float& gf, float& gg, float& go, float& tcv) {
    constexpr float kL2e = 1.4426950408889634f;
    auto capped_ex2 = [](float a) {
        float r;
        asm("min.NaN.f32 %0, %1, 0f42200000;" : "=f"(r) : "f"(a));
        return ex2_approx(r);
    };
    const float ei = capped_ex2(-kL2e * vi), ef = capped_ex2(-kL2e * vf), eg = capped_ex2(-2.0f * kL2e * vg);
    const float eo = capped_ex2(-kL2e * vo), ec = capped_ex2(-2.0f * kL2e * ct);
    const float a = 1.0f + ei, b = 1.0f + ef, cc = 1.0f + eg;
    const float ab = a * b;
    const float r1 = rcp_approx(ab * cc);                            // <= 2^120: finite
    gi = r1 * (b * cc);
    gf = r1 * (a * cc);
    gg = (1.0f - eg) * (r1 * ab);
    const float d = 1.0f + eo, e = 1.0f + ec;
    const float r2 = rcp_approx(d * e);
    go = r2 * e;
    tcv = (1.0f - ec) * (r2 * d);
}

// HALF: half tiles as in lstm_fwd_x3_kernel -- copy rp = q / 2 takes K chunk 2 g + rp (8 units per thread), writes its
// d(gates) to BOTH row copies in shared memory (so D_R is complete on every row) and to the canonical row in HBM (the
// weight-gradient kernel then reads rows 0..63 only).
//
// kDx (input attributions, no weight gradients): neither layer stores DGX nor the d attn partials.  Layer 0 also emits
// dx_t = dG_t . W_ih0 into fp32 [B][T][8]: three more MMAs per K16 slice (N = 16 over image chunks 0-1 | 8-9, i.e. W_ih and the
// bias column, whose 8 products are discarded) into their own TMEM accumulator, issued after R's commit so that they stay off
// the d(gates) -> dh_rec chain, with their own barrier.  Every epilogue warp waits for them before it overwrites the d(gates)
// operand they read; the g == 0 warps read dx(t+1) then, i.e. before dg_ready(t), which the next dx MMAs wait for.
template <int LAYER, bool HALF, bool kDx = false>
__global__ void __launch_bounds__(kTxThreads, 1)
lstm_bwd_x3_kernel(const __half* __restrict__ act_in,               // L0: XS;  L1: TCLX (the layer's forward input)
                   const __half* __restrict__ h,                    // TCLX: this layer's h
                   const float* __restrict__ cstate,                // TCL32
                   const float* __restrict__ dh_in,                 // TCL32 (L0: din of layer 1;  L1 without fused head)
                   const unsigned char* __restrict__ packed,        // this layer's part of the x3 weight image
                   const __half* __restrict__ zeros,                // >= 24 KB of zeros (h_{-1})
                   const unsigned char* __restrict__ mask, uint64_t seed, uint32_t thresh16, float drop_scale,   // L1: dropout of its input
                   float* __restrict__ din,                         // TCL32, L1 only
                   __half* __restrict__ dg_out,                     // DGX
                   const float* __restrict__ dz,
                   const float* __restrict__ stats,                 // L1: softmax (max, sum);  kDx L0: per-window unscale of dz [B]
                   const float* __restrict__ zpool,
                   const float* __restrict__ attn_w, const float* __restrict__ attn_b, int64_t B,
                   float* __restrict__ attn_partial,                // L1: [grid][52] d attn_w | d attn_b;  kDx L0: dx [B][T][8]
                   int T, int64_t Bp, int ntiles, int64_t drop_stride) {
    // (kDx re-uses two pointers that layer 0 has no use for: a new parameter changes the register allocation of every
    // instantiation, and the default ones must keep their SASS)
    using SM = TxBwdSmem<LAYER>;
    constexpr int kInChunks = LAYER == 0 ? 2 : 12;
    constexpr int kHp = LAYER == 0 ? 2 : 12;                         // first h_{t-1} chunk of the act stage
    constexpr int kNR = LAYER == 0 ? 48 : 96;                        // columns of D_R: [din (48) |] dh_rec (48)
    constexpr int kRecCol = LAYER == 0 ? 0 : 48;
    constexpr uint32_t kIdescG = make_idesc(kN, kFmtVal, kFmtVal);
    constexpr uint32_t kIdescR = make_idesc(kNR, kFmtVal, kFmtVal, false, true);      // dG (K-major) x W image (MN-major)
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SM& S = *reinterpret_cast<SM*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    {
        const uint4* src = reinterpret_cast<const uint4*>(packed);
        uint4* db = reinterpret_cast<uint4*>(S.b);
        for (int i = tid; i < SM::kBChunks * kBChunk / 16; i += kTxThreads) db[i] = src[i];
        const uint4 ones = make_uint4(kValOnes2, 0u, 0u, 0u), zero = make_uint4(0u, 0u, 0u, 0u);
        for (int i = tid; i < kRows; i += kTxThreads) {
            reinterpret_cast<uint4*>(S.onez)[i] = ones;
            reinterpret_cast<uint4*>(S.onez + kAChunk)[i] = zero;
        }
        if (tid == 0) {
            mbar_init(&S.act_full, 1); mbar_init(&S.act_free, 1);
            mbar_init(&S.g_full[0], 1); mbar_init(&S.g_full[1], 1); mbar_init(&S.r_full, 1);
            mbar_init(&S.dg_ready, 12 * 32);
            if constexpr (kDx && LAYER == 0) mbar_init(&S.dx_full, 1);
            fence_mbar_init();
        }
        if (dz != nullptr) {
            for (int i = tid; i < kH; i += kTxThreads) S.wa[i] = attn_w[i];
            if (tid == 0) S.ba = attn_b[0];
        }
        if (warp == kTxTmaWarp) tmem_alloc_all(&S.tmem_base);
        tc_fence_before();
        fence_proxy_async_smem();
        __syncthreads();
        tc_fence_after();
    }
    const bool head = LAYER == 1 && dz != nullptr;
    const uint32_t tmem = __shfl_sync(0xffffffffu, S.tmem_base, 0);
    // two gate accumulators (the recompute of step t-1 runs under the epilogue of step t) + D_R: 2 x 192 + 96 = 480 columns
    const uint32_t tm_r = tmem + 2 * kN;
    float dwa[16], dba = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) dwa[j] = 0.f;

    uint32_t act_cnt = 0, dgp = 0, rphase = 0;       // role-private running phase counters
    uint32_t gph[2] = {0, 0};                         // epilogue: g_full phases consumed, per accumulator
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t b0 = (int64_t)tile * kRows;
        if (warp == kTxTmaWarp) {
            // ================= TMA producer: [in_t | h_{t-1}] for t = T-1 .. 0 (single stage) =====================
            if (lane == 0)
                for (int i = 0; i < T; ++i, ++act_cnt) {
                    const int t = T - 1 - i;
                    mbar_wait(&S.act_free, (act_cnt & 1) ^ 1);
                    mbar_arrive_expect_tx(&S.act_full, (kInChunks + 12) * kAChunk);
                    bulk_load(S.act, act_in + (((int64_t)t * ntiles + tile) * kInChunks) * (kAChunk / 2), kInChunks * kAChunk, &S.act_full);
                    const __half* hsrc = t > 0 ? h + tclx_off(t - 1, ntiles, tile, 0, 0) : zeros;
                    bulk_load(S.act + kHp * kAChunk, hsrc, 12 * kAChunk, &S.act_full);
                }
        } else if (warp == kTxMmaWarp) {
            // ================= MMA issuer: per iteration  R(t+1) -> G(t) -> commit ================================
            const bool leader = elect_one();
            const uint32_t a_act = smem_u32(S.act), a_ones = smem_u32(S.onez), a_zero = a_ones + kAChunk;
            const uint64_t d_b = umma_desc(smem_u32(S.b), kBChunk, 128);                    // K-major (gate recompute)
            const uint64_t d_bm = umma_desc(smem_u32(S.b), 128, kBChunk);                   // MN-major: N = input feature, K = gate row
            const uint64_t d_dgk = umma_desc(smem_u32(S.dg), kAChunk, 128);                 // d(gates), K-major A
            const uint64_t d_hp = umma_desc(a_act + kHp * kAChunk, kAChunk, 128);
            const uint64_t d_in = umma_desc(a_act, kAChunk, 128);
            const uint64_t d_bias = umma_desc(a_ones, kAChunk, 128);
            // first weight chunk of the R operand: L0: W_hh (chunks 2..7 hi, 9..14 lo);  L1: [W_ih | W_hh] (0..11 hi, 13..24 lo)
            constexpr int kRHi = LAYER == 0 ? 2 : 0, kRLo = LAYER == 0 ? 9 : 13;
            // gate recompute of step `t` into accumulator `buf`
            auto issue_g = [&](const int buf) {
                const uint32_t tm_g = tmem + buf * kN;
                mbar_wait(&S.act_full, act_cnt & 1); ++act_cnt;
                tc_fence_after();
                if (LAYER == 0) {
                    if (leader) {
                        umma_bf16_i(tm_g, umma_desc(a_act, a_ones - a_act, 128), d_b, kIdescG, 0u);
                        umma_bf16_i(tm_g, umma_desc(a_act, a_zero - a_act, 128), desc_adv(d_b, 8 * kBChunk), kIdescG, 1u);
                        umma_bf16_i(tm_g, umma_desc(a_act + kAChunk, a_zero - (a_act + kAChunk), 128), d_b, kIdescG, 1u);
                    }
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        if (leader) {
                            umma_bf16_i(tm_g, desc_adv(d_hp, 2 * k * kAChunk), desc_adv(d_b, (2 + 2 * k) * kBChunk), kIdescG, 1u);
                            umma_bf16_i(tm_g, desc_adv(d_hp, 2 * k * kAChunk), desc_adv(d_b, (9 + 2 * k) * kBChunk), kIdescG, 1u);
                            umma_bf16_i(tm_g, desc_adv(d_hp, (6 + 2 * k) * kAChunk), desc_adv(d_b, (2 + 2 * k) * kBChunk), kIdescG, 1u);
                        }
                } else {
                    if (leader) umma_bf16_i(tm_g, d_bias, desc_adv(d_b, 12 * kBChunk), kIdescG, 0u);
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        if (leader) {
                            umma_bf16_i(tm_g, desc_adv(d_in, 2 * k * kAChunk), desc_adv(d_b, 2 * k * kBChunk), kIdescG, 1u);
                            umma_bf16_i(tm_g, desc_adv(d_in, 2 * k * kAChunk), desc_adv(d_b, (13 + 2 * k) * kBChunk), kIdescG, 1u);
                            umma_bf16_i(tm_g, desc_adv(d_in, (6 + 2 * k) * kAChunk), desc_adv(d_b, 2 * k * kBChunk), kIdescG, 1u);
                            umma_bf16_i(tm_g, desc_adv(d_hp, 2 * k * kAChunk), desc_adv(d_b, (6 + 2 * k) * kBChunk), kIdescG, 1u);
                            umma_bf16_i(tm_g, desc_adv(d_hp, 2 * k * kAChunk), desc_adv(d_b, (19 + 2 * k) * kBChunk), kIdescG, 1u);
                            umma_bf16_i(tm_g, desc_adv(d_hp, (6 + 2 * k) * kAChunk), desc_adv(d_b, (6 + 2 * k) * kBChunk), kIdescG, 1u);
                        }
                }
                if (leader) umma_commit(&S.act_free);          // the stage may be refilled as soon as G has read it
                if (leader) umma_commit(&S.g_full[buf]);
            };
            // Per iteration i (step t = T-1-i): R(t+1) first -- it is the only MMA on the step's critical path (d(gates) ->
            // dh_rec -> d(gates)) --, then the gate recompute of the NEXT step into the other accumulator, where it runs
            // under this step's epilogue.
            issue_g(0);                                             // G(T-1)
            for (int i = 0; i <= T; ++i) {
                if (i >= 1) {
                    mbar_wait(&S.dg_ready, dgp & 1); ++dgp;
                    tc_fence_after();
#pragma unroll
                    for (int ks = 0; ks < 12; ++ks)
                        if (leader) {
                            const uint64_t ahi = desc_adv(d_dgk, 2 * ks * kAChunk), alo = desc_adv(d_dgk, (24 + 2 * ks) * kAChunk);
                            umma_bf16_i(tm_r, ahi, desc_adv(d_bm, kRHi * kBChunk + ks * 256), kIdescR, ks == 0 ? 0u : 1u);
                            umma_bf16_i(tm_r, ahi, desc_adv(d_bm, kRLo * kBChunk + ks * 256), kIdescR, 1u);
                            umma_bf16_i(tm_r, alo, desc_adv(d_bm, kRHi * kBChunk + ks * 256), kIdescR, 1u);
                        }
                }
                if (leader) umma_commit(&S.r_full);            // R(t+1) done (i == 0: nothing pending)
                if constexpr (kDx && LAYER == 0) {
                    if (i >= 1) {                               // dx(t+1) = dG . [W_ih | bias] (N = 16; columns 8-15 unused)
#pragma unroll
                        for (int ks = 0; ks < 12; ++ks)
                            if (leader) {
                                const uint64_t ahi = desc_adv(d_dgk, 2 * ks * kAChunk), alo = desc_adv(d_dgk, (24 + 2 * ks) * kAChunk);
                                umma_bf16_i(tmem + kTxDxCol, ahi, desc_adv(d_bm, ks * 256), kTxIdescDx, ks == 0 ? 0u : 1u);
                                umma_bf16_i(tmem + kTxDxCol, ahi, desc_adv(d_bm, 8 * kBChunk + ks * 256), kTxIdescDx, 1u);
                                umma_bf16_i(tmem + kTxDxCol, alo, desc_adv(d_bm, ks * 256), kTxIdescDx, 1u);
                            }
                        if (leader) umma_commit(&S.dx_full);
                    }
                }
                if (i + 1 < T) issue_g((i + 1) & 1);           // G(t-1): accumulator (i+1)&1 was drained (and its barrier consumed) in iteration i-1
            }
        } else {
            // ================= epilogue: thread = window row x 16 units ===========================================
            const int q = warp & 3, g = warp >> 2;
            const int row = q * 32 + lane;
            const uint32_t lane_base = (uint32_t)(q * 32) << 16;
            constexpr int kNB = HALF ? 1 : 2, kU = 8 * kNB;          // 8-unit chunks / units per thread
            const int rp = HALF ? (q >> 1) : 0;
            const int crow = HALF ? (row & 63) : row;                // canonical row (first copy)
            const int chunk0 = HALF ? 2 * g + rp : 2 * g;            // first K chunk (8 units) of this thread
            const int gr0 = 2 * chunk0;                              // its first 4-unit granule
            const int u0 = 8 * chunk0;                               // its first hidden unit
            const int64_t bwin = HALF ? (int64_t)tile * 64 + crow : b0 + row;
            const uint32_t xbar = HALF ? 1 + (q & 1) : 1 + q, xcnt = HALF ? 192 : 96;      // the warps that share a window
            // dx(tx): the image's W_ih0 carries the x16 of the x / 16 input split; dz of the window was scaled by 1 / stats[b]
            float* const dx = attn_partial;
            const float dxs = (kDx && LAYER == 0 && bwin < B) ? kX3XScale * stats[bwin] : 0.f;
            auto take_dx = [&](const int tx) {
                // phase: T per tile, consumed in order -- this CTA's earlier tiles, then steps T-1 .. tx of this one
                const uint32_t k = (uint32_t)((tile - (int)blockIdx.x) / (int)gridDim.x) * (uint32_t)T + (uint32_t)(T - 1 - tx);
                mbar_wait(&S.dx_full, k & 1);
                tc_fence_after();
                if (g == 0) {                                        // one writer per window: g == 0, first row copy
                    uint32_t r[8];
                    tmem_ld8(tmem + kTxDxCol + lane_base, r);
                    if (rp == 0 && bwin < B) {
                        float4* o = reinterpret_cast<float4*>(dx + (bwin * T + tx) * 8);
                        o[0] = make_float4(__uint_as_float(r[0]) * dxs, __uint_as_float(r[1]) * dxs, __uint_as_float(r[2]) * dxs, __uint_as_float(r[3]) * dxs);
                        o[1] = make_float4(__uint_as_float(r[4]) * dxs, __uint_as_float(r[5]) * dxs, __uint_as_float(r[6]) * dxs, __uint_as_float(r[7]) * dxs);
                    }
                }
            };
            float dc[kU], ccur[kU];
#pragma unroll
            for (int j = 0; j < kU; ++j) dc[j] = 0.f;
#pragma unroll
            for (int j = 0; j < kU; j += 4) {
                const float4 a = *reinterpret_cast<const float4*>(cstate + tcl32x_off(T - 1, ntiles, tile, gr0 + j / 4, row));
                ccur[j] = a.x; ccur[j + 1] = a.y; ccur[j + 2] = a.z; ccur[j + 3] = a.w;
            }
            float dzr[kU], zr[kU], sm_m = 0.f, inv_l = 1.f;
            if (head) {
                const int64_t b = bwin;
#pragma unroll
                for (int j = 0; j < kU; ++j) {
                    dzr[j] = (b < B) ? dz[b * kH + u0 + j] : 0.f;
                    zr[j] = (b < B) ? zpool[b * kH + u0 + j] : 0.f;
                }
                if (b < B) { sm_m = stats[2 * b]; inv_l = 1.0f / stats[2 * b + 1]; }
            }
            for (int i = 0; i <= T; ++i) {
                const int t = T - 1 - i;
                float cp[kU], dh[kU];
                if (i < T) {
                    // ---- prefetch c_{t-1} and this step's dh BEFORE waiting for the tensor pipe -------------------
#pragma unroll
                    for (int j = 0; j < kU; j += 4) {
                        float4 c4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (t > 0) c4 = *reinterpret_cast<const float4*>(cstate + tcl32x_off(t - 1, ntiles, tile, gr0 + j / 4, row));
                        cp[j] = c4.x; cp[j + 1] = c4.y; cp[j + 2] = c4.z; cp[j + 3] = c4.w;
                    }
                    if (head) {
                        // head backward, time loop (lstm_eeg_model.py:35-37): alpha_t = softmax weight, centred form
                        // ds_t = alpha_t dz . (h_t - z) (no cancellation), dh_t = alpha_t dz + ds_t w_a
                        float hv[kU];
#pragma unroll
                        for (int pr = 0; pr < kNB; ++pr) {
                            // (fetching h one step ahead into registers was measured: no gain, the step is bound by instruction issue)
                            const uint4 ph = *reinterpret_cast<const uint4*>(h + tclx_off(t, ntiles, tile, chunk0 + pr, row));
                            const uint4 pl = *reinterpret_cast<const uint4*>(h + tclx_off(t, ntiles, tile, 6 + chunk0 + pr, row));
                            const uint32_t wh[4] = {ph.x, ph.y, ph.z, ph.w}, wl[4] = {pl.x, pl.y, pl.z, pl.w};
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                hv[pr * 8 + 2 * u] = val_lo(wh[u]) + val_lo(wl[u]);
                                hv[pr * 8 + 2 * u + 1] = val_hi(wh[u]) + val_hi(wl[u]);
                            }
                        }
                        float sp = 0.f, gp = 0.f;
#pragma unroll
                        for (int j = 0; j < kU; ++j) { sp = fmaf(S.wa[u0 + j], hv[j], sp); gp = fmaf(dzr[j], hv[j] - zr[j], gp); }
                        S.xch[g][row] = make_float2(sp, gp);
                        named_bar_sync(xbar, xcnt);
                        float xs = 0.f, xg = 0.f;
#pragma unroll
                        for (int e = 0; e < 3; ++e) {                 // fixed order
                            const float2 xe = S.xch[e][crow];
                            xs += xe.x; xg += xe.y;
                            if (HALF) { const float2 xf = S.xch[e][crow + 64]; xs += xf.x; xg += xf.y; }
                        }
                        named_bar_sync(xbar, xcnt);                   // single exchange buffer (shared memory is full): read before rewrite
                        const float alpha = expf(xs + S.ba - sm_m) * inv_l;
                        const float ds = alpha * xg;
#pragma unroll
                        for (int j = 0; j < kU; ++j) {
                            dh[j] = fmaf(alpha, dzr[j], ds * S.wa[u0 + j]);
                            if constexpr (!kDx) dwa[j] = fmaf(ds, hv[j], dwa[j]);
                        }
                        if constexpr (!kDx) dba += ds;
                    } else {
#pragma unroll
                        for (int j = 0; j < kU; j += 4) {
                            const float4 d4 = *reinterpret_cast<const float4*>(dh_in + tcl32x_off(t, ntiles, tile, gr0 + j / 4, row));
                            dh[j] = d4.x; dh[j + 1] = d4.y; dh[j + 2] = d4.z; dh[j + 3] = d4.w;
                        }
                    }
                }
                // ---- phase A (half tiles: registers to spare): the gates of step t have been in TMEM since the previous epilogue, so
                // everything that does not depend on dh_rec -- the 5 ex2 + 2 rcp per cell and the products around them -- is
                // evaluated while the tensor pipe runs R(t+1) (36 small MMAs: the epilogue warps were idle a third of the step).
                //   po = dh cA,  dct = dh cB + dc,  dc' = dct cGf,  (pi, pf, pg) = dct (cI, cF c_{t-1}, cG)
                constexpr bool kPre = HALF;
                const uint32_t tm_g = tmem + (i & 1) * kN;
                float cA[8], cB[8], cI[8], cF[8], cG[8], cGf[8];
                if (kPre && i < T) {
                    mbar_wait(&S.g_full[i & 1], gph[i & 1] & 1); ++gph[i & 1];
                    tc_fence_after();
                    uint32_t v[32];
                    tmem_ld32(tm_g + lane_base + gr0 * 16, v);
#pragma unroll
                    for (int gi = 0; gi < 2; ++gi)
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int j = gi * 4 + u;
                            float a_i, a_f, a_g, a_o, tcv;
                            gates_exact(__uint_as_float(v[gi * 16 + u]), __uint_as_float(v[gi * 16 + 4 + u]), __uint_as_float(v[gi * 16 + 8 + u]),
                                        __uint_as_float(v[gi * 16 + 12 + u]), ccur[j], a_i, a_f, a_g, a_o, tcv);
                            cA[j] = tcv * (a_o * (1.0f - a_o));
                            cB[j] = a_o * (1.0f - tcv * tcv);
                            cI[j] = a_g * (a_i * (1.0f - a_i));
                            cF[j] = a_f * (1.0f - a_f);
                            cG[j] = a_i * (1.0f - a_g * a_g);
                            cGf[j] = a_f;
                        }
                }
                mbar_wait(&S.r_full, rphase & 1); ++rphase;
                if (!kPre && i < T) { mbar_wait(&S.g_full[i & 1], gph[i & 1] & 1); ++gph[i & 1]; }
                tc_fence_after();
                if (i >= 1) {
                    if (LAYER == 1) {
                        // din of step t+1 = D_R[:, 0:48] (x dropout mask x scale) -> dh_in of layer 0
                        uint32_t r[kU];
                        if constexpr (HALF) tmem_ld8(tm_r + lane_base + u0, reinterpret_cast<uint32_t(&)[8]>(r));
                        else tmem_ld16(tm_r + lane_base + u0, reinterpret_cast<uint32_t(&)[16]>(r));
                        const int64_t grow = (int64_t)(t + 1) * Bp + b0 + crow;                          // mask-tensor row
                        const int64_t gkey = HALF ? (int64_t)(t + 1) * drop_stride + bwin : grow;        // counter-based generator
#pragma unroll
                        for (int pr = 0; pr < kNB; ++pr) {
                            float o[8];
                            if (mask || thresh16 < 65536u) {
                                const int blk = chunk0 + pr;
                                const uint32_t keep = mask ? mask_keep8(*reinterpret_cast<const uint2*>(mask + grow * kH + blk * 8))
                                                           : dropout_keep8(seed, gkey, blk, thresh16);
#pragma unroll
                                for (int u = 0; u < 8; ++u) o[u] = ((keep >> u) & 1u) ? __uint_as_float(r[pr * 8 + u]) * drop_scale : 0.f;
                            } else {
#pragma unroll
                                for (int u = 0; u < 8; ++u) o[u] = __uint_as_float(r[pr * 8 + u]);
                            }
                            *reinterpret_cast<float4*>(din + tcl32x_off(t + 1, ntiles, tile, gr0 + 2 * pr, row)) = make_float4(o[0], o[1], o[2], o[3]);
                            *reinterpret_cast<float4*>(din + tcl32x_off(t + 1, ntiles, tile, gr0 + 2 * pr + 1, row)) = make_float4(o[4], o[5], o[6], o[7]);
                        }
                    }
                    if (i < T) {
                        uint32_t r[kU];
                        if constexpr (HALF) tmem_ld8(tm_r + lane_base + kRecCol + u0, reinterpret_cast<uint32_t(&)[8]>(r));
                        else tmem_ld16(tm_r + lane_base + kRecCol + u0, reinterpret_cast<uint32_t(&)[16]>(r));
#pragma unroll
                        for (int j = 0; j < kU; ++j) dh[j] += __uint_as_float(r[j]);
                    }
                }
                if constexpr (kDx && LAYER == 0)
                    if (i == T) take_dx(0);
                if (i == T) break;
#pragma unroll
                for (int pr = 0; pr < kNB; ++pr) {
                    uint32_t v[32];
                    if (!kPre) tmem_ld32(tm_g + lane_base + (gr0 + 2 * pr) * 16, v);
#pragma unroll
                    for (int gi = 0; gi < 2; ++gi) {
                        float pi[4], pf[4], pg[4], po[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int j = pr * 8 + gi * 4 + u;
                            if (kPre) {                                // phase B: only the products with dh_t are left
                                const int jj = gi * 4 + u;             // (kNB == 1)
                                const float dct = fmaf(dh[j], cB[jj], dc[j]);
                                po[u] = dh[j] * cA[jj];
                                dc[j] = dct * cGf[jj];
                                pi[u] = dct * cI[jj];
                                pf[u] = dct * (cp[j] * cF[jj]);
                                pg[u] = dct * cG[jj];
                            } else {
                                float a_i, a_f, a_g, a_o, tcv;
                                gates_exact(__uint_as_float(v[gi * 16 + u]), __uint_as_float(v[gi * 16 + 4 + u]), __uint_as_float(v[gi * 16 + 8 + u]),
                                            __uint_as_float(v[gi * 16 + 12 + u]), ccur[j], a_i, a_f, a_g, a_o, tcv);
                                const float d_o = dh[j] * tcv;
                                const float dct = fmaf(dh[j] * a_o, 1.0f - tcv * tcv, dc[j]);
                                dc[j] = dct * a_f;
                                pi[u] = dct * a_g * a_i * (1.0f - a_i);
                                pf[u] = dct * cp[j] * a_f * (1.0f - a_f);
                                pg[u] = dct * a_i * (1.0f - a_g * a_g);
                                po[u] = d_o * a_o * (1.0f - a_o);
                            }
                            ccur[j] = cp[j];                           // c_{t-1} is the next iteration's c_t
                        }
                        // granule G -> columns 16 G .. 16 G + 15 = chunks 2 G ([i x4 | f x4]) and 2 G + 1 ([g x4 | o x4])
                        const int G = gr0 + 2 * pr + gi;
                        const float e0[8] = {pi[0], pi[1], pi[2], pi[3], pf[0], pf[1], pf[2], pf[3]};
                        const float e1[8] = {pg[0], pg[1], pg[2], pg[3], po[0], po[1], po[2], po[3]};
                        uint32_t hi[4], lo[4];
                        split_pack8(e0, hi, lo);
                        if constexpr (kDx && LAYER == 0)
                            if (i >= 1 && pr == 0 && gi == 0) take_dx(t + 1);      // before the first overwrite of S.dg
                        st_shared_v4(S.dg + (2 * G) * kAChunk + row * 16, hi[0], hi[1], hi[2], hi[3]);
                        st_shared_v4(S.dg + (24 + 2 * G) * kAChunk + row * 16, lo[0], lo[1], lo[2], lo[3]);
                        if (HALF) {
                            st_shared_v4(S.dg + (2 * G) * kAChunk + (row ^ 64) * 16, hi[0], hi[1], hi[2], hi[3]);
                            st_shared_v4(S.dg + (24 + 2 * G) * kAChunk + (row ^ 64) * 16, lo[0], lo[1], lo[2], lo[3]);
                        }
                        if constexpr (!kDx) {
                            *reinterpret_cast<uint4*>(dg_out + dgx_any<HALF>(t, ntiles, tile, 2 * G, crow)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                            *reinterpret_cast<uint4*>(dg_out + dgx_any<HALF>(t, ntiles, tile, 24 + 2 * G, crow)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        }
                        split_pack8(e1, hi, lo);
                        st_shared_v4(S.dg + (2 * G + 1) * kAChunk + row * 16, hi[0], hi[1], hi[2], hi[3]);
                        st_shared_v4(S.dg + (24 + 2 * G + 1) * kAChunk + row * 16, lo[0], lo[1], lo[2], lo[3]);
                        if (HALF) {
                            st_shared_v4(S.dg + (2 * G + 1) * kAChunk + (row ^ 64) * 16, hi[0], hi[1], hi[2], hi[3]);
                            st_shared_v4(S.dg + (24 + 2 * G + 1) * kAChunk + (row ^ 64) * 16, lo[0], lo[1], lo[2], lo[3]);
                        }
                        if constexpr (!kDx) {
                            *reinterpret_cast<uint4*>(dg_out + dgx_any<HALF>(t, ntiles, tile, 2 * G + 1, crow)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                            *reinterpret_cast<uint4*>(dg_out + dgx_any<HALF>(t, ntiles, tile, 24 + 2 * G + 1, crow)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        }
                    }
                }
                tc_fence_before();
                fence_proxy_async_smem();
                mbar_arrive(&S.dg_ready);
            }
        }
        __syncthreads();
    }

    // ---- per-CTA partial of d attn_w / d attn_b (fused head backward) ---------------------------------------------
    if (head && !kDx) {
        float* red = reinterpret_cast<float*>(S.dg);               // [12 warps][17]; every MMA has completed (tile-end barrier)
        if (warp < 12) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float v = warp_sum(j < (HALF ? 8 : 16) ? dwa[j] : 0.f);
                if (lane == 0) red[warp * 17 + j] = v;
            }
            const float vb = warp_sum(dba);
            if (lane == 0) red[warp * 17 + 16] = vb;
        }
        __syncthreads();
        if (!HALF) {
            if (tid < kH) {
                const int g = tid / 16, j = tid % 16;
                attn_partial[(size_t)blockIdx.x * 52 + tid] =
                    red[(4 * g) * 17 + j] + red[(4 * g + 1) * 17 + j] + red[(4 * g + 2) * 17 + j] + red[(4 * g + 3) * 17 + j];
            } else if (tid == kH) {
                attn_partial[(size_t)blockIdx.x * 52 + kH] = red[16] + red[17 + 16] + red[2 * 17 + 16] + red[3 * 17 + 16];
            }
        } else {
            // unit 8 chunk + j belongs to the warps (q, g) with g = chunk / 2 and q / 2 = chunk % 2; ds is the same in every
            // warp of a window: count it once (g = 0, copy 0 = quarters 0 and 1)
            if (tid < kH) {
                const int chunk = tid / 8, j = tid % 8, w0 = 4 * (chunk / 2) + 2 * (chunk % 2);
                attn_partial[(size_t)blockIdx.x * 52 + tid] = red[w0 * 17 + j] + red[(w0 + 1) * 17 + j];
            } else if (tid == kH) {
                attn_partial[(size_t)blockIdx.x * 52 + kH] = red[16] + red[17 + 16];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kTxTmaWarp) { tc_fence_after(); tmem_free_all(tmem); }
}

// ---------------------------------------------------------------------------------------------------------------
// weight gradients: dW^T[feature][gate column] = sum over (t, tile) of act^T . dG, both operands MN-major
// ---------------------------------------------------------------------------------------------------------------
constexpr int kWgThreads = 6 * 32;            // warps 0-3: final readout, 4: MMA issuer, 5: TMA producer
// Stages of [128 feature rows x K window rows] (act) and [64 gate columns x K] (one d(gates) column group).  Half tiles keep only
// the 64 real window rows of every chunk (1 KB instead of 2 KB), which buys twice the stages: with half-size stages and the same
// depth the kernel was latency-bound (bytes in flight), not HBM-bound.
template <bool HALF>
struct TxWgSmem {
    static constexpr int kChunkB = HALF ? kAChunk / 2 : kAChunk;
    static constexpr int kSt = HALF ? 4 : 2;
    alignas(128) unsigned char act[kSt][32 * kChunkB];   // hi block = chunks 0..15, lo block = chunks 16..31 (see below)
    alignas(128) unsigned char dg[kSt][16 * kChunkB];    // one 64-column group: hi x8 | lo x8
    alignas(8) uint64_t act_full[kSt], act_empty[kSt], dg_full[kSt], dg_empty[kSt];
    uint64_t done;
    uint32_t tmem_base;
};
// act stage, feature rows of the accumulator (M = 128 = 16 chunks):
//   L1: chunks 0-5 in_hi | 6-11 hprev_hi | 12 ones | 13-15 zeros ;  16-21 in_lo | 22-27 hprev_lo | 28-31 zeros
//   L0: chunk 0 x_hi | 1-6 hprev_hi | 7 ones | 8-15 zeros        ;  16 x_lo | 17-22 hprev_lo | 23-31 zeros
template <int LAYER, bool HALF>          // HALF: rows 64..127 of the slabs are copies (or unwritten): K = 64 window rows
__global__ void __launch_bounds__(kWgThreads, 1)
lstm_wgrad_x3_kernel(const __half* __restrict__ dg,       // DGX
                     const __half* __restrict__ act_in,   // L0: XS;  L1: TCLX
                     const __half* __restrict__ h,        // TCLX (this layer's h: h_{t-1} operand)
                     const __half* __restrict__ zeros,
                     float* __restrict__ partial,         // [grid][128][192]
                     int T, int ntiles) {
    using SM = TxWgSmem<HALF>;
    constexpr int kCB = SM::kChunkB, kSt = SM::kSt, kKRows = HALF ? 64 : kRows;
    constexpr int kInC = LAYER == 0 ? 1 : 6;              // hi chunks of the input
    constexpr int kOnesChunk = kInC + 6;
    constexpr uint32_t kIdescW = make_idesc(64, kFmtVal, kFmtVal, true, true);
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SM& S = *reinterpret_cast<SM*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    {
        const uint4 ones = make_uint4(kValOnes2 & 0xFFFFu, 0u, 0u, 0u), zero = make_uint4(0u, 0u, 0u, 0u);   // {1, 0, 0, ...}: one bias row
        for (int i = tid; i < kSt * 32 * kKRows; i += kWgThreads) {
            const int s = i / (32 * kKRows), ch = (i / kKRows) % 32, r = i % kKRows;
            reinterpret_cast<uint4*>(S.act[s] + ch * kCB)[r] = ch == kOnesChunk ? ones : zero;
        }
        if (tid == 0) {
            for (int s = 0; s < kSt; ++s) {
                mbar_init(&S.act_full[s], 1); mbar_init(&S.act_empty[s], 1);
                mbar_init(&S.dg_full[s], 1); mbar_init(&S.dg_empty[s], 1);
            }
            mbar_init(&S.done, 1);
            fence_mbar_init();
        }
        if (warp == 5) tmem_alloc_all(&S.tmem_base);
        tc_fence_before();
        fence_proxy_async_smem();
        __syncthreads();
        tc_fence_after();
    }
    const uint32_t tmem = __shfl_sync(0xffffffffu, S.tmem_base, 0);
    const int64_t nitems = (int64_t)T * ntiles;
    if (warp == 5) {
        if constexpr (HALF) {
            // half tiles: only rows 0..63 of every chunk carry windows (and only those were written by the backward kernel), so
            // the first 1 KB of each 2 KB chunk is fetched -- one bulk copy per chunk, spread over the lanes of this warp
            uint32_t k = 0, gk = 0;
            constexpr int kNAct = 2 * kInC + 12;
            for (int64_t w = blockIdx.x; w < nitems; w += gridDim.x, ++k) {
                const int t = (int)(w / ntiles), tile = (int)(w % ntiles);
                const uint32_t a = k % kSt;
                if (lane == 0) {
                    mbar_wait(&S.act_empty[a], ((k / kSt) & 1) ^ 1);
                    mbar_arrive_expect_tx(&S.act_full[a], kNAct * kCB);
                }
                __syncwarp();
                const __half* isrc = act_in + (((int64_t)t * ntiles + tile) * (2 * kInC)) * (kAChunk / 2);
                const __half* hsrc = t > 0 ? h + tclx_off(t - 1, ntiles, tile, 0, 0) : zeros;
                if (lane < kNAct) {
                    const int c = lane;                                    // source chunk: [in hi | in lo | h hi x6 | h lo x6]
                    const bool is_in = c < 2 * kInC;
                    const int cc = is_in ? c : c - 2 * kInC;               // chunk inside its slab
                    const bool lo = is_in ? cc >= kInC : cc >= 6;
                    const int dst = (lo ? 16 : 0) + (is_in ? (lo ? cc - kInC : cc) : kInC + (lo ? cc - 6 : cc));
                    bulk_load(S.act[a] + dst * kCB, (is_in ? isrc : hsrc) + cc * (kAChunk / 2), kCB, &S.act_full[a]);
                }
                for (int g = 0; g < 3; ++g, ++gk) {
                    const uint32_t r = gk % kSt;
                    if (lane == 0) {
                        mbar_wait(&S.dg_empty[r], ((gk / kSt) & 1) ^ 1);
                        mbar_arrive_expect_tx(&S.dg_full[r], 16 * kCB);
                        bulk_load(S.dg[r], dg + dgx_half_off(t, ntiles, tile, 8 * g, 0), 8 * kCB, &S.dg_full[r]);
                        bulk_load(S.dg[r] + 8 * kCB, dg + dgx_half_off(t, ntiles, tile, 24 + 8 * g, 0), 8 * kCB, &S.dg_full[r]);
                    }
                }
            }
        } else if (lane == 0) {   // (if constexpr: the full-size stage offsets below do not exist in the half-tile layout)
            uint32_t k = 0, gk = 0;
            for (int64_t w = blockIdx.x; w < nitems; w += gridDim.x, ++k) {
                const int t = (int)(w / ntiles), tile = (int)(w % ntiles);
                const uint32_t a = k % kSt;
                mbar_wait(&S.act_empty[a], ((k / kSt) & 1) ^ 1);
                mbar_arrive_expect_tx(&S.act_full[a], (2 * kInC + 12) * kAChunk);
                const __half* isrc = act_in + (((int64_t)t * ntiles + tile) * (2 * kInC)) * (kAChunk / 2);
                bulk_load(S.act[a], isrc, kInC * kAChunk, &S.act_full[a]);
                bulk_load(S.act[a] + 16 * kAChunk, isrc + kInC * (kAChunk / 2), kInC * kAChunk, &S.act_full[a]);
                const __half* hsrc = t > 0 ? h + tclx_off(t - 1, ntiles, tile, 0, 0) : zeros;
                bulk_load(S.act[a] + kInC * kAChunk, hsrc, 6 * kAChunk, &S.act_full[a]);
                bulk_load(S.act[a] + (16 + kInC) * kAChunk, hsrc + 6 * (kAChunk / 2), 6 * kAChunk, &S.act_full[a]);
                for (int g = 0; g < 3; ++g, ++gk) {
                    const uint32_t r = gk % kSt;
                    mbar_wait(&S.dg_empty[r], ((gk / kSt) & 1) ^ 1);
                    mbar_arrive_expect_tx(&S.dg_full[r], 16 * kAChunk);
                    bulk_load(S.dg[r], dg + dgx_off(t, ntiles, tile, 8 * g, 0), 8 * kAChunk, &S.dg_full[r]);
                    bulk_load(S.dg[r] + 8 * kAChunk, dg + dgx_off(t, ntiles, tile, 24 + 8 * g, 0), 8 * kAChunk, &S.dg_full[r]);
                }
            }
        }
    } else if (warp == 4) {
        const bool leader = elect_one();
        const uint64_t d_act0 = umma_desc(smem_u32(S.act[0]), 128, kCB);      // MN-major: chunk (8 feature rows) stride = kCB
        const uint64_t d_dg0 = umma_desc(smem_u32(S.dg[0]), 128, kCB);
        uint32_t k = 0, gk = 0;
        for (int64_t w = blockIdx.x; w < nitems; w += gridDim.x, ++k) {
            const uint32_t a = k % kSt;
            mbar_wait(&S.act_full[a], (k / kSt) & 1);
            const uint64_t d_act = desc_adv(d_act0, a * 32 * kCB);
            for (int g = 0; g < 3; ++g, ++gk) {
                const uint32_t r = gk % kSt;
                mbar_wait(&S.dg_full[r], (gk / kSt) & 1);
                tc_fence_after();
                const uint32_t td = tmem + 64 * g;
                const uint64_t d_dg = desc_adv(d_dg0, r * 16 * kCB);
#pragma unroll
                for (int ks = 0; ks < (HALF ? 4 : 8); ++ks)
                    if (leader) {
                        const uint64_t ahi = desc_adv(d_act, ks * 256), alo = desc_adv(d_act, 16 * kCB + ks * 256);
                        const uint64_t bhi = desc_adv(d_dg, ks * 256), blo = desc_adv(d_dg, 8 * kCB + ks * 256);
                        umma_bf16_i(td, ahi, bhi, kIdescW, (k == 0 && ks == 0) ? 0u : 1u);
                        umma_bf16_i(td, ahi, blo, kIdescW, 1u);
                        umma_bf16_i(td, alo, bhi, kIdescW, 1u);
                    }
                if (leader) umma_commit(&S.dg_empty[r]);
            }
            if (leader) umma_commit(&S.act_empty[a]);
        }
        if (leader) umma_commit(&S.done);
    } else {
        // ================= readout of this CTA's partial: lane = feature row, 192 gate columns =========================
        mbar_wait(&S.done, 0);
        tc_fence_after();
        const int row = warp * 32 + lane;
        const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
        float* out = partial + ((size_t)blockIdx.x * kRows + row) * kN;
        const bool any = (int64_t)blockIdx.x < nitems;          // a CTA without work items never wrote its accumulator
#pragma unroll 1
        for (int cc = 0; cc < kN; cc += 8) {
            uint32_t r[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
            if (any) tmem_ld8(tmem + lane_base + cc, r);
            *reinterpret_cast<float4*>(out + cc) = make_float4(__uint_as_float(r[0]), __uint_as_float(r[1]), __uint_as_float(r[2]), __uint_as_float(r[3]));
            *reinterpret_cast<float4*>(out + cc + 4) = make_float4(__uint_as_float(r[4]), __uint_as_float(r[5]), __uint_as_float(r[6]), __uint_as_float(r[7]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) { tc_fence_after(); tmem_free_all(tmem); }
}

// Sum the per-CTA partials [nparts][128 feature rows][192 permuted gate columns] in a fixed order, scatter to torch layouts.
__global__ void reduce_dw_x3_kernel(const float* __restrict__ partial, int nparts, int layer, float* __restrict__ dw_ih,
                                    float* __restrict__ dw_hh, float* __restrict__ db) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= kRows * kN) return;
    const int f = idx / kN, n = idx % kN;
    const int kin = layer == 0 ? 8 : kH;
    if (f > kin + kH) return;                                 // rows: [in (kin) | h_{t-1} (48) | bias | unused]
    float s = 0.f;
    for (int p = 0; p < nparts; ++p) s += partial[(size_t)p * kRows * kN + idx];
    const int j = (n / 16) * 4 + (n % 4), gate = (n % 16) / 4, col = gate * kH + j;      // torch row of the weight tensors
    if (f < kin) dw_ih[col * kin + f] = layer == 0 ? s * kX3XScaleInv : s;             // layer 0: the stored input is x / 16
    else if (f < kin + kH) dw_hh[col * kH + (f - kin)] = s;
    else db[col] = s;
}

static_assert(sizeof(TxFwdSmem<0>) <= 232448 && sizeof(TxFwdSmem<1>) <= 232448, "forward: shared memory budget (227 KB)");
static_assert(sizeof(TxBwdSmem<0>) <= 232448 && sizeof(TxBwdSmem<1>) <= 232448, "backward: shared memory budget (227 KB)");
static_assert(sizeof(TxWgSmem<false>) <= 232448 && sizeof(TxWgSmem<true>) <= 232448, "weight gradients: shared memory budget (227 KB)");

static int tx_sms() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

}  // namespace tc
}  // namespace na

// ---- C ABI ---------------------------------------------------------------------------------------------------
extern "C" int na_x3_split_input(const float* x, void* xs, int64_t B, int64_t T, int64_t Bp, int64_t half_stride, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(B >= 1 && T >= 1 && T < (1 << 20) && Bp >= B && Bp % tc::kRows == 0, NA_EINVAL,
               "na_x3_split_input: bad shape B=%lld T=%lld Bp=%lld (Bp must be a multiple of 128)", (long long)B, (long long)T, (long long)Bp);
    NA_REQUIRE(half_stride == 0 || B <= Bp / 2, NA_EINVAL, "na_x3_split_input: half tiles need B <= Bp / 2");
    NA_REQUIRE_PTR(x); NA_REQUIRE_PTR(xs);
    const int64_t nslots = half_stride ? Bp / 2 : Bp;                  // a multiple of 64
    const dim3 grid((unsigned)(nslots / 32), (unsigned)((T + 8 * tc::kSplitTC - 1) / (8 * tc::kSplitTC)));
    tc::x3_split_input_kernel<<<grid, 256, 0, as_stream(stream)>>>(x, reinterpret_cast<__half*>(xs), B, (int)T, Bp, half_stride ? 1 : 0);
    count_launch();
    return check_launch("na_x3_split_input");
}

extern "C" int na_lstm_fwd_train_x3(int64_t layer, const void* in, const void* packed_x3, const float* attn_w, const float* attn_b,
                                    const unsigned char* mask, uint64_t seed, int64_t thresh16, float drop_scale, void* h, void* hd,
                                    float* c, float* zpool, float* stats, int64_t B, int64_t T, int64_t Bp, int64_t half_stride,
                                    na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(layer == 0 || layer == 1, NA_EINVAL, "na_lstm_fwd_train_x3: layer must be 0 or 1");
    NA_REQUIRE(half_stride >= 0 && (half_stride == 0 || B <= Bp / 2), NA_EINVAL, "na_lstm_fwd_train_x3: half tiles need B <= Bp / 2");
    NA_REQUIRE(T >= 1 && T < (1 << 20) && Bp >= tc::kRows && Bp % tc::kRows == 0, NA_EINVAL,
               "na_lstm_fwd_train_x3: bad shape T=%lld Bp=%lld (Bp must be a multiple of 128)", (long long)T, (long long)Bp);
    NA_REQUIRE_PTR(in); NA_REQUIRE_PTR(packed_x3); NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(c);
    NA_OPTIONAL_PTR(mask); NA_OPTIONAL_PTR(hd); NA_OPTIONAL_PTR(zpool);
    NA_REQUIRE(thresh16 >= 0 && thresh16 <= 65536, NA_EINVAL, "na_lstm_fwd_train_x3: thresh16 outside [0,65536]");
    NA_REQUIRE(layer == 1 || (mask != nullptr || thresh16 < 65536) == (hd != nullptr), NA_EINVAL,
               "na_lstm_fwd_train_x3: layer 0 needs hd exactly when dropout is on (mask tensor or thresh16 < 65536)");
    NA_REQUIRE(layer == 0 || (attn_w && attn_b && zpool && stats && B >= 1 && B <= Bp), NA_EINVAL,
               "na_lstm_fwd_train_x3: layer 1 needs attn_w, attn_b, zpool, stats and 1 <= B <= Bp");
    const int ntiles = (int)(Bp / tc::kRows);
    const int grid = train_grid_cap(ntiles < tc::tx_sms() ? ntiles : tc::tx_sms());
    const unsigned char* pk = reinterpret_cast<const unsigned char*>(packed_x3) + (layer == 0 ? 0 : tc::kX3B0Chunks * tc::kBChunk);
    const int64_t dstride = half_stride > 0 ? half_stride : Bp;
#define NA_X3_FWD(L, HF)                                                                                                              \
    {                                                                                                                                \
        const size_t smem = sizeof(tc::TxFwdSmem<L>);                                                                                \
        cudaError_t e = cudaFuncSetAttribute(tc::lstm_fwd_x3_kernel<L, HF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e != cudaSuccess) return fail((int)e, "na_lstm_fwd_train_x3: shared memory opt-in failed (%s)", cudaGetErrorString(e));   \
        tc::lstm_fwd_x3_kernel<L, HF><<<grid, tc::kTxThreads, smem, as_stream(stream)>>>(                                           \
            reinterpret_cast<const __half*>(in), pk, L == 0 ? nullptr : attn_w, L == 0 ? nullptr : attn_b, L == 0 ? mask : nullptr,   \
            L == 0 ? seed : 0, L == 0 ? (uint32_t)thresh16 : 65536u, L == 0 ? drop_scale : 1.0f, reinterpret_cast<__half*>(h),        \
            L == 0 ? reinterpret_cast<__half*>(hd) : nullptr, c, L == 0 ? nullptr : zpool, L == 0 ? nullptr : stats, B, (int)T, Bp,   \
            ntiles, dstride);                                                                                                        \
    }
    if (layer == 0) { if (half_stride > 0) NA_X3_FWD(0, true) else NA_X3_FWD(0, false) }
    else { if (half_stride > 0) NA_X3_FWD(1, true) else NA_X3_FWD(1, false) }
#undef NA_X3_FWD
    count_launch();
    return check_launch("na_lstm_fwd_train_x3");
}

extern "C" int64_t na_train_x3_smem_bytes(int64_t which) {     // 0/1: forward L0/L1, 2/3: backward L0/L1, 4: weight gradients
    switch (which) {
        case 0: return sizeof(na::tc::TxFwdSmem<0>);
        case 1: return sizeof(na::tc::TxFwdSmem<1>);
        case 2: return sizeof(na::tc::TxBwdSmem<0>);
        case 3: return sizeof(na::tc::TxBwdSmem<1>);
        default: return sizeof(na::tc::TxWgSmem<true>) > sizeof(na::tc::TxWgSmem<false>) ? sizeof(na::tc::TxWgSmem<true>) : sizeof(na::tc::TxWgSmem<false>);
    }
}

extern "C" int64_t na_train_x3_scratch_floats(void) {
    const int64_t sms = na::tc::tx_sms();
    return sms * 52 + sms * na::tc::kRows * na::tc::kN;      // attention partials, then weight-gradient partials
}

namespace {
// One launch of lstm_bwd_x3_kernel<layer, half, kDx> (its arguments checked by the caller).
template <bool kDx>
int launch_bwd_x3(const char* name, int64_t layer, const void* act_in, const void* h, const float* cstate, const float* dh_in,
                  const void* packed_x3, const void* zeros, const unsigned char* in_mask, uint64_t seed, int64_t thresh16,
                  float drop_scale, float* din, void* dg, const float* dz, const float* stats, const float* zpool,
                  const float* attn_w, const float* attn_b, int64_t B, float* attn_partial, float* dx, const float* dx_scale,
                  int64_t T, int64_t Bp, int64_t half_stride, cudaStream_t st, int* grid_out) {
    using namespace na;
    const int ntiles = (int)(Bp / tc::kRows);
    const int grid = train_grid_cap(ntiles < tc::tx_sms() ? ntiles : tc::tx_sms());
    const unsigned char* pk = reinterpret_cast<const unsigned char*>(packed_x3) + (layer == 0 ? 0 : tc::kX3B0Chunks * tc::kBChunk);
    const int64_t dstride = half_stride > 0 ? half_stride : Bp;
#define NA_X3_BWD(L, HF)                                                                                                              \
    {                                                                                                                                \
        const size_t smem = sizeof(tc::TxBwdSmem<L>);                                                                                \
        cudaError_t e = cudaFuncSetAttribute(tc::lstm_bwd_x3_kernel<L, HF, kDx>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e != cudaSuccess) return fail((int)e, "%s: shared memory opt-in (%zu B) failed: %s", name, smem, cudaGetErrorString(e)); \
        tc::lstm_bwd_x3_kernel<L, HF, kDx><<<grid, tc::kTxThreads, smem, st>>>(                                                      \
            reinterpret_cast<const __half*>(act_in), reinterpret_cast<const __half*>(h), cstate, dh_in, pk,                           \
            reinterpret_cast<const __half*>(zeros), L == 0 ? nullptr : in_mask, L == 0 ? 0 : seed, L == 0 ? 65536u : (uint32_t)thresh16, \
            L == 0 ? 1.0f : drop_scale, L == 0 ? nullptr : din, reinterpret_cast<__half*>(dg), L == 0 ? nullptr : dz,                 \
            L == 0 ? dx_scale : stats, L == 0 ? nullptr : zpool, L == 0 ? nullptr : attn_w, L == 0 ? nullptr : attn_b, B,           \
            L == 0 ? dx : attn_partial, (int)T, Bp, ntiles, dstride);                                                                \
    }
    if (layer == 0) { if (half_stride > 0) NA_X3_BWD(0, true) else NA_X3_BWD(0, false) }
    else { if (half_stride > 0) NA_X3_BWD(1, true) else NA_X3_BWD(1, false) }
#undef NA_X3_BWD
    count_launch();
    *grid_out = grid;
    return check_launch(name);
}
}  // namespace

extern "C" int na_lstm_bwd_x3(int64_t layer, const void* act_in, const void* h, const float* cstate, const float* dh_in,
                              const void* packed_x3, const void* zeros, const unsigned char* in_mask, uint64_t seed, int64_t thresh16,
                              float drop_scale, float* din, void* dg, const float* dz, const float* stats, const float* zpool,
                              const float* attn_w, const float* attn_b, int64_t B, float* d_attn, float* scratch,
                              int64_t T, int64_t Bp, int64_t half_stride, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(layer == 0 || layer == 1, NA_EINVAL, "na_lstm_bwd_x3: layer must be 0 or 1");
    NA_REQUIRE(half_stride >= 0 && (half_stride == 0 || layer == 0 || dz != nullptr), NA_EUNSUPPORTED,
               "na_lstm_bwd_x3: half tiles need the fused head backward on layer 1");
    NA_REQUIRE(T >= 1 && T < (1 << 20) && Bp >= tc::kRows && Bp % tc::kRows == 0, NA_EINVAL,
               "na_lstm_bwd_x3: bad shape T=%lld Bp=%lld", (long long)T, (long long)Bp);
    NA_REQUIRE_PTR(act_in); NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(cstate); NA_REQUIRE_PTR(packed_x3); NA_REQUIRE_PTR(zeros);
    NA_REQUIRE_PTR(dg); NA_REQUIRE_PTR(scratch);
    NA_OPTIONAL_PTR(dh_in); NA_OPTIONAL_PTR(dz); NA_OPTIONAL_PTR(in_mask); NA_OPTIONAL_PTR(din);
    NA_REQUIRE((dz != nullptr) != (dh_in != nullptr), NA_EINVAL, "na_lstm_bwd_x3: give exactly one of dh_in and dz");
    NA_REQUIRE(dz == nullptr || (layer == 1 && stats && zpool && attn_w && attn_b && d_attn && B >= 1 && B <= Bp), NA_EINVAL,
               "na_lstm_bwd_x3: the fused head backward is for layer 1 and needs stats, zpool, attn_w, attn_b, d_attn, B");
    NA_REQUIRE(layer == 0 || din != nullptr, NA_EINVAL, "na_lstm_bwd_x3: layer 1 needs din");
    NA_REQUIRE(thresh16 >= 0 && thresh16 <= 65536, NA_EINVAL, "na_lstm_bwd_x3: thresh16 outside [0,65536]");
    cudaStream_t st = as_stream(stream);
    float* attn_partial = scratch;
    int grid = 0;
    int rc = launch_bwd_x3<false>("na_lstm_bwd_x3", layer, act_in, h, cstate, dh_in, packed_x3, zeros, in_mask, seed, thresh16,
                                  drop_scale, din, dg, dz, stats, zpool, attn_w, attn_b, B, attn_partial, nullptr, nullptr, T, Bp,
                                  half_stride, st, &grid);
    if (rc) return rc;
    if (dz != nullptr) return reduce_partials(attn_partial, d_attn, grid, 52, st);
    return NA_OK;
}

extern "C" int na_lstm_bwd_x3_dx(int64_t layer, const void* act_in, const void* h, const float* cstate, const float* dh_in,
                                 const void* packed_x3, const void* zeros, const unsigned char* in_mask, uint64_t seed,
                                 int64_t thresh16, float drop_scale, float* din, const float* dz, const float* stats,
                                 const float* zpool, const float* attn_w, const float* attn_b, int64_t B, float* dx,
                                 const float* dz_inv_scale, int64_t T, int64_t Bp, int64_t half_stride, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(layer == 0 || layer == 1, NA_EINVAL, "na_lstm_bwd_x3_dx: layer must be 0 or 1");
    NA_REQUIRE(half_stride >= 0 && (half_stride == 0 || layer == 0 || dz != nullptr), NA_EUNSUPPORTED,
               "na_lstm_bwd_x3_dx: half tiles need the fused head backward on layer 1");
    NA_REQUIRE(half_stride == 0 || B <= Bp / 2, NA_EINVAL, "na_lstm_bwd_x3_dx: half tiles need B <= Bp / 2");
    NA_REQUIRE(T >= 1 && T < (1 << 20) && Bp >= tc::kRows && Bp % tc::kRows == 0, NA_EINVAL,
               "na_lstm_bwd_x3_dx: bad shape T=%lld Bp=%lld", (long long)T, (long long)Bp);
    NA_REQUIRE_PTR(act_in); NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(cstate); NA_REQUIRE_PTR(packed_x3); NA_REQUIRE_PTR(zeros);
    NA_OPTIONAL_PTR(dh_in); NA_OPTIONAL_PTR(dz); NA_OPTIONAL_PTR(in_mask); NA_OPTIONAL_PTR(din);
    NA_OPTIONAL_PTR(dx); NA_OPTIONAL_PTR(dz_inv_scale);
    NA_REQUIRE((dz != nullptr) != (dh_in != nullptr), NA_EINVAL, "na_lstm_bwd_x3_dx: give exactly one of dh_in and dz");
    NA_REQUIRE(dz == nullptr || (layer == 1 && stats && zpool && attn_w && attn_b), NA_EINVAL,
               "na_lstm_bwd_x3_dx: the fused head backward is for layer 1 and needs stats, zpool, attn_w, attn_b");
    NA_REQUIRE(B >= 1 && B <= Bp, NA_EINVAL, "na_lstm_bwd_x3_dx: need 1 <= B <= Bp, got B=%lld Bp=%lld", (long long)B, (long long)Bp);
    NA_REQUIRE(layer == 0 || din != nullptr, NA_EINVAL, "na_lstm_bwd_x3_dx: layer 1 needs din");
    NA_REQUIRE(layer == 1 || (dx != nullptr && dz_inv_scale != nullptr), NA_EINVAL, "na_lstm_bwd_x3_dx: layer 0 needs dx and dz_inv_scale");
    NA_REQUIRE(thresh16 >= 0 && thresh16 <= 65536, NA_EINVAL, "na_lstm_bwd_x3_dx: thresh16 outside [0,65536]");
    int grid = 0;
    return launch_bwd_x3<true>("na_lstm_bwd_x3_dx", layer, act_in, h, cstate, dh_in, packed_x3, zeros, in_mask, seed, thresh16,
                               drop_scale, din, nullptr, dz, stats, zpool, attn_w, attn_b, B, nullptr, dx, dz_inv_scale, T, Bp,
                               half_stride, as_stream(stream), &grid);
}

extern "C" int na_lstm_wgrad_x3(int64_t layer, const void* dg, const void* act_in, const void* h, const void* zeros,
                                float* dw_ih, float* dw_hh, float* db, float* scratch, int64_t T, int64_t Bp, int64_t half_stride,
                                na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(layer == 0 || layer == 1, NA_EINVAL, "na_lstm_wgrad_x3: layer must be 0 or 1");
    NA_REQUIRE(T >= 1 && T < (1 << 20) && Bp >= tc::kRows && Bp % tc::kRows == 0, NA_EINVAL,
               "na_lstm_wgrad_x3: bad shape T=%lld Bp=%lld", (long long)T, (long long)Bp);
    NA_REQUIRE_PTR(dg); NA_REQUIRE_PTR(act_in); NA_REQUIRE_PTR(h); NA_REQUIRE_PTR(zeros);
    NA_REQUIRE_PTR(dw_ih); NA_REQUIRE_PTR(dw_hh); NA_REQUIRE_PTR(db); NA_REQUIRE_PTR(scratch);
    cudaStream_t st = as_stream(stream);
    const int ntiles = (int)(Bp / tc::kRows);
    const int64_t nitems = T * ntiles;
    const int grid = train_grid_cap((int)(nitems < tc::tx_sms() ? nitems : tc::tx_sms()));
    float* partial = scratch + (size_t)tc::tx_sms() * 52;
    const size_t smem = half_stride > 0 ? sizeof(tc::TxWgSmem<true>) : sizeof(tc::TxWgSmem<false>);
#define NA_X3_WG(L, HF)                                                                                                               \
    {                                                                                                                                \
        cudaError_t e = cudaFuncSetAttribute(tc::lstm_wgrad_x3_kernel<L, HF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e != cudaSuccess) return fail((int)e, "na_lstm_wgrad_x3: shared memory opt-in failed (%s)", cudaGetErrorString(e));       \
        tc::lstm_wgrad_x3_kernel<L, HF><<<grid, tc::kWgThreads, smem, st>>>(                                                          \
            reinterpret_cast<const __half*>(dg), reinterpret_cast<const __half*>(act_in), reinterpret_cast<const __half*>(h),         \
            reinterpret_cast<const __half*>(zeros), partial, (int)T, ntiles);                                                         \
    }
    if (layer == 0) { if (half_stride > 0) NA_X3_WG(0, true) else NA_X3_WG(0, false) }
    else { if (half_stride > 0) NA_X3_WG(1, true) else NA_X3_WG(1, false) }
#undef NA_X3_WG
    count_launch();
    int rc = check_launch("na_lstm_wgrad_x3");
    if (rc) return rc;
    tc::reduce_dw_x3_kernel<<<(tc::kRows * tc::kN + 255) / 256, 256, 0, st>>>(partial, grid, (int)layer, dw_ih, dw_hh, db);
    count_launch();
    return check_launch("na_lstm_wgrad_x3(reduce)");
}
