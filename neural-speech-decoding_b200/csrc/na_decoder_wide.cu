// Tensor-core tier for WIDE hidden sizes (H = 96, 144, 192; BASELINE configs[4] "stress": H = 192, T = 2500):
// the whole 2-layer decoder forward x -> logits/probs in one persistent tcgen05 / TMEM / TMA kernel.
//
// What changes against the H = 48 kernel (na_decoder_tc2.cu) and why:
//   * [W_ih | b | W_hh] of both layers is 0.93 MB of fp16 at H = 192 -- it cannot stay resident in the 227 KB of
//     shared memory of an SM (the "W_hh SMEM residency limit" the stress config is about).  What IS resident is
//     every activation operand: three rotating A buffers [H/8][128][8] fp16 hold h0_{t-1} / h0_t / h1_{t-1} / h1_t
//     (each step retires one version), so the recurrent state never leaves the SM.  The weights are STREAMED:
//     a TMA producer warp walks the packed weight image (laid out in exactly the order the MMAs consume it, so every
//     ring stage is one contiguous 12 KB cp.async.bulk) through a 4-stage shared-memory ring, every step.  The
//     image stays L2-resident (126 MB L2), so the stream is L2 -> SMEM traffic, not HBM.
//   * The gate accumulator of one layer is [128 x 4H] = 768 fp32 columns > the 512 TMEM columns, so a layer step is
//     cut into NCH = H/48 unit-chunk TASKS of N = 192 gate columns (48 units x 4 gates, granule-permuted as in v2);
//     TMEM holds two task accumulators (double buffer): the MMAs of task i+1 run while the epilogue warps
//     (12 warps: lane quarter x 16-unit group) apply the cell update of task i.
//     Task order of step t: L0 chunks 0..NCH-1, then L1 chunks 0..NCH-1.  L1's K order is
//     [bias | h1_{t-1} | h0_t chunk 0 .. NCH-1], so only its last slices wait for the last layer-0 epilogue.
//   * Cell state c0, c1 and the attention-pool accumulator z (128 x 384 + 128 x 192 fp32 per tile = 288 KB) fit
//     neither registers nor shared memory: they live in a per-CTA global workspace that stays L2-resident, are
//     prefetched before the accumulator wait and written back after the update (coalesced 16 B per lane).
//   * Attention score (lstm_eeg_model.py:35): as in v2 it is computed by the tensor core, one step late, from the
//     recurrent operand -- here by small N = 16 MMAs against a resident score operand, into columns 192..207 of
//     the accumulator of task L1.chunk0 -- and the online softmax pooling of step t-1 reads h1_{t-1} back from
//     its A buffer.  One flush round after the last step delivers the last score.
//   * Head (LayerNorm, fc0, RReLU(eval), fc3, softmax): per window, once per tile, from a shared-memory scratch
//     that re-uses the A buffers; fc0 weights are read from global memory (warp-uniform, L1-resident).
// Roofline at H = 192 (per 128-window tile step): tensor 4 x (13 + 25) MMAs x 96 cycles = 14.6 k cycles, MUFU
// 128 x 384 x 5 / 16 = 15.4 k cycles, L2 -> SM 0.93 MB weights + 0.59 MB state.  DESIGN.md section 5b.
#include "na_tc_common.cuh"

namespace na {
namespace tc {

constexpr int kWThreads = 14 * 32;
constexpr int kWXStages = 2;
#ifndef NA_WIDE_RING
#define NA_WIDE_RING 4
#endif
#ifndef NA_WIDE_SPS
#define NA_WIDE_SPS 2
#endif
constexpr int kWRing = NA_WIDE_RING;           // weight ring stages
constexpr int kWSps = NA_WIDE_SPS;             // K16 slices per ring stage (one mbarrier round trip per stage)
constexpr int kWSlice = kN * 32;               // bytes of one K16 weight slice: [2 K-chunks][192 rows][8] fp16 = 6,144
constexpr int kWStage = kWSps * kWSlice;
constexpr int kWD = 208;                       // TMEM columns per task accumulator (192 gates + 16 score)
constexpr int kWFc = NA_FC_HIDDEN;
constexpr uint32_t kIdesc16 = make_idesc(16, kFmtVal, kFmtVal);

template <int NCH>
struct WideCfg {
    static constexpr int H = 48 * NCH;
    static constexpr int kHC = H / 8;                    // K-chunks (8 units) of a hidden vector
    static constexpr int kHS = H / 16;                   // K16 slices of a hidden vector
    static constexpr int kABuf = kHC * kAChunk;          // bytes of one A buffer
    static constexpr int kSl0 = 1 + kHS;                 // slices of a layer-0 task: [x | ones], h0_{t-1}
    static constexpr int kSl1 = 1 + 2 * kHS;             // slices of a layer-1 task: [ones | 0], h1_{t-1}, h0_t
    static constexpr int kScoreSlices = 1 + kHS;         // score operand: [ones | 0], h1 slices
    static constexpr int64_t kStepBytes = (int64_t)NCH * (kSl0 + kSl1) * kWSlice;      // streamed per step
    static constexpr int64_t kScoreBytes = (int64_t)kScoreSlices * 2 * 16 * 16;        // [slice][2 chunks][16 rows][8]
    static constexpr int64_t kPackedBytes = kStepBytes + kScoreBytes;
    static constexpr int64_t kStateFloats = (int64_t)NCH * 3 * 4 * kRows * 4;          // one state array of a CTA
};

template <int NCH>
struct WideSmem {
    using C = WideCfg<NCH>;
    alignas(128) unsigned char p[3][C::kABuf];               // rotating A buffers (H = 192: 3 x 49,152)
    alignas(128) unsigned char ring[kWRing][kWStage];        // streamed weights, 4 x 12,288
    alignas(128) unsigned char x[kWXStages][2 * kAChunk];    // [x chunk | ones chunk]
    alignas(128) unsigned char onez[2 * kAChunk];            // [ones | zeros]
    alignas(128) unsigned char bscore[C::kScoreSlices * 512];
    float lnw[C::H], lnb[C::H];
    float b0[kWFc], w3[NA_MAX_CLASSES * kWFc], b3[NA_MAX_CLASSES];
    alignas(8) uint64_t x_full[kWXStages], x_empty[kWXStages];
    uint64_t b_full[kWRing], b_empty[kWRing];
    uint64_t d_full[2], d_empty[2];
    uint64_t a_ready[2][NCH];                                // [layer][chunk]: H chunk of this step written
    uint32_t tmem_base;
};

// ---- weight image ----------------------------------------------------------------------------------------
// Stream order = task order (L0 chunk 0..NCH-1, L1 chunk 0..NCH-1), slices in K order, each slice
// [2 K-chunks][192 rows][8] fp16 with row n = (jj/4)*16 + gate*4 + jj%4 of chunk-local unit jj; then the score
// operand.  Pre-scaling as in v2: i,f,o rows x 0.5 (sigmoid via tanh), hidden-state columns x 0.5 (H = 2h).
template <int NCH>
__global__ void pack_wide_kernel(const float* __restrict__ w_ih0, const float* __restrict__ w_hh0,
                                 const float* __restrict__ b_ih0, const float* __restrict__ b_hh0,
                                 const float* __restrict__ w_ih1, const float* __restrict__ w_hh1,
                                 const float* __restrict__ b_ih1, const float* __restrict__ b_hh1,
                                 const float* __restrict__ attn_w, const float* __restrict__ attn_b,
                                 uint16_t* __restrict__ out) {
    using C = WideCfg<NCH>;
    constexpr int H = C::H;
    constexpr int per_slice = kWSlice / 2;                       // fp16 elements
    constexpr int n_stream = (int)(C::kStepBytes / 2), n_score = (int)(C::kScoreBytes / 2);
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n_stream + n_score; idx += gridDim.x * blockDim.x) {
        float v = 0.f;
        if (idx < n_stream) {
            int sl = idx / per_slice;                            // global slice index within the step
            const int e = idx % per_slice;
            const int kc = e / (kN * 8), n = (e / 8) % kN, kk = e % 8;
            int layer, chunk, s;
            if (sl < NCH * C::kSl0) { layer = 0; chunk = sl / C::kSl0; s = sl % C::kSl0; }
            else { sl -= NCH * C::kSl0; layer = 1; chunk = sl / C::kSl1; s = sl % C::kSl1; }
            const int jj = (n / 16) * 4 + (n % 4), gate = (n % 16) / 4;
            const int row = gate * H + chunk * 48 + jj;          // row of the torch weight tensors
            const float gs = (gate == 2) ? 1.0f : 0.5f, hs = 0.5f * gs;
            const int k = kc * 8 + kk;                           // 0..15 within the slice
            if (layer == 0) {
                if (s == 0) {
                    const float b = gs * (b_ih0[row] + b_hh0[row]);
                    const float bh = val16_to_float(val16(b));
                    if (k < 8) v = gs * kF16InScaleInv * w_ih0[row * 8 + k];      // x is stored as x / 16
                    else if (k == 8) v = bh;
                    else if (k == 9) v = b - bh;
                } else v = hs * w_hh0[row * H + (s - 1) * 16 + k];
            } else {
                if (s == 0) {
                    const float b = gs * (b_ih1[row] + b_hh1[row]);
                    const float bh = val16_to_float(val16(b));
                    if (k == 0) v = bh;
                    else if (k == 1) v = b - bh;
                } else if (s <= C::kHS) v = hs * w_hh1[row * H + (s - 1) * 16 + k];
                else v = hs * w_ih1[row * H + (s - 1 - C::kHS) * 16 + k];
            }
        } else {
            const int e = idx - n_stream;                        // [slice][2][16 rows][8]
            const int s = e / 256, kc = (e / 128) % 2, r = (e / 8) % 16, kk = e % 8;
            const int k = kc * 8 + kk;
            if (r < 2) {
                float full = 0.f;
                if (s == 0) full = (k == 0) ? attn_b[0] : 0.f;
                else full = 0.5f * attn_w[(s - 1) * 16 + k];     // multiplies H1 = 2 h1
                const float hi = val16_to_float(val16(full));
                v = (r == 0) ? hi : full - hi;
            }
        }
        out[idx] = val16(v);
    }
}

// ---- thread-block-cluster helpers (weight-stream multicast) ---------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// 1-D TMA bulk copy global -> the SAME shared-memory offset of every CTA in cta_mask; each destination CTA's
// mbarrier (same offset) receives the complete_tx bytes.
__device__ __forceinline__ void bulk_load_mc(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
        : "memory");
}
// tcgen05.commit that arrives on the mbarrier at this offset in every CTA of cta_mask
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}

__device__ __forceinline__ void w_tmem_ld2(uint32_t taddr, uint32_t (&v)[2]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(v[0]), "=r"(v[1]) : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// cell update of 4 units (granule); v = [i x4 | f x4 | g x4 | o x4] (i, f, o pre-halved); H = 2h as 2 x fp16x2
__device__ __forceinline__ void w_cell_granule(const uint32_t* v, float* c, uint32_t* hp) {
    float h[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float ti = tanh_apx(__uint_as_float(v[u]));
        const float tf = tanh_apx(__uint_as_float(v[4 + u]));
        const float tg = tanh_apx(__uint_as_float(v[8 + u]));
        const float to = tanh_apx(__uint_as_float(v[12 + u]));
        const float w = fmaf(tf, c[u], c[u]);
        const float uu = fmaf(ti, tg, tg);
        c[u] = 0.5f * (w + uu);
        const float tcell = tanh_apx(c[u]);
        h[u] = fmaf(to, tcell, tcell);
    }
    hp[0] = pack_val(h[0], h[1]);
    hp[1] = pack_val(h[2], h[3]);
}

__device__ __forceinline__ uint4 ld_shared_v4(const void* p) {
    uint4 r;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(smem_u32(p)));
    return r;
}

// kEx: also store the attention scores (time-major [T][B]) and the pooled vector / LayerNorm output ([B][H]) of every
// window b < B, in the reference's scale (h, not H = 2h); the g == 0 warp of the window's lane quarter writes them.
template <int NCH, bool kEx = false>
__global__ void __launch_bounds__(kWThreads, 1)
decoder_infer_wide_kernel(const __nv_bfloat16* __restrict__ x,        // TMP [T][Bp][8] fp16 bits
                          const unsigned char* __restrict__ packed,   // pack_wide_kernel image
                          const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                          const float* __restrict__ fc0_w, const float* __restrict__ fc0_b,
                          const float* __restrict__ fc3_w, const float* __restrict__ fc3_b,
                          float* __restrict__ state,                  // [grid][3][kStateFloats]: c0, c1, z
                          float* __restrict__ logits, float* __restrict__ probs,
                          int T, int64_t B, int64_t Bp, int NC, int nquarters, int cs, int dbg,
                          float* __restrict__ scores_tm,              // kEx: [T][B] scores, [B][H] pooled / LayerNorm output
                          float* __restrict__ pooled, float* __restrict__ embedding) {
    // dbg (timing experiments only, results invalid): 1 = skip the cell update, 2 = skip the gate MMAs, 4 = skip the weight loads
    // cs = thread-block-cluster size (1, 2 or 4): the CTAs of a cluster stream the SAME weight image in lockstep, so
    // each ring stage is fetched from L2 once per cluster -- rank r loads 1/cs of it and multicasts it to all.
    using C = WideCfg<NCH>;
    constexpr int H = C::H;
    constexpr int kMmaWarp = 12, kTmaWarp = 13;
    constexpr int kTasks = 2 * NCH;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    WideSmem<NCH>& S = *reinterpret_cast<WideSmem<NCH>*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    // warp index through a shuffle: tells the compiler it is warp-uniform, so the role branches below are uniform
    // control flow and the MMA / TMA descriptors are computed on the uniform datapath
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);

    // ---- one-time setup --------------------------------------------------------------------------
    {
        const uint4* sc = reinterpret_cast<const uint4*>(packed + C::kStepBytes);
        for (int i = tid; i < (int)(C::kScoreBytes / 16); i += kWThreads) reinterpret_cast<uint4*>(S.bscore)[i] = sc[i];
        const uint4 ones = make_uint4(kValOnes2, 0u, 0u, 0u);     // fp16 {1,1,0,0,0,0,0,0}
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        for (int i = tid; i < kRows; i += kWThreads) {
#pragma unroll
            for (int s = 0; s < kWXStages; ++s) reinterpret_cast<uint4*>(S.x[s] + kAChunk)[i] = ones;
            reinterpret_cast<uint4*>(S.onez)[i] = ones;
            reinterpret_cast<uint4*>(S.onez + kAChunk)[i] = zero;
        }
        for (int i = tid; i < H; i += kWThreads) { S.lnw[i] = ln_w[i]; S.lnb[i] = ln_b[i]; }
        for (int i = tid; i < kWFc; i += kWThreads) S.b0[i] = fc0_b[i];
        for (int i = tid; i < NC * kWFc; i += kWThreads) S.w3[i] = fc3_w[i];
        for (int i = tid; i < NC; i += kWThreads) S.b3[i] = fc3_b[i];
        if (tid == 0) {
            for (int s = 0; s < kWXStages; ++s) { mbar_init(&S.x_full[s], 1); mbar_init(&S.x_empty[s], 1); }
            for (int s = 0; s < kWRing; ++s) { mbar_init(&S.b_full[s], 1); mbar_init(&S.b_empty[s], cs); }     // every CTA's consumer releases it
            for (int s = 0; s < 2; ++s) { mbar_init(&S.d_full[s], 1); mbar_init(&S.d_empty[s], 384); }
            for (int l = 0; l < 2; ++l)
                for (int j = 0; j < NCH; ++j) mbar_init(&S.a_ready[l][j], 384);
            fence_mbar_init();
        }
        if (warp == kTmaWarp) tmem_alloc_all(&S.tmem_base);
        tc_fence_before();
        fence_proxy_async_smem();
        __syncthreads();
        tc_fence_after();
        if (cs > 1) cluster_sync_all();             // peers' mbarriers are initialised before anything is multicast to them
    }
    const uint32_t tmem = __shfl_sync(0xffffffffu, S.tmem_base, 0);
    const uint32_t crank = cs > 1 ? cluster_ctarank() : 0u;
    const uint16_t cmask = (uint16_t)((1u << cs) - 1u);

    // Tiles of 4 quarters (128 windows), strided over the CTAs; EVERY CTA runs the same number of rounds (the CTAs
    // of a cluster share the weight ring in lockstep) -- a CTA without a tile runs an idle round (nq = 0).
    const int ntiles = (nquarters + 3) / 4;
    const int rounds = (ntiles + (int)gridDim.x - 1) / (int)gridDim.x;
    int n0 = 0;                 // running step index across tiles (A-buffer rotation, a_ready / x parities)
    uint32_t tg = 0;            // running task index (accumulator double buffer; + 1 flush round per tile)
    uint32_t gi = 0;            // running ring-stage index
    for (int rd = 0; rd < rounds; ++rd, n0 += T) {
        const int tile = rd * (int)gridDim.x + (int)blockIdx.x;
        const int q0 = tile * 4;
        const int nq = tile < ntiles ? min(4, nquarters - q0) : 0;
        const uint32_t x_bytes = (uint32_t)nq * 32u * 16u;
        const int64_t b0 = (int64_t)q0 * 32;
        // ---- h0_{-1} = h1_{-1} = 0: clear the A buffers -------------------------------------------------
        {
            uint4* z = reinterpret_cast<uint4*>(S.p[0]);
            for (int i = tid; i < 3 * C::kABuf / 16; i += kWThreads) z[i] = make_uint4(0, 0, 0, 0);
            fence_proxy_async_smem();
            __syncthreads();
        }

        if (warp == kTmaWarp) {
            // ================= TMA producer: x_t and the weight stream ===================================
            if (lane == 0) {
                for (int t = 0; t < T; ++t) {
                    const int n = n0 + t, sx = n % kWXStages, ux = n / kWXStages;
                    mbar_wait(&S.x_empty[sx], (ux & 1) ^ 1);
                    if (x_bytes) {
                        mbar_arrive_expect_tx(&S.x_full[sx], x_bytes);
                        bulk_load(S.x[sx], x + ((int64_t)t * Bp + b0) * 8, x_bytes, &S.x_full[sx]);
                    } else mbar_arrive(&S.x_full[sx]);              // idle round
                    const unsigned char* src = packed;
                    for (int task = 0; task < kTasks; ++task) {
                        const int nsl = task < NCH ? C::kSl0 : C::kSl1;
                        for (int s = 0; s < nsl; s += kWSps, ++gi) {
                            const uint32_t bytes = (uint32_t)min(kWSps, nsl - s) * kWSlice;
                            const int sb = gi % kWRing;
                            mbar_wait(&S.b_empty[sb], ((gi / kWRing) & 1) ^ 1);        // released by every CTA of the cluster
                            mbar_arrive_expect_tx(&S.b_full[sb], bytes);
                            if (dbg & 4) { asm volatile("mbarrier.complete_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&S.b_full[sb])), "r"(bytes) : "memory"); }
                            else if (cs == 1) bulk_load(S.ring[sb], src, bytes, &S.b_full[sb]);
                            else {
                                const uint32_t part = bytes / (uint32_t)cs;
                                bulk_load_mc(S.ring[sb] + crank * part, src + crank * part, part, &S.b_full[sb], cmask);
                            }
                            src += bytes;
                        }
                    }
                }
            }
        } else if (warp == kMmaWarp) {
            // ================= MMA issuer ============================================================
            // The WHOLE warp runs this loop with warp-uniform control flow (so descriptor arithmetic stays on the
            // uniform datapath and feeds UTCHMMA without per-MMA R2UR moves); one fixed lane issues.  Tasks and
            // slices are fully unrolled: every descriptor is a per-step base plus a compile-time offset.  (The first
            // version -- one thread, runtime slice bookkeeping -- spent ~300 cycles per 96-cycle MMA and starved
            // the tensor pipe: profiles/r1_wide_ncu_full.csv.)
            const bool leader = elect_one();
            const uint64_t d_p0 = umma_desc(smem_u32(S.p[0]), kAChunk, 128);
            constexpr uint64_t kBufStep = (uint64_t)(C::kABuf >> 4);
            const uint64_t d_x0 = umma_desc(smem_u32(S.x[0]), kAChunk, 128), d_onez = umma_desc(smem_u32(S.onez), kAChunk, 128);
            const uint64_t d_ring0 = umma_desc(smem_u32(S.ring[0]), kN * 16, 128);
            const uint64_t d_score = umma_desc(smem_u32(S.bscore), 256, 128);
            constexpr uint64_t kSl16 = (uint64_t)((2 * kAChunk) >> 4);      // A descriptor step per K16 slice
            bool ring_ready = false;                               // "b_full of ring stage gi has completed its phase"
            for (int t = 0; t <= T; ++t) {                         // t == T: flush round (scores of the last step)
                const int n = n0 + t;
                const int ia = n % 3, ib = (n + 1) % 3, ic = (n + 2) % 3;         // h0_{n-1} | h0_n | h1_{n-1};  h1_n -> ia
                const uint64_t d_ia = d_p0 + kBufStep * ia, d_ib = d_p0 + kBufStep * ib, d_ic = d_p0 + kBufStep * ic;
                if (t == T) {
                    const int dbuf = tg & 1;
                    mbar_wait(&S.d_empty[dbuf], ((tg >> 1) & 1) ^ 1);
#pragma unroll
                    for (int j = 0; j < NCH; ++j) mbar_wait(&S.a_ready[1][j], (n - 1) & 1);      // h1_{T-1}
                    tc_fence_after();
                    if (leader) {
#pragma unroll
                        for (int s = 0; s < C::kScoreSlices; ++s)
                            umma_bf16_i(tmem + dbuf * kWD + kN, s == 0 ? d_onez : d_ic + kSl16 * (s - 1), d_score + 32 * s, kIdesc16,
                                        s == 0 ? 0u : 1u);
                        umma_commit(&S.d_full[dbuf]);
                    }
                    ++tg;
                    break;
                }
                {
                    const int sx = n % kWXStages, ux = n / kWXStages;
                    mbar_wait(&S.x_full[sx], ux & 1);
                }
                const uint64_t d_xs = d_x0 + kSl16 * (n % kWXStages);
#pragma unroll
                for (int task = 0; task < kTasks; ++task, ++tg) {
                    constexpr int kL0 = C::kSl0, kL1 = C::kSl1;
                    const bool l1 = task >= NCH;                   // compile-time after unrolling
                    const bool first_l1 = task == NCH;
                    const int nsl = l1 ? kL1 : kL0;
                    const int dbuf = tg & 1;
                    mbar_wait(&S.d_empty[dbuf], ((tg >> 1) & 1) ^ 1);              // epilogue of task tg-2 has drained it
                    tc_fence_after();
                    const uint32_t tmem_d = tmem + dbuf * kWD;
#pragma unroll
                    for (int s = 0; s < kL1; s += kWSps) {
                        if (s >= nsl) break;
                        const int sb = gi % kWRing;
                        // the status of this stage was probed one group ago (try_wait latency hidden behind the MMA issue)
                        if (!ring_ready) mbar_wait(&S.b_full[sb], (gi / kWRing) & 1);
                        ring_ready = mbar_try_wait(&S.b_full[(gi + 1) % kWRing], ((gi + 1) / kWRing) & 1);
                        const uint64_t d_b = d_ring0 + (uint64_t)(sb * (kWStage >> 4));
#pragma unroll
                        for (int h = 0; h < kWSps; ++h) {
                            const int ss = s + h;
                            if (ss >= nsl) break;
                            uint64_t da;
                            if (!l1) da = ss == 0 ? d_xs : d_ia + kSl16 * (ss - 1);
                            else if (ss == 0) da = d_onez;
                            else if (ss <= C::kHS) {
                                if (first_l1 && (ss - 1) % 3 == 0 && t > 0) {               // first use of an h1_{n-1} chunk
                                    mbar_wait(&S.a_ready[1][(ss - 1) / 3], (n - 1) & 1);
                                    tc_fence_after();
                                }
                                da = d_ic + kSl16 * (ss - 1);
                            } else {
                                if (first_l1 && (ss - 1 - C::kHS) % 3 == 0) {               // first use of an h0_n chunk
                                    mbar_wait(&S.a_ready[0][(ss - 1 - C::kHS) / 3], n & 1);
                                    tc_fence_after();
                                }
                                da = d_ib + kSl16 * (ss - 1 - C::kHS);
                            }
                            if (leader && !(dbg & 2)) {
                                umma_bf16(tmem_d, da, d_b + (uint64_t)(h * (kWSlice >> 4)), ss == 0 ? 0u : 1u);
                                if (first_l1 && ss <= C::kHS)                               // score of step n-1 (same A operand)
                                    umma_bf16_i(tmem_d + kN, da, d_score + 32 * ss, kIdesc16, ss == 0 ? 0u : 1u);
                            }
                        }
                        if (leader) {
                            if (cs == 1) umma_commit(&S.b_empty[sb]);
                            else umma_commit_mc(&S.b_empty[sb], cmask);
                        }
                        ++gi;
                    }
                    if (leader) {
                        umma_commit(&S.d_full[dbuf]);
                        if (task == NCH - 1) umma_commit(&S.x_empty[n % kWXStages]);        // last reader of x_t
                    }
                }
            }
            __syncwarp();
        } else {
            // ================= epilogue warps: (lane quarter q, 16-unit group g) of every task ===============
            const int q = warp & 3, g = warp >> 2;
            const int row = q * 32 + lane;
            const uint32_t lane_base = (uint32_t)(q * 32) << 16;
            const bool idle = q >= nq;
            float* st_c0 = state + (int64_t)blockIdx.x * 3 * C::kStateFloats;
            float* st_c1 = st_c0 + C::kStateFloats;
            float* st_z = st_c1 + C::kStateFloats;
            // float4 index of (chunk j, this warp's group, slot s, this row)
            auto sidx = [&](int j, int s) { return (((j * 3 + g) * 4 + s) * kRows + row); };
            float mx = -INFINITY, l = 0.f;
            float scl = 1.f, e = 0.f;                              // pooling factors of the step being pooled
            for (int t = 0; t <= T; ++t) {
                const int n = n0 + t;
                const int ia = n % 3, ib = (n + 1) % 3, ic = (n + 2) % 3;
                const bool flush = (t == T);
#pragma unroll
                for (int task = 0; task < kTasks; ++task) {
                    if (flush && task != 0) break;
                    const int layer = flush ? 1 : (task >= NCH ? 1 : 0);
                    const int j = flush ? 0 : (task % NCH);
                    const int dbuf = tg & 1;
                    const uint32_t tmem_d = tmem + dbuf * kWD;
                    if (idle) {                                    // keep the barrier protocol only
                        mbar_wait(&S.d_full[dbuf], (tg >> 1) & 1);
                        mbar_arrive(&S.d_empty[dbuf]);
                        if (!flush) mbar_arrive(&S.a_ready[layer][j]);
                        ++tg;
                        continue;
                    }
                    // ---- prefetch this task's state (L2) before waiting for the accumulator ----------------
                    float4 cs[4], zs[4];
                    const float4* pc = reinterpret_cast<const float4*>(layer ? st_c1 : st_c0);
                    const float4* pz = reinterpret_cast<const float4*>(st_z);
                    if (!flush) {
#pragma unroll
                        for (int s = 0; s < 4; ++s) cs[s] = (t == 0 || (dbg & 8)) ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldcg(pc + sidx(j, s));
                    }
                    if (layer == 1 && !flush) {
#pragma unroll
                        for (int s = 0; s < 4; ++s) zs[s] = (t <= 1 || (dbg & 8)) ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldcg(pz + sidx(j, s));
                    }
                    mbar_wait(&S.d_full[dbuf], (tg >> 1) & 1);
                    tc_fence_after();
                    if (layer == 1 && j == 0) {                    // score of step t-1 -> pooling factors
                        uint32_t sc2[2];
                        w_tmem_ld2(tmem_d + lane_base + kN, sc2);
                        if (t >= 1) {
                            const float score = __uint_as_float(sc2[0]) + __uint_as_float(sc2[1]);
                            const float mnew = fmaxf(mx, score);
                            scl = __expf(mx - mnew);
                            e = __expf(score - mnew);
                            l = fmaf(l, scl, e);
                            mx = mnew;
                            if constexpr (kEx)      // the score columns hold w_a / 2 . H1 + b_a = w_a . h1 + b_a
                                if (g == 0 && scores_tm && b0 + row < B) scores_tm[(int64_t)(t - 1) * B + b0 + row] = score;
                        }
                    }
                    if (flush) {
                        // last pooling update for every chunk, straight to the head scratch (global z)
                        tc_fence_before();
                        mbar_arrive(&S.d_empty[dbuf]);
                        for (int jj = 0; jj < NCH; ++jj) {
                            const unsigned char* hsrc = S.p[ic] + (jj * 6 + 2 * g) * kAChunk + row * 16;
#pragma unroll
                            for (int pr = 0; pr < 2; ++pr) {
                                const uint4 hv = ld_shared_v4(hsrc + pr * kAChunk);
                                float4 z0 = T == 1 ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldcg(pz + sidx(jj, 2 * pr));
                                float4 z1 = T == 1 ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldcg(pz + sidx(jj, 2 * pr + 1));
                                z0.x = fmaf(e, val_lo(hv.x), z0.x * scl); z0.y = fmaf(e, val_hi(hv.x), z0.y * scl);
                                z0.z = fmaf(e, val_lo(hv.y), z0.z * scl); z0.w = fmaf(e, val_hi(hv.y), z0.w * scl);
                                z1.x = fmaf(e, val_lo(hv.z), z1.x * scl); z1.y = fmaf(e, val_hi(hv.z), z1.y * scl);
                                z1.z = fmaf(e, val_lo(hv.w), z1.z * scl); z1.w = fmaf(e, val_hi(hv.w), z1.w * scl);
                                __stcg(reinterpret_cast<float4*>(st_z) + sidx(jj, 2 * pr), z0);
                                __stcg(reinterpret_cast<float4*>(st_z) + sidx(jj, 2 * pr + 1), z1);
                            }
                        }
                        ++tg;
                        continue;
                    }
                    if (layer == 1 && t >= 1) {                    // pooling of step t-1 for this chunk: z = z*scl + e*H1_{t-1}
                        const unsigned char* hsrc = S.p[ic] + (j * 6 + 2 * g) * kAChunk + row * 16;
#pragma unroll
                        for (int pr = 0; pr < 2; ++pr) {
                            const uint4 hv = ld_shared_v4(hsrc + pr * kAChunk);
                            float4& z0 = zs[2 * pr];
                            float4& z1 = zs[2 * pr + 1];
                            z0.x = fmaf(e, val_lo(hv.x), z0.x * scl); z0.y = fmaf(e, val_hi(hv.x), z0.y * scl);
                            z0.z = fmaf(e, val_lo(hv.y), z0.z * scl); z0.w = fmaf(e, val_hi(hv.y), z0.w * scl);
                            z1.x = fmaf(e, val_lo(hv.z), z1.x * scl); z1.y = fmaf(e, val_hi(hv.z), z1.y * scl);
                            z1.z = fmaf(e, val_lo(hv.w), z1.z * scl); z1.w = fmaf(e, val_hi(hv.w), z1.w * scl);
                        }
#pragma unroll
                        for (int s = 0; s < 4; ++s) if (!(dbg & 8)) __stcg(reinterpret_cast<float4*>(st_z) + sidx(j, s), zs[s]);
                    }
                    // ---- gates -> cell update -> H chunk into the A buffer (layer 0: h0_n -> ib, layer 1: h1_n -> ia)
                    unsigned char* dst = S.p[layer ? ia : ib] + (j * 6 + 2 * g) * kAChunk + row * 16;
#pragma unroll
                    for (int pr = 0; pr < 2; ++pr) {
                        uint32_t v[32], hb[4];
                        tmem_ld32(tmem_d + lane_base + (4 * g + 2 * pr) * 16, v);
                        if (dbg & 1) { hb[0] = v[0]; hb[1] = v[5]; hb[2] = v[17]; hb[3] = v[30]; }
                        else {
                        w_cell_granule(v, &cs[2 * pr].x, hb);
                        w_cell_granule(v + 16, &cs[2 * pr + 1].x, hb + 2);
                        }
                        st_shared_v4(dst + pr * kAChunk, hb[0], hb[1], hb[2], hb[3]);
                    }
                    tc_fence_before();
                    fence_proxy_async_smem();
                    mbar_arrive(&S.a_ready[layer][j]);
                    mbar_arrive(&S.d_empty[dbuf]);
                    float4* pcw = reinterpret_cast<float4*>(layer ? st_c1 : st_c0);
#pragma unroll
                    for (int s = 0; s < 4; ++s) if (!(dbg & 8)) __stcg(pcw + sidx(j, s), cs[s]);
                    ++tg;
                }
            }
            // ---- head: LN -> fc0 -> RReLU(eval) -> fc3 -> softmax, one thread per window -----------------------
            // (every MMA of the tile has completed: the flush accumulator was seen; the A buffers are free)
            named_bar_sync(1, 384);                                // all final z stores of the CTA are visible
            if (g == 0 && !idle) {
                float* zf = reinterpret_cast<float*>(S.p[0]) + row * (H + 1);     // 128 x (H+1) floats <= 3 A buffers
                const float inv_l = 0.5f / l;                      // z accumulated H = 2h
                const float4* pz = reinterpret_cast<const float4*>(st_z);
                float mean = 0.f;
                for (int gr = 0; gr < H / 4; ++gr) {               // granule gr = chunk*12 + group*4 + slot
                    const int jj = gr / 12, gg = (gr % 12) / 4, s = gr % 4;
                    const float4 zv = __ldcg(pz + (((jj * 3 + gg) * 4 + s) * kRows + row));
                    const float a0 = zv.x * inv_l, a1 = zv.y * inv_l, a2 = zv.z * inv_l, a3 = zv.w * inv_l;
                    zf[gr * 4] = a0; zf[gr * 4 + 1] = a1; zf[gr * 4 + 2] = a2; zf[gr * 4 + 3] = a3;
                    mean += (a0 + a1) + (a2 + a3);
                }
                mean *= (1.0f / H);
                if constexpr (kEx)
                    if (pooled && b0 + row < B) for (int k = 0; k < H; ++k) pooled[(b0 + row) * H + k] = zf[k];
                float var = 0.f;
                for (int k = 0; k < H; ++k) { const float d = zf[k] - mean; var = fmaf(d, d, var); }
                const float rstd = rsqrtf(var * (1.0f / H) + kLnEps);
                for (int k = 0; k < H; ++k) zf[k] = fmaf((zf[k] - mean) * rstd, S.lnw[k], S.lnb[k]);
                if constexpr (kEx)
                    if (embedding && b0 + row < B) for (int k = 0; k < H; ++k) embedding[(b0 + row) * H + k] = zf[k];
                float lg[NA_MAX_CLASSES];
#pragma unroll
                for (int k = 0; k < NA_MAX_CLASSES; ++k) lg[k] = (k < NC) ? S.b3[k] : -INFINITY;
                for (int o = 0; o < kWFc; ++o) {
                    float a = S.b0[o];
                    const float* wrow = fc0_w + o * H;
                    for (int k = 0; k < H; ++k) a = fmaf(__ldg(wrow + k), zf[k], a);
                    a = a >= 0.f ? a : a * kRReluEvalSlope;
#pragma unroll
                    for (int k = 0; k < NA_MAX_CLASSES; ++k)
                        if (k < NC) lg[k] = fmaf(S.w3[k * kWFc + o], a, lg[k]);
                }
                const int64_t b = b0 + row;
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
        // MMA / TMA roles advance their task counter past the rounds the epilogue counted
        __syncthreads();       // tile done
    }

    tc_fence_before();
    __syncthreads();
    if (cs > 1) cluster_sync_all();                 // no peer multicasts into / arrives on this CTA's smem after it exits
    if (warp == kTmaWarp) {
        tc_fence_after();
        tmem_free_all(tmem);
    }
}

int g_wide_dbg = 0;
void set_wide_dbg(int v) { g_wide_dbg = v; }
// Measured (B200, H = 192): multicast halves the L2 reads but not the time -- the stream is bound by the ring round trip
// (TMA latency + tcgen05.commit -> mbarrier), not by L2 bandwidth -- so the default stays 1.
int g_wide_cluster = 1;      // na_set_tuning("tc_wide_cluster", 1 | 2 | 4)
void set_wide_cluster(int v) { g_wide_cluster = (v == 1 || v == 2 || v == 4) ? v : 1; }

template <int NCH, bool kEx>
static int launch_wide(const void* x, const void* packed, const float* ln_w, const float* ln_b, const float* fc0_w,
                       const float* fc0_b, const float* fc3_w, const float* fc3_b, float* state, float* logits, float* probs,
                       int T, int64_t B, int64_t Bp, int NC, int sms, cudaStream_t stream, float* scores_tm, float* pooled,
                       float* embedding) {
    const size_t smem = sizeof(WideSmem<NCH>) + 1024;
    cudaError_t e = cudaFuncSetAttribute(decoder_infer_wide_kernel<NCH, kEx>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "na_decoder_infer_wide_bf16: shared memory opt-in failed (%s)", cudaGetErrorString(e));
    const int nquarters = (int)((B + 31) / 32);
    const int ntiles = (nquarters + 3) / 4;
    int cs = g_wide_cluster;
    if (ntiles < 2) cs = 1;
    int grid = ntiles < sms ? ntiles : sms;
    grid = (grid + cs - 1) / cs * cs;                          // whole clusters; surplus CTAs run idle rounds
    if (grid > sms) grid = sms / cs * cs;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kWThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, decoder_infer_wide_kernel<NCH, kEx>, reinterpret_cast<const __nv_bfloat16*>(x),
                           reinterpret_cast<const unsigned char*>(packed), ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, state, logits, probs,
                           T, B, Bp, NC, nquarters, cs, g_wide_dbg, scores_tm, pooled, embedding);
    if (e != cudaSuccess) return fail((int)e, "na_decoder_infer_wide_bf16: launch failed (%s)", cudaGetErrorString(e));
    count_launch();
    return check_launch("na_decoder_infer_wide_bf16");
}

static int wide_sms() {
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

#define NA_WIDE_DISPATCH(H, EXPR)                                                            \
    switch (H) {                                                                             \
        case 96: { constexpr int NCH = 2; EXPR; } break;                                     \
        case 144: { constexpr int NCH = 3; EXPR; } break;                                    \
        case 192: { constexpr int NCH = 4; EXPR; } break;                                    \
        default: break;                                                                      \
    }

extern "C" int64_t na_decoder_wide_packed_bytes(int64_t H) {
    int64_t r = -1;
    NA_WIDE_DISPATCH(H, r = na::tc::WideCfg<NCH>::kPackedBytes);
    return r;
}

extern "C" int64_t na_decoder_wide_state_bytes(int64_t H) {
    int64_t r = -1;
    NA_WIDE_DISPATCH(H, r = (int64_t)na::tc::wide_sms() * 3 * na::tc::WideCfg<NCH>::kStateFloats * 4);
    return r;
}

extern "C" int na_decoder_pack_wide_bf16(const float* w_ih0, const float* w_hh0, const float* b_ih0, const float* b_hh0,
                                         const float* w_ih1, const float* w_hh1, const float* b_ih1, const float* b_hh1,
                                         const float* attn_w, const float* attn_b, void* packed, int64_t H,
                                         na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(H == 96 || H == 144 || H == 192, NA_EUNSUPPORTED, "na_decoder_pack_wide_bf16: hidden_size=%lld (96, 144, 192)", (long long)H);
    NA_REQUIRE_PTR(w_ih0); NA_REQUIRE_PTR(w_hh0); NA_REQUIRE_PTR(b_ih0); NA_REQUIRE_PTR(b_hh0);
    NA_REQUIRE_PTR(w_ih1); NA_REQUIRE_PTR(w_hh1); NA_REQUIRE_PTR(b_ih1); NA_REQUIRE_PTR(b_hh1);
    NA_REQUIRE_PTR(attn_w); NA_REQUIRE(attn_b != nullptr, NA_EINVAL, "na_decoder_pack_wide_bf16: null attn_b");
    NA_REQUIRE_PTR(packed);
    NA_WIDE_DISPATCH(H, (tc::pack_wide_kernel<NCH><<<256, 256, 0, as_stream(stream)>>>(
                            w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1, attn_w, attn_b, reinterpret_cast<uint16_t*>(packed))));
    count_launch();
    return check_launch("na_decoder_pack_wide_bf16");
}

extern "C" int na_decoder_infer_wide_bf16_ex(const void* x_bf16_tmp, const void* packed, const float* ln_w, const float* ln_b,
                                             const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                                             void* state, float* logits, float* probs, float* scores_tm, float* pooled,
                                             float* embedding, int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC,
                                             na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(H == 96 || H == 144 || H == 192, NA_EUNSUPPORTED, "na_decoder_infer_wide_bf16: hidden_size=%lld (96, 144, 192)", (long long)H);
    NA_REQUIRE(T >= 1 && T < (1 << 20) && B >= 1 && Bp >= B && Bp % tc::kRows == 0, NA_EINVAL,
               "na_decoder_infer_wide_bf16: bad shape T=%lld B=%lld Bp=%lld (Bp must be a multiple of %d)", (long long)T,
               (long long)B, (long long)Bp, tc::kRows);
    NA_REQUIRE(NC >= 1 && NC <= NA_MAX_CLASSES, NA_EUNSUPPORTED, "na_decoder_infer_wide_bf16: num_classes=%lld", (long long)NC);
    NA_REQUIRE_PTR(x_bf16_tmp); NA_REQUIRE_PTR(packed); NA_REQUIRE_PTR(state); NA_REQUIRE_PTR(logits);
    NA_OPTIONAL_PTR(probs);
    NA_OPTIONAL_PTR(scores_tm); NA_OPTIONAL_PTR(pooled); NA_OPTIONAL_PTR(embedding);
    NA_REQUIRE(ln_w && ln_b && fc0_w && fc0_b && fc3_w && fc3_b, NA_EINVAL, "na_decoder_infer_wide_bf16: null parameter pointer");
    int rc = NA_EUNSUPPORTED;
    if (!(scores_tm || pooled || embedding)) {
        NA_WIDE_DISPATCH(H, (rc = tc::launch_wide<NCH, false>(x_bf16_tmp, packed, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b,
                                                              reinterpret_cast<float*>(state), logits, probs, (int)T, B, Bp, (int)NC,
                                                              tc::wide_sms(), as_stream(stream), nullptr, nullptr, nullptr)));
    } else {
        NA_WIDE_DISPATCH(H, (rc = tc::launch_wide<NCH, true>(x_bf16_tmp, packed, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b,
                                                             reinterpret_cast<float*>(state), logits, probs, (int)T, B, Bp, (int)NC,
                                                             tc::wide_sms(), as_stream(stream), scores_tm, pooled, embedding)));
    }
    return rc;
}

extern "C" int na_decoder_infer_wide_bf16(const void* x_bf16_tmp, const void* packed, const float* ln_w, const float* ln_b,
                                          const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                                          void* state, float* logits, float* probs, int64_t T, int64_t B, int64_t Bp,
                                          int64_t H, int64_t NC, na_stream_t stream) {
    return na_decoder_infer_wide_bf16_ex(x_bf16_tmp, packed, ln_w, ln_b, fc0_w, fc0_b, fc3_w, fc3_b, state, logits, probs,
                                         nullptr, nullptr, nullptr, T, B, Bp, H, NC, stream);
}
