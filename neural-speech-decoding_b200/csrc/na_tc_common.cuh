// tcgen05 / TMEM helpers shared by the tensor-core kernels (na_decoder_tc.cu, na_train_tc.cu).
#pragma once
#include "na_common.cuh"
#include "na_sm100.cuh"
#include <cuda_fp16.h>

namespace na {
namespace tc {

constexpr int kRows = 128;                   // windows per CTA tile = UMMA M
constexpr int kH = 48;
constexpr int kN = 4 * kH;                   // 192 gate columns
constexpr int kAChunk = kRows * 16;          // bytes of one A K-chunk (8 bf16 per row)
constexpr int kBChunk = kN * 16;             // bytes of one B K-chunk (192 rows)
constexpr uint32_t kTmemCols = 512;

// ---- tcgen05 wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    // K-major, no swizzle: LBO = byte stride between the two 8-element K-chunks of one K16 step,
    // SBO = byte stride between 8-row groups.  Bits: addr>>4 [0,14), LBO>>4 [16,30),
    // SBO>>4 [32,46), version=1 [46,48), layout_type=0 [61,64).
    uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

// Advance a descriptor's start address by `bytes` (a multiple of 16; the 14-bit address field never carries
// for shared-memory offsets).  The MMA-issuing thread builds each base descriptor ONCE and steps it with
// one add per MMA: issuing 30+ MMAs per step with a full descriptor rebuild each (~16 instructions on the
// uniform datapath) was the serial bottleneck of the BPTT kernel.
__device__ __forceinline__ uint64_t desc_adv(uint64_t d, uint32_t bytes) { return d + (uint64_t)(bytes >> 4); }

// 16-bit operand formats of the tier.  VALUE operands (EEG samples, h, weights, bias) have a bounded
// range, so they are IEEE fp16: 3 more mantissa bits than bf16 at the same tensor throughput -- the
// weight rounding is a FIXED perturbation applied at every one of the 1250 dependent steps, so those
// bits matter.  GRADIENT operands (d gates) have an unbounded range and stay bf16.
constexpr uint32_t kFmtF16 = 0, kFmtBF16 = 1;
// (kind::f16 rejects mixed f16 x bf16 operands -- illegal instruction on sm_100a -- so d(gates) are
// fp16 too; the host scales the incoming gradient by a power of two so they sit in fp16's range.)
constexpr uint32_t kFmtVal = kFmtF16, kFmtGrad = kFmtF16;

// Instruction descriptor, kind::f16, 16-bit x 16-bit -> f32, M = 128.  a_mn / b_mn: operand is MN-major.
__host__ __device__ constexpr uint32_t make_idesc(int n, uint32_t a_fmt, uint32_t b_fmt, bool a_mn = false,
                                                  bool b_mn = false) {
    return (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kRows >> 4) << 24);
}
constexpr uint32_t kIdesc = make_idesc(kN, kFmtVal, kFmtVal);   // gate GEMM: N = 192, both operands K-major

__device__ __forceinline__ void umma_bf16_i(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    umma_bf16_i(tmem_d, adesc, bdesc, kIdesc, accumulate);
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// one lane of a fully converged warp (elect.sync): the compiler knows the guarded region is single-threaded
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ float tanh_apx(float v) {
    float r;
    asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float sigmoid_apx(float v) { return fmaf(0.5f, tanh_apx(0.5f * v), 0.5f); }

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
}
// value-format (fp16) pack / unpack / scalar conversion
__device__ __forceinline__ uint32_t pack_val(float lo, float hi) {
    __half2 p = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ float val_lo(uint32_t p) { return __low2float(*reinterpret_cast<__half2*>(&p)); }
__device__ __forceinline__ float val_hi(uint32_t p) { return __high2float(*reinterpret_cast<__half2*>(&p)); }
__device__ __forceinline__ uint16_t val16(float v) { return __half_as_ushort(__float2half_rn(v)); }
__device__ __forceinline__ float val16_to_float(uint16_t b) { return __half2float(__ushort_as_half(b)); }
constexpr uint32_t kValOnes2 = 0x3C003C00u;              // {1.0, 1.0} in the value format

__device__ __forceinline__ void st_shared_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(p)), "r"(a), "r"(b), "r"(c), "r"(d)
                 : "memory");
}

// One window's row of N fp32 values (N % 4 == 0) to global memory, 16 B per store (the row starts 16-byte aligned:
// the intermediates outputs of the inference kernels, [B][H] with H a multiple of 4).
template <int N>
__device__ __forceinline__ void store_row(float* dst, const float* v) {
    static_assert(N % 4 == 0, "row length");
#pragma unroll
    for (int j = 0; j < N; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
}

// One LSTM cell update for the 8 units of a block; v = [i x8 | f x8 | g x8 | o x8] pre-activations.
// Returns h packed as 4 x bf16x2.
__device__ __forceinline__ void cell_block(const uint32_t (&v)[32], float* c, uint32_t (&hp)[4]) {
    float h[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const float gi = sigmoid_apx(__uint_as_float(v[u]));
        const float gf = sigmoid_apx(__uint_as_float(v[8 + u]));
        const float gg = tanh_apx(__uint_as_float(v[16 + u]));
        const float go = sigmoid_apx(__uint_as_float(v[24 + u]));
        c[u] = fmaf(gf, c[u], gi * gg);
        h[u] = go * tanh_apx(c[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) hp[u] = pack_val(h[2 * u], h[2 * u + 1]);
}


// ---- inter-layer dropout (lstm_eeg_model.py:21) without a mask tensor ---------------------------------
// Counter-based: the keep-bits of the 8 units of block `blk` of window-row `grow` (= t*Bp + b) are a pure
// function of (seed, grow, blk), so the backward regenerates exactly the forward's mask.  16-bit
// resolution: P(keep) = thresh16 / 65536.
__device__ __forceinline__ uint32_t fmix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    return h;
}
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t seed, int64_t grow, int blk, uint32_t thresh16) {
    const uint64_t idx = (uint64_t)grow * 6u + (uint32_t)blk;
    const uint32_t base = fmix32(((uint32_t)idx ^ (uint32_t)seed) * 0x9E3779B1u + ((uint32_t)(idx >> 32) ^ (uint32_t)(seed >> 32)));
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t w = fmix32(base + (uint32_t)(i + 1) * 0x9E3779B9u);
        bits |= ((w & 0xFFFFu) < thresh16 ? 1u : 0u) << (2 * i);
        bits |= ((w >> 16) < thresh16 ? 1u : 0u) << (2 * i + 1);
    }
    return bits;
}
// keep-bits from 8 mask bytes (explicit mask tensor)
__device__ __forceinline__ uint32_t mask_keep8(uint2 mk) {
    uint32_t bits = 0;
#pragma unroll
    for (int u = 0; u < 8; ++u) bits |= ((((u < 4 ? mk.x : mk.y) >> (8 * (u & 3))) & 0xFFu) ? 1u : 0u) << u;
    return bits;
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_alloc_all(uint32_t* smem_dst) {     // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free_all(uint32_t taddr) {          // the same warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(kTmemCols) : "memory");
}

}  // namespace tc
}  // namespace na
