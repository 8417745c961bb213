// C-ABI plumbing: version, thread-local error string, launch counter, K5 trial mean, and the
// dispatch of na_lstm_layer_{fwd,bwd}_f32 between the specialised and the generic tier.
#include "na_common.cuh"
#include <string.h>

namespace na {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

char* err_buf() { return g_err; }

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
static int g_train_max_ctas = 0;
int train_grid_cap(int grid) { return (g_train_max_ctas > 0 && g_train_max_ctas < grid) ? g_train_max_ctas : grid; }

int check_launch(const char* what) {
    const cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) return NA_OK;
    snprintf(g_err, sizeof(g_err), "%s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
    return (int)e;
}

int lstm_layer_fwd_generic(const float* in, const float* wt, const float* bias, float* hout, float* cout,
                           float* gates, const float* drop_mask, float drop_scale, float* hout_drop,
                           int64_t T, int64_t Bp, int64_t K, int64_t H, const float* h_init, const float* c_init,
                           cudaStream_t st);
int lstm_layer_bwd_generic(const float* dh_out, const float* gates, const float* cstate, const float* w_ih,
                           const float* w_hh, float* dgates, float* din, const float* in_drop_mask,
                           float drop_scale, int64_t T, int64_t Bp, int64_t K, int64_t H, const float* c_init,
                           const float* dh_last, const float* dc_last, float* dh_init, float* dc_init, cudaStream_t st);

bool lstm_h48_supported(int64_t K, int64_t H, bool save_c, bool save_g);
int lstm_layer_fwd_h48(const float* in, const float* wt, const float* bias, float* hout, float* cout,
                       float* gates, int64_t T, int64_t Bp, int64_t K, cudaStream_t st);
void set_h48_groups(int ng);
int mask_scale(const float* h, const float* mask, float scale, float* out, int64_t n, cudaStream_t st);

void set_iir_occ3(int v);
namespace tc { void set_infer_tanh_fma(int v); void set_x3_rcp_fma(int v); void set_infer_hs(int hs); void set_infer_rep(int v); void set_wide_cluster(int v); void set_wide_dbg(int v); void set_train_fwd_v2(int v); }
static int g_lstm_tier = 0;   // 0 = auto (specialised when available), 1 = generic only

// K5.  fp32 zeros, += in trial order, one IEEE division: bit-identical to tester.py:54,89,97.
__global__ void trial_mean_kernel(const float* __restrict__ in, float* __restrict__ out, int R, int64_t N) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    float acc = 0.f;
    for (int r = 0; r < R; ++r) acc = __fadd_rn(acc, in[(int64_t)r * N + i]);
    out[i] = __fdiv_rn(acc, (float)R);
}

}  // namespace na

extern "C" int na_version(void) { return NA_VERSION; }
extern "C" const char* na_last_error(void) { return na::err_buf(); }
extern "C" int64_t na_launch_count(void) { return na::g_launches.load(std::memory_order_relaxed); }

extern "C" int na_trial_mean_f32(const float* in, float* out, int64_t R, int64_t N, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(R >= 1 && R <= (1 << 24) && N >= 0, NA_EINVAL, "na_trial_mean_f32: bad shape R=%lld N=%lld",
               (long long)R, (long long)N);
    if (N == 0) return NA_OK;
    NA_REQUIRE_PTR(in);
    NA_REQUIRE_PTR(out);
    trial_mean_kernel<<<(unsigned)((N + 255) / 256), 256, 0, as_stream(stream)>>>(in, out, (int)R, N);
    count_launch();
    return check_launch("na_trial_mean_f32");
}

static int check_lstm_shape(const char* fn, int64_t T, int64_t Bp, int64_t K, int64_t H) {
    using namespace na;
    NA_REQUIRE(T >= 1 && Bp >= NA_BATCH_ALIGN && Bp % NA_BATCH_ALIGN == 0, NA_EINVAL,
               "%s: bad shape T=%lld Bp=%lld (Bp must be a positive multiple of %d)", fn, (long long)T,
               (long long)Bp, NA_BATCH_ALIGN);
    NA_REQUIRE(K >= 1 && H >= 1 && H <= 1024 && K <= 4096, NA_EUNSUPPORTED, "%s: unsupported K=%lld H=%lld", fn,
               (long long)K, (long long)H);
    NA_REQUIRE(T <= INT32_MAX && T * Bp * 4 * H < ((int64_t)1 << 40), NA_EUNSUPPORTED, "%s: problem too large", fn);
    return NA_OK;
}

extern "C" int na_lstm_layer_fwd_f32_hx(const float* in, const float* wt, const float* bias, float* hout,
                                        float* cout, float* gates, const float* drop_mask, float drop_scale,
                                        float* hout_drop, int64_t T, int64_t Bp, int64_t K, int64_t H,
                                        const float* h_init, const float* c_init, na_stream_t stream) {
    using namespace na;
    if (int rc = check_lstm_shape("na_lstm_layer_fwd_f32", T, Bp, K, H)) return rc;
    NA_REQUIRE_PTR(in); NA_REQUIRE_PTR(wt); NA_REQUIRE_PTR(bias); NA_REQUIRE_PTR(hout);
    NA_OPTIONAL_PTR(cout); NA_OPTIONAL_PTR(gates); NA_OPTIONAL_PTR(drop_mask); NA_OPTIONAL_PTR(hout_drop);
    NA_OPTIONAL_PTR(h_init); NA_OPTIONAL_PTR(c_init);
    NA_REQUIRE((drop_mask == nullptr) == (hout_drop == nullptr), NA_EINVAL,
               "na_lstm_layer_fwd_f32: drop_mask and hout_drop must be given together");
    NA_REQUIRE((h_init == nullptr) == (c_init == nullptr), NA_EINVAL,
               "na_lstm_layer_fwd_f32_hx: h_init and c_init must be given together");
    if (g_lstm_tier == 0 && h_init == nullptr && lstm_h48_supported(K, H, cout != nullptr, gates != nullptr)) {
        if (int rc = lstm_layer_fwd_h48(in, wt, bias, hout, cout, gates, T, Bp, K, as_stream(stream))) return rc;
        if (drop_mask) return mask_scale(hout, drop_mask, drop_scale, hout_drop, T * Bp * H, as_stream(stream));
        return NA_OK;
    }
    return lstm_layer_fwd_generic(in, wt, bias, hout, cout, gates, drop_mask, drop_scale, hout_drop, T, Bp, K, H,
                                  h_init, c_init, as_stream(stream));
}

extern "C" int na_lstm_layer_fwd_f32(const float* in, const float* wt, const float* bias, float* hout,
                                     float* cout, float* gates, const float* drop_mask, float drop_scale,
                                     float* hout_drop, int64_t T, int64_t Bp, int64_t K, int64_t H,
                                     na_stream_t stream) {
    return na_lstm_layer_fwd_f32_hx(in, wt, bias, hout, cout, gates, drop_mask, drop_scale, hout_drop, T, Bp, K, H,
                                    nullptr, nullptr, stream);
}

extern "C" int na_set_tuning(const char* key, int64_t value) {
    using namespace na;
    NA_REQUIRE(key != nullptr, NA_EINVAL, "na_set_tuning: null key");
    if (!strcmp(key, "lstm_tier")) { g_lstm_tier = (int)value; return NA_OK; }
    if (!strcmp(key, "h48_groups")) { set_h48_groups((int)value); return NA_OK; }
    if (!strcmp(key, "tc_infer_hs")) { tc::set_infer_hs((int)value); return NA_OK; }
    if (!strcmp(key, "tc_infer_rep")) { tc::set_infer_rep((int)value); return NA_OK; }
    if (!strcmp(key, "tc_train_fwd_v2")) { tc::set_train_fwd_v2((int)value); return NA_OK; }
    if (!strcmp(key, "tc_wide_dbg")) { tc::set_wide_dbg((int)value); return NA_OK; }
    if (!strcmp(key, "tc_infer_tanh_fma")) { tc::set_infer_tanh_fma((int)value); return NA_OK; }
    if (!strcmp(key, "x3_rcp_fma")) { tc::set_x3_rcp_fma((int)value); return NA_OK; }
    if (!strcmp(key, "iir_occ3")) { set_iir_occ3((int)value); return NA_OK; }
    if (!strcmp(key, "train_max_ctas")) { g_train_max_ctas = (int)value; return NA_OK; }
    if (!strcmp(key, "tc_wide_cluster")) { tc::set_wide_cluster((int)value); return NA_OK; }
    return fail(NA_EINVAL, "na_set_tuning: unknown key '%s'", key);
}

namespace na {
// FFMA issue-rate probe: 16 independent fp32 FMA chains per thread.  Used by bench.py to MEASURE
// the CUDA-core fp32 peak that bounds the exact-fp32 recurrence (there is no such number in
// MEASURED_PEAKS.json).  2 * 16 * iters flops per thread.
__global__ void __launch_bounds__(256) ffma_probe_kernel(float* out, int iters, float a, float b) {
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = (float)(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = fmaf(v[i], a, b);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += v[i];
    if (s == 12345.678f) out[0] = s;   // never true; keeps the chains alive
}
}  // namespace na

extern "C" int na_ffma_probe(float* out, int64_t blocks, int64_t iters, na_stream_t stream) {
    using namespace na;
    NA_REQUIRE(blocks >= 1 && iters >= 1 && iters <= (1 << 30), NA_EINVAL, "na_ffma_probe: bad arguments");
    NA_REQUIRE_PTR(out);
    ffma_probe_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(out, (int)iters, 0.999f, 0.001f);
    count_launch();
    return check_launch("na_ffma_probe");
}

extern "C" int na_lstm_layer_bwd_f32_hx(const float* dh_out, const float* gates, const float* cstate,
                                        const float* w_ih, const float* w_hh, float* dgates, float* din,
                                        const float* in_drop_mask, float drop_scale, int64_t T, int64_t Bp,
                                        int64_t K, int64_t H, const float* c_init, const float* dh_last,
                                        const float* dc_last, float* dh_init, float* dc_init, na_stream_t stream) {
    using namespace na;
    if (int rc = check_lstm_shape("na_lstm_layer_bwd_f32", T, Bp, K, H)) return rc;
    NA_REQUIRE_PTR(dh_out); NA_REQUIRE_PTR(gates); NA_REQUIRE_PTR(cstate); NA_REQUIRE_PTR(w_ih);
    NA_REQUIRE_PTR(w_hh); NA_REQUIRE_PTR(dgates);
    NA_OPTIONAL_PTR(din); NA_OPTIONAL_PTR(in_drop_mask);
    NA_OPTIONAL_PTR(c_init); NA_OPTIONAL_PTR(dh_last); NA_OPTIONAL_PTR(dc_last); NA_OPTIONAL_PTR(dh_init);
    NA_OPTIONAL_PTR(dc_init);
    return lstm_layer_bwd_generic(dh_out, gates, cstate, w_ih, w_hh, dgates, din, in_drop_mask, drop_scale, T, Bp,
                                  K, H, c_init, dh_last, dc_last, dh_init, dc_init, as_stream(stream));
}

extern "C" int na_lstm_layer_bwd_f32(const float* dh_out, const float* gates, const float* cstate,
                                     const float* w_ih, const float* w_hh, float* dgates, float* din,
                                     const float* in_drop_mask, float drop_scale, int64_t T, int64_t Bp,
                                     int64_t K, int64_t H, na_stream_t stream) {
    return na_lstm_layer_bwd_f32_hx(dh_out, gates, cstate, w_ih, w_hh, dgates, din, in_drop_mask, drop_scale, T, Bp,
                                    K, H, nullptr, nullptr, nullptr, nullptr, nullptr, stream);
}
