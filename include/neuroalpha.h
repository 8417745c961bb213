/*
 * neuroalpha.h -- C ABI of libneuroalpha_b200.so (sm_100a).
 *
 * This is the drop-in boundary for the NeuroAlpha decoder hot path
 * (aa217/Neural-Speech-Decoding).  The reference has no FFI / plugin layer: its only
 * interface for this path is the Python class `EEG_LSTM` and its callers
 *     Neuro-Alpha-App/Utilities/lstm_eeg_model.py:13-39   EEG_LSTM.__init__/forward
 *     Neuro-Alpha-App/Utilities/lstm_eeg_model.py:86-101  SimplePredictor.predict
 *     Neuro-Alpha-App/Utilities/tester.py:54,89,97        run_trials probability averaging
 *     Neuro-Alpha-App/Frontend/app.py:166-170             normalize_eeg (z-score)
 * Each entry point below names the reference lines whose arithmetic it replaces.
 * INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer on the current CUDA device, contiguous and
 *     16-byte aligned, allocated and owned by the caller.  Kernels never allocate.
 *   - Launches are asynchronous on `stream` (a cudaStream_t passed as void*); there
 *     is no hidden synchronisation and no global mutable state except a thread-local
 *     error string.
 *   - Return value: 0 = ok; >0 = cudaError_t of a failed launch; <0 = NA_E* below.
 *     No exception crosses the ABI; na_last_error() gives the message.
 *   - "time-major padded" (TMP) layout: [T][Bp][F] fp32, Bp = batch rounded up to a
 *     multiple of NA_BATCH_ALIGN; rows b >= B are padding and hold finite values.
 *   - Gate order everywhere is torch's [i, f, g, o] (lstm_eeg_model.py:16-22 -> nn.LSTM).
 */
#ifndef NEUROALPHA_H_
#define NEUROALPHA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NA_VERSION 100          /* 0.1.0 */
#define NA_BATCH_ALIGN 32       /* Bp granularity of the TMP layout */
#define NA_FC_HIDDEN 32         /* lstm_eeg_model.py:26 -- fc hidden width is fixed at 32 */
#define NA_MAX_CLASSES 16

enum {
    NA_OK = 0,
    NA_EINVAL = -1,        /* bad shape / null pointer */
    NA_EALIGN = -2,        /* pointer not 16-byte aligned */
    NA_EUNSUPPORTED = -3,  /* size outside what the kernels implement */
    NA_EDEVICE = -4        /* not an sm_100 device */
};

enum { NA_F32 = 0, NA_BF16 = 1, NA_F16 = 2 };

typedef void* na_stream_t;      /* cudaStream_t */

int na_version(void);
const char* na_last_error(void);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches). */
int64_t na_launch_count(void);

/* Tuning / test knobs (process-global, not thread-safe; set before launching work):
 *   "lstm_tier"  0 = auto (specialised H=48 kernels when the shape allows), 1 = generic tier only
 *   "h48_groups" 0 = auto, 1..4 = groups (32-window tiles) resident per CTA in the H=48 kernels
 *   "tc_infer_hs" / "tc_infer_rep" / "tc_train_fwd_v2" / "tc_wide_dbg" / "tc_wide_cluster"   A/B switches of the 16-bit tier
 *   "tc_infer_tanh_fma", "x3_rcp_fma"   MUFU -> FMA-pipe offloads (default 0: measured slower, DESIGN.md section 10b)
 *   "iir_occ3"        1 = three CTAs per SM in na_iir_chain (default 0 = two)
 *   "train_max_ctas"  test knob: caps the grid of the persistent tensor-core training kernels (0 = one CTA per SM), so that
 *                     small batches exercise the several-tiles-per-CTA paths; scratch sizes ignore it
 */
int na_set_tuning(const char* key, int64_t value);

/* Measurement aid: launches `blocks` CTAs of 256 threads, each thread running 16 independent
 * fp32 FMA chains for `iters` iterations (2*16*iters flops per thread).  bench.py times it to
 * obtain the CUDA-core fp32 peak the exact-fp32 recurrence is bounded by. */
int na_ffma_probe(float* out, int64_t blocks, int64_t iters, na_stream_t stream);

/* ---- K1: windowing + optional per-window per-channel z-score -------------------------
 * Replaces Frontend/app.py:166-170 (normalize_eeg: (x-mean)/(std+1e-6), population std,
 * over the time axis) and the "latest int(window_seconds*sr) samples" windowing of
 * Utilities/streaming_process.py:35,55.
 *   x      [n_samples, C] fp32 stream; window w covers samples [w*hop, w*hop+T)
 *          (a [B,T,C] batch is the case hop == T)
 *   y      normalize ? z-scored : copied windows, fp32 or bf16 (out_dtype), in
 *          out_tmp ? TMP layout [T][Bp][C] (rows >= B zero-filled) : [B][T][C]
 */
int na_window_zscore(const float* x, void* y, int64_t B, int64_t T, int64_t C, int64_t hop,
                     int normalize, int out_tmp, int64_t Bp, int out_dtype, na_stream_t stream);

/* ---- weight packing ---------------------------------------------------------------------
 * nn.LSTM parameters of one layer (lstm_eeg_model.py:16-22; shapes SURVEY 8a):
 *   w_ih [4H,K], w_hh [4H,H], b_ih [4H], b_hh [4H]  ->
 *   wt   [(K+H)][4H]  k-major concatenation [W_ih | W_hh]^T,   bias [4H] = b_ih + b_hh
 */
int na_pack_lstm_layer(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                       float* wt, float* bias, int64_t K, int64_t H, na_stream_t stream);

/* ---- K3: one LSTM layer, all timesteps, h0 = c0 = 0 -------------------------------------
 * Replaces `self.lstm(x)` (lstm_eeg_model.py:34), one layer per call.
 *   in    TMP [T][Bp][K]       hout TMP [T][Bp][H]
 *   cout  TMP [T][Bp][H]  or NULL   (cell state, saved for backward)
 *   gates TMP [T][Bp][4H] or NULL   (activated i,f,g,o, saved for backward)
 *   drop_mask TMP [T][Bp][H] of 0/1 + hout_drop TMP [T][Bp][H], both or neither: inter-layer
 *          dropout (lstm_eeg_model.py:21).  hout_drop = hout * mask * drop_scale
 *          (drop_scale = 1/(1-p)) is what the next layer consumes; hout stays the raw h
 *          (the recurrence and dW_hh need it).
 */
int na_lstm_layer_fwd_f32(const float* in, const float* wt, const float* bias,
                          float* hout, float* cout, float* gates,
                          const float* drop_mask, float drop_scale, float* hout_drop,
                          int64_t T, int64_t Bp, int64_t K, int64_t H, na_stream_t stream);

/* Fused BPTT of one layer.  dh_out TMP [T][Bp][H] is dLoss/d(hout).  Produces dgates TMP
 * [T][Bp][4H] (pre-activation gate gradients) and, if din != NULL, din TMP [T][Bp][K] =
 * dLoss/d(in); when in_drop_mask != NULL (the mask that produced this layer's input in the
 * forward) din is multiplied by mask*drop_scale so it is directly the lower layer's dh_out.
 * Weight gradients follow from dgates with na_lstm_layer_wgrad_f32.  w_ih [4H,K] / w_hh
 * [4H,H] are the unpacked nn.LSTM tensors.
 */
int na_lstm_layer_bwd_f32(const float* dh_out, const float* gates, const float* cstate,
                          const float* w_ih, const float* w_hh,
                          float* dgates, float* din, const float* in_drop_mask, float drop_scale,
                          int64_t T, int64_t Bp, int64_t K, int64_t H, na_stream_t stream);

/* dW_ih [4H,K] = sum_rows dgates^T in ; dW_hh [4H,H] = sum_{t>=1} dgates_t^T h_{t-1} ;
 * db [4H] = column sums (gradient of both b_ih and b_hh).  Deterministic two-stage
 * reduction; `partials` is caller scratch of na_wgrad_partial_floats(K,H) floats.
 */
int64_t na_wgrad_partial_floats(int64_t K, int64_t H);
int na_lstm_layer_wgrad_f32(const float* dgates, const float* in, const float* h,
                            float* dw_ih, float* dw_hh, float* db, float* partials,
                            int64_t T, int64_t Bp, int64_t K, int64_t H, na_stream_t stream);

/* ---- K3 with an initial state (nn.LSTM's hx) -----------------------------------------------
 * The three calls above with the layer's initial state and its gradients; every extra pointer is
 * TMP-row [Bp][H] fp32 (rows >= B zero), optional, and with all of them NULL each call is exactly
 * its sibling.
 *   fwd:   h_init / c_init = h_{-1} / c_{-1} (both or neither).  With them the generic kernel runs
 *          for every shape (the H = 48 kernels start from zeros).
 *   bwd:   c_init = c_{-1} (it enters d(forget gate) at t = 0); dh_last / dc_last = dLoss/dh_{T-1}
 *          / dLoss/dc_{T-1} from outside the sequence output (nn.LSTM's h_n / c_n), added at
 *          t = T-1; dh_init / dc_init receive dLoss/dh_{-1} / dLoss/dc_{-1}.
 *   wgrad: h_init adds the step-0 term dgates_0^T h_init to dW_hh.
 */
int na_lstm_layer_fwd_f32_hx(const float* in, const float* wt, const float* bias,
                             float* hout, float* cout, float* gates,
                             const float* drop_mask, float drop_scale, float* hout_drop,
                             int64_t T, int64_t Bp, int64_t K, int64_t H,
                             const float* h_init, const float* c_init, na_stream_t stream);
int na_lstm_layer_bwd_f32_hx(const float* dh_out, const float* gates, const float* cstate,
                             const float* w_ih, const float* w_hh,
                             float* dgates, float* din, const float* in_drop_mask, float drop_scale,
                             int64_t T, int64_t Bp, int64_t K, int64_t H,
                             const float* c_init, const float* dh_last, const float* dc_last,
                             float* dh_init, float* dc_init, na_stream_t stream);
int na_lstm_layer_wgrad_f32_hx(const float* dgates, const float* in, const float* h,
                               float* dw_ih, float* dw_hh, float* db, float* partials,
                               int64_t T, int64_t Bp, int64_t K, int64_t H,
                               const float* h_init, na_stream_t stream);

/* ---- K4: attention pool + LayerNorm + MLP head (+ softmax) -------------------------------
 * Replaces lstm_eeg_model.py:35-39 and, when probs != NULL, F.softmax at :97.
 *   h TMP [T][Bp][H];  attn_w [H], attn_b [1], ln_w [H], ln_b [H],
 *   fc0_w [32,H], fc0_b [32], fc3_w [NC,32], fc3_b [NC]
 *   rrelu_slope [B,32] or NULL (eval: (1/8+1/3)/2), drop_mask [B,32] 0/1 or NULL, drop_scale
 *   logits [B,NC]; probs [B,NC] or NULL
 *   saved (training, may be NULL): stats [B][2] = softmax-over-time (max, sum),
 *   zpool [B,H] (pre-LN pooled vector)
 */
int na_head_fwd_f32(const float* h, const float* attn_w, const float* attn_b,
                    const float* ln_w, const float* ln_b,
                    const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                    const float* rrelu_slope, const float* drop_mask, float drop_scale,
                    float* logits, float* probs, float* stats, float* zpool,
                    int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC, na_stream_t stream);

/* ---- intermediates of the eval forward (lstm_eeg_model.py:35-38: what forward hooks on attn / ln would see) -----------
 * Every *_ex entry point takes the arguments of its sibling plus three optional outputs after `probs`; each may be NULL,
 * and with all three NULL the call is exactly the sibling.  They are written by the same launch as the logits:
 *   scores_tm  [T][B] fp32, TIME-MAJOR (row t = the B windows' scores s_t = attn.weight . h_t + attn.bias of step t;
 *              the kernels hold 32 consecutive windows per warp, so each step is one contiguous run of stores)
 *   pooled     [B][H] fp32, sum_t alpha_t h_t (the attention-pooled vector before LayerNorm)
 *   embedding  [B][H] fp32, LayerNorm(pooled) (the input of fc)
 * Only rows b < B are written; 16-byte alignment as for the other outputs.
 * na_attention_softmax_f32: scores_tm [T][B] -> attn [B][T] = softmax over time per window (exp(s - max) / sum in fp32,
 * torch.softmax's formula; a NaN score gives the window a NaN row).  In the 16-bit tier (na_decoder_infer_bf16_ex and
 * _x32_ex, na_decoder_infer_wide_bf16_ex) the intermediates carry that tier's 2e-2 contract; the v1 kernel
 * (na_set_tuning("tc_infer_hs", 1 | 2)) does not write them: a non-NULL extra returns NA_EUNSUPPORTED.
 */
int na_head_fwd_f32_ex(const float* h, const float* attn_w, const float* attn_b,
                       const float* ln_w, const float* ln_b,
                       const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                       const float* rrelu_slope, const float* drop_mask, float drop_scale,
                       float* logits, float* probs, float* scores_tm, float* pooled, float* embedding,
                       float* stats, float* zpool,
                       int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC, na_stream_t stream);
int na_attention_softmax_f32(const float* scores_tm, float* attn, int64_t T, int64_t B, na_stream_t stream);

/* Backward of na_head_fwd_f32.  dlogits [B,NC] -> dh TMP [T][Bp][H] (padding rows zeroed)
 * and the 8 head parameter gradients, packed in `dparams` as
 * [attn_w H | attn_b 1 | ln_w H | ln_b H | fc0_w 32H | fc0_b 32 | fc3_w 32NC | fc3_b NC].
 * `partials` is scratch of na_head_partial_floats(B,H,NC) floats.
 */
int64_t na_head_param_floats(int64_t H, int64_t NC);
int64_t na_head_partial_floats(int64_t B, int64_t H, int64_t NC);
int na_head_bwd_f32(const float* dlogits, const float* h, const float* stats, const float* zpool,
                    const float* attn_w, const float* attn_b, const float* ln_w, const float* ln_b,
                    const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                    const float* rrelu_slope, const float* drop_mask, float drop_scale,
                    float* dh, float* dparams, float* partials,
                    int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC, na_stream_t stream);

/* ---- ingestion of the collector's CSV windows (SURVEY 8(f) rank 2) ---------------------------------
 * Replaces np.loadtxt(path, delimiter=",", dtype=np.float32) over the files np.savetxt(fmt="%.7f") wrote
 * (Neural_decoding_data_collector.py:129-139): `text` = the raw bytes of n_files files back to back (device memory),
 * offsets[n_files + 1] = their byte ranges (device int64), out = fp32 [n_files][fields_per_file] in file order
 * (row-major rows x columns of each file), status[2n] = number of fields found in file n, status[2n+1] = number of
 * fields that are not plain [sign]digits[.digits] with <= 15 significant digits (the caller must treat either
 * mismatch as an error; the kernel never approximates).  Bit-identical to numpy: decimal -> correctly rounded
 * double (one IEEE division of two exact operands) -> float32.  max_file_bytes = the longest file (<= 200 KB).
 * `text` must be 16-byte aligned and readable up to the next 16-byte boundary after its last byte.
 */
int na_csv_parse_f32(const void* text, const int64_t* offsets, float* out, int* status, int64_t n_files,
                     int64_t fields_per_file, int64_t max_file_bytes, na_stream_t stream);

/* ---- collector-side filter chain (SURVEY 8(f) rank 4) ------------------------------------------------
 * Replaces the per-channel BrainFlow calls of Neural_decoding_data_collector.py:109-127 on raw windows:
 * x fp32 [B][T][C] -> y fp32 [B][T][C]; per (b, c) series: detrend(CONSTANT) if `detrend`, then for each of the
 * nfilt filters a zero-phase application (forward DirectFormII cascade, reversal, the same cascade -- state carried
 * over if carry_state, as BrainFlow re-uses the filter object -- reversal), then np.round(., round_decimals)
 * (< 0: none) and -0 -> 0.  Arithmetic in float64.  coef = the sections of all filters back to back, 5 doubles each
 * (b0 b1 b2 a1 a2, a0 = 1); nsec[f] = sections of filter f (<= 8 filters x <= 8 sections; each section count is
 * checked by the caller; max_sections = the largest nsec[f], passed in so that no device-to-host copy is needed);
 * scratch = T * roundup(B*C, 128) doubles for T > 2560, otherwise unused and may be NULL (one warp per series, the
 * series stays in registers).  Parity unpinned: BrainFlow is not available in this image.
 */
int na_iir_chain(const float* x, float* y, double* scratch, const double* coef, const int* nsec, int64_t nfilt,
                 int64_t B, int64_t T, int64_t C, int detrend, int round_decimals, int carry_state, int64_t max_sections,
                 na_stream_t stream);

/* ---- tensor-core tier: whole decoder forward, bf16 operands / fp32 accumulate ----------------
 * One persistent warp-specialised tcgen05 / TMEM / TMA kernel: K2 (input-gate contraction,
 * fused as extra K-steps of the per-step MMA), K3 (2-layer recurrence, wavefronted), K4 (online
 * attention pool + LayerNorm + MLP head) and the class softmax.  Replaces
 * lstm_eeg_model.py:32-39 + :97 in eval mode for the flagship shape C=8, H=48, L=2.
 * Contract (north_star): logits within 2e-2 (relative to max|logit|) of the fp32 reference,
 * argmax identical on the repo's windows.
 *   na_decoder_pack_bf16: the 8 nn.LSTM tensors of both layers -> `packed`
 *       (na_decoder_packed_bf16_bytes() bytes): B operands [W_ih | bias hi,lo | W_hh] in the UMMA
 *       K-major core-matrix layout, two sections: gate columns permuted to (unit/8, gate, unit%8) for the
 *       training kernels, and to (unit/4, gate, unit%4) with the sigmoid / H = 2h scalings folded in for
 *       the inference kernel (na_decoder_tc2.cu).
 *   na_decoder_infer_bf16: x TMP bf16 [T][Bp][8] (na_window_zscore with out_dtype = NA_BF16,
 *       Bp a multiple of 128) -> logits [B,NC] fp32 (+ probs [B,NC] if not NULL).
 */
int64_t na_decoder_packed_bf16_bytes(void);
int na_decoder_pack_bf16(const float* w_ih0, const float* w_hh0, const float* b_ih0, const float* b_hh0,
                         const float* w_ih1, const float* w_hh1, const float* b_ih1, const float* b_hh1,
                         void* packed, na_stream_t stream);
int na_decoder_infer_bf16(const void* x_bf16_tmp, const void* packed,
                          const float* attn_w, const float* attn_b, const float* ln_w, const float* ln_b,
                          const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                          float* logits, float* probs,
                          int64_t T, int64_t B, int64_t Bp, int64_t NC, na_stream_t stream);

/* The same forward straight from the caller's batch-first fp32 windows x [B][T][8] (`forward(x)`): the
 * fp32 -> fp16 time-major pack is fused into the kernel (no intermediate copy of the input). */
int na_decoder_infer_bf16_x32(const float* x, const void* packed,
                              const float* attn_w, const float* attn_b, const float* ln_w, const float* ln_b,
                              const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                              float* logits, float* probs, int64_t T, int64_t B, int64_t NC, na_stream_t stream);
/* The same two with the intermediates outputs (see na_head_fwd_f32_ex). */
int na_decoder_infer_bf16_ex(const void* x_bf16_tmp, const void* packed,
                             const float* attn_w, const float* attn_b, const float* ln_w, const float* ln_b,
                             const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                             float* logits, float* probs, float* scores_tm, float* pooled, float* embedding,
                             int64_t T, int64_t B, int64_t Bp, int64_t NC, na_stream_t stream);
int na_decoder_infer_bf16_x32_ex(const float* x, const void* packed,
                                 const float* attn_w, const float* attn_b, const float* ln_w, const float* ln_b,
                                 const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                                 float* logits, float* probs, float* scores_tm, float* pooled, float* embedding,
                                 int64_t T, int64_t B, int64_t NC, na_stream_t stream);

/* ---- exact tier on the tensor cores (fp32 accuracy, 1e-5 contract) ------------------------------------
 * The same forward as na_decoder_infer_bf16_x32 at fp32 accuracy: every operand is split into fp16 hi + lo halves and
 * each product is three tcgen05 MMAs (hi.hi + hi.lo + lo.hi, fp32 accumulation); activations by ex2.approx + rcp.approx
 * (~2e-7), cell state / pooling / head in fp32.  Replaces the FFMA kernels for the flagship shape (C=8, H=48, L=2) in
 * eval mode; x = the caller's batch-first fp32 windows [B][T][8].  `packed` = na_decoder_pack_x3 output
 * (na_decoder_packed_x3_bytes() bytes).
 */
int64_t na_decoder_packed_x3_bytes(void);
int na_decoder_pack_x3(const float* w_ih0, const float* w_hh0, const float* b_ih0, const float* b_hh0,
                       const float* w_ih1, const float* w_hh1, const float* b_ih1, const float* b_hh1,
                       void* packed, na_stream_t stream);
int na_decoder_infer_x3(const float* x, const void* packed,
                        const float* attn_w, const float* attn_b, const float* ln_w, const float* ln_b,
                        const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                        float* logits, float* probs, int64_t T, int64_t B, int64_t NC, na_stream_t stream);
/* ... with the intermediates outputs (see na_head_fwd_f32_ex). */
int na_decoder_infer_x3_ex(const float* x, const void* packed,
                           const float* attn_w, const float* attn_b, const float* ln_w, const float* ln_b,
                           const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                           float* logits, float* probs, float* scores_tm, float* pooled, float* embedding,
                           int64_t T, int64_t B, int64_t NC, na_stream_t stream);
/* The two LSTM layers alone, as nn.LSTM(8, 48, num_layers=2, batch_first=True) in eval mode, with the same arithmetic:
 * no pooling and no head.  Accuracy against float64 (max|d| / max|ref| per tensor): h_n / c_n within 1e-5; the per-step
 * out carries the operand split's error (about 22 bits per operand) through the recurrence: 6.2e-5 over 625 steps of
 * the shipped EEG windows, where fp32 FFMA arithmetic gives 6.5e-6 (na_lstm_layer_fwd_f32).  h_init / c_init [2][B][48] = the initial state (both or neither; NULL = zeros);
 * out [B][T][48] = the last layer's h at every step; h_n / c_n [2][B][48] = both layers' h and c after the last step.
 * Only rows b < B are written; every pointer 16-byte aligned. */
int na_decoder_lstm_x3(const float* x, const void* packed, const float* h_init, const float* c_init, float* out,
                       float* h_n, float* c_n, int64_t T, int64_t B, na_stream_t stream);

/* ---- tensor-core tier, wide hidden sizes (H = 96, 144, 192; BASELINE configs[4]: H = 192, T = 2500) --------
 * Same contract as na_decoder_infer_bf16 (lstm_eeg_model.py:32-39 + :97, eval mode; input_size 8, 2 layers),
 * for EEG_LSTM(hidden_size = H).  [W_ih | b | W_hh] no longer fits in shared memory, so the kernel keeps
 * the ACTIVATIONS resident (three rotating h buffers per SM) and streams the weights through a TMA ring
 * from an L2-resident image in MMA consumption order; cell state and pooling accumulators live in
 * `state` (na_decoder_wide_state_bytes(H) bytes, caller-allocated scratch, contents irrelevant between calls;
 * one buffer per concurrent launch).
 *   na_decoder_pack_wide_bf16: the 8 nn.LSTM tensors + attn.weight [1,H] + attn.bias [1] -> `packed`
 *       (na_decoder_wide_packed_bytes(H) bytes).  Both size queries return -1 for an unsupported H.
 *   na_decoder_infer_wide_bf16: x as for na_decoder_infer_bf16 -> logits [B,NC] (+ probs if not NULL).
 */
int64_t na_decoder_wide_packed_bytes(int64_t H);
int64_t na_decoder_wide_state_bytes(int64_t H);
int na_decoder_pack_wide_bf16(const float* w_ih0, const float* w_hh0, const float* b_ih0, const float* b_hh0,
                              const float* w_ih1, const float* w_hh1, const float* b_ih1, const float* b_hh1,
                              const float* attn_w, const float* attn_b, void* packed, int64_t H, na_stream_t stream);
int na_decoder_infer_wide_bf16(const void* x_bf16_tmp, const void* packed, const float* ln_w, const float* ln_b,
                               const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                               void* state, float* logits, float* probs,
                               int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC, na_stream_t stream);
/* ... with the intermediates outputs (see na_head_fwd_f32_ex; pooled / embedding are [B][H]). */
int na_decoder_infer_wide_bf16_ex(const void* x_bf16_tmp, const void* packed, const float* ln_w, const float* ln_b,
                                  const float* fc0_w, const float* fc0_b, const float* fc3_w, const float* fc3_b,
                                  void* state, float* logits, float* probs, float* scores_tm, float* pooled,
                                  float* embedding, int64_t T, int64_t B, int64_t Bp, int64_t H, int64_t NC,
                                  na_stream_t stream);

/* ---- tensor-core tier, training (bf16 operands; fp32 accumulate, cell state, gradients) ------------
 * Layouts: TMP fp32 [T][Bp][48]; TCL bf16 [T][Bp/128][F/8][128][8] (tile-chunk layout: a tile's
 * step-t slab is contiguous and already in the UMMA core-matrix layout); mask u8 [T][Bp][48].
 * Bp must be a multiple of 128.  Flagship shape only (C=8, H=48, L=2).
 *
 * na_lstm2_fwd_train_bf16: x (16-bit TMP, na_window_zscore) -> h0 (TCL), h0d = h0*mask*scale (TCL; NULL
 *   when there is no dropout), c0, c1 (TCL32: fp32 [T][Bp/128][12][128][4]), h1 (TCL).  Replaces
 *   `self.lstm(x)` (lstm_eeg_model.py:34) in train mode.  The attention pool of lstm_eeg_model.py:35-37 is
 *   either fused (zpool [B,48] + stats [B,2] = (max, sum) of the softmax over time; needs attn_w, attn_b, B)
 *   or left to na_head_fwd_f32 (then h1f, a fp32 TMP copy of h1, is written instead).
 * na_lstm_bwd_bf16: fused BPTT + weight gradients of one layer (layer = 0 | 1).  act_in = the layer's
 *   input (x for layer 0, h0d/h0 for layer 1; TCL), h = its raw output (TCL), cstate / dh_out (TMP).
 *   Gates are recomputed on the tensor cores; d(gates) never leave shared memory; dW_ih / dW_hh / db
 *   accumulate in TMEM in fp32 and are reduced over CTAs in a fixed order.  Layer 1 also writes
 *   din = d(act_in) * in_mask * drop_scale (TCL32) = dh_out of layer 0.  Exactly one of dh_out (TMP for layer
 *   1, TCL32 for layer 0) and dz (layer 1 only: fused head backward, see below) is given.
 *   packed_fwd = na_decoder_pack_bf16 output; zeros = >= 12,288 B of zeros; scratch =
 *   36,864 + 4 * na_train_bf16_partial_floats() bytes.
 */
/* Dropout of the tier: either an explicit keep-mask tensor (mask != NULL) or, with mask == NULL and
 * thresh16 < 65536, a counter-based in-kernel generator: unit block (t*Bp + b, blk) keeps a unit with
 * probability thresh16/65536 as a pure function of (seed, row, blk) -- the backward regenerates the
 * forward's mask, no mask tensor exists.  thresh16 == 65536 and mask == NULL: no dropout.
 * na_dropout_mask_u8 materialises that mask ([T][Bp][48] u8) for tests.  * HALF TILES (half_stride > 0; strong scaling at small batches): a tile holds 64 distinct windows, rows 64..127 of the
 * input (the caller replicates them), of h0 / h0d / h1 (the kernels write both copies) mirror rows 0..63, and the two
 * copies of a window split its hidden units, so a tile costs about half a step and B windows occupy B / 64 SMs.  Window b
 * lives in rows (b / 64) * 128 + b % 64 (+ 64); B <= Bp / 2; half_stride = the row stride of the counter-based dropout
 * generator's key (the full-tile padded batch, so that both layouts draw the same mask).  Pass 0 for full tiles.
 */
int na_dropout_mask_u8(uint64_t seed, int64_t thresh16, int64_t T, int64_t Bp, unsigned char* out, na_stream_t stream);
int64_t na_train_bf16_partial_floats(void);
int na_lstm2_fwd_train_bf16(const void* x_bf16_tmp, const void* packed, const unsigned char* mask,
                            uint64_t seed, int64_t thresh16, float drop_scale, void* h0, void* h0d, float* c0, void* h1, float* h1f,
                            float* c1, const float* attn_w, const float* attn_b, float* zpool, float* stats,
                            int64_t B, int64_t T, int64_t Bp, int64_t half_stride, na_stream_t stream);
int na_lstm_bwd_bf16(int64_t layer, const void* act_in, const void* h, const float* cstate,
                     const float* dh_out, const void* packed_fwd, const float* w_ih, const float* w_hh,
                     const void* zeros, const unsigned char* in_mask, uint64_t seed, int64_t thresh16,
                     float drop_scale, float* din, float* dw_ih, float* dw_hh, float* db, void* scratch,
                     const float* dz, const float* stats, const float* zpool, const float* attn_w,
                     const float* attn_b, int64_t B, float* d_attn,
                     int64_t T, int64_t Bp, int64_t half_stride, na_stream_t stream);

/* Tail-only forms of K4 for the fused tier: na_lstm2_fwd_train_bf16 already pooled (zpool, stats), and
 * na_lstm_bwd_bf16(layer 1, dz != NULL) rebuilds dh_t = alpha_t dz + ds_t w_a per step and owns d attn_w /
 * d attn_b (d_attn [49]).  na_head_tail_bwd_f32 zeroes the attn slots of `dparams`. */
int na_head_tail_fwd_f32(const float* zpool, const float* attn_w, const float* attn_b, const float* ln_w,
                         const float* ln_b, const float* fc0_w, const float* fc0_b, const float* fc3_w,
                         const float* fc3_b, const float* rrelu_slope, const float* drop_mask, float drop_scale,
                         float* logits, float* probs, int64_t B, int64_t H, int64_t NC, na_stream_t stream);
int na_head_tail_bwd_f32(const float* dlogits, const float* zpool, const float* attn_w, const float* attn_b,
                         const float* ln_w, const float* ln_b, const float* fc0_w, const float* fc0_b,
                         const float* fc3_w, const float* fc3_b, const float* rrelu_slope, const float* drop_mask,
                         float drop_scale, float* dz, float* dparams, float* partials,
                         int64_t B, int64_t H, int64_t NC, na_stream_t stream);

/* ---- exact tier TRAINING on the tensor cores (fp32 accuracy, 1e-5 contract on logits and gradients) -----------
 * Replaces torch autograd of lstm_eeg_model.py:32-39 (SURVEY a15) at the flagship shape (C=8, H=48, 2 layers) with the
 * operand-split scheme of na_decoder_infer_x3 (fp16 hi + lo, three tcgen05 MMAs per product, fp32 accumulate, ex2 / rcp
 * activations).  One launch per layer and direction (csrc/na_train_x3.cu).  Layouts, all for 128-window tiles
 * (NT = Bp / 128, chunk = [128 rows][8 fp16]):
 *   XS    fp16 [T][NT][2][128][8]    x / 16 split into hi (chunk 0) and lo (chunk 1)       na_x3_split_input
 *   TCLX  fp16 [T][NT][12][128][8]   h split: chunks 0-5 hi (units 8c..8c+7), 6-11 lo
 *   TCL32 fp32 [T][NT][12][128][4]   cell state, din
 *   DGX   fp16 [T][NT][48][128][8]   d(gates) split: chunks 0-23 hi, 24-47 lo; column n = (j/4)*16 + gate*4 + j%4
 *         (half tiles, half_stride > 0: [T][NT][48][64][8] -- only the 64 real window rows of a tile are stored)
 * `packed_x3` = na_decoder_pack_x3 output.  Inter-layer dropout as in the 16-bit tier: explicit u8 keep-mask [T][Bp][48]
 * or (mask NULL, thresh16 < 65536) the counter-based generator keyed by `seed`; thresh16 = 65536: none.
 *   na_lstm_fwd_train_x3  layer 0: in = XS -> h (TCLX), hd = h after dropout (TCLX, exactly when dropout is on), c;
 *                         layer 1: in = TCLX (hd or h of layer 0) -> h, c, pooled z [B][48], softmax stats (max, sum) [B][2]
 *   na_lstm_bwd_x3        BPTT of one layer: d(gates) -> dg (DGX); layer 1 also din (TCL32, dropout applied) and, with
 *                         dz != NULL, the time loop of the head backward fused (dh_in must be NULL then), d_attn [52] =
 *                         d attn_w (48) | d attn_b | pad; layer 0: dh_in = din of layer 1.  zeros: >= 24,576 zero bytes.
 *                         scratch: na_train_x3_scratch_floats() floats.
 *   na_lstm_bwd_x3_dx     na_lstm_bwd_x3 for input attributions: the same BPTT without its weight-gradient byproducts (no dg,
 *                         no d_attn, no scratch); layer 0 also writes dx = d/dx of the layer-0 input, fp32 batch-first
 *                         [B][T][8], rows b < B only, each multiplied by dz_inv_scale[b] ([B], the inverse of the factor
 *                         that window's dz was scaled by).
 *   na_lstm_wgrad_x3      time-parallel dW_ih, dW_hh, db (= both biases) from dg and the saved activations; same scratch.
 * half_stride > 0 selects HALF TILES exactly as in na_lstm2_fwd_train_bf16 (64 windows per tile, rows 64..127 mirror rows
 * 0..63, B <= Bp / 2, half_stride = the dropout generator's row stride); 0 = full tiles.
 */
int na_x3_split_input(const float* x, void* xs, int64_t B, int64_t T, int64_t Bp, int64_t half_stride, na_stream_t stream);
int na_lstm_fwd_train_x3(int64_t layer, const void* in, const void* packed_x3, const float* attn_w, const float* attn_b,
                         const unsigned char* mask, uint64_t seed, int64_t thresh16, float drop_scale, void* h, void* hd,
                         float* c, float* zpool, float* stats, int64_t B, int64_t T, int64_t Bp, int64_t half_stride,
                         na_stream_t stream);
int64_t na_train_x3_scratch_floats(void);
int64_t na_train_x3_smem_bytes(int64_t which);
int na_lstm_bwd_x3(int64_t layer, const void* act_in, const void* h, const float* cstate, const float* dh_in,
                   const void* packed_x3, const void* zeros, const unsigned char* in_mask, uint64_t seed, int64_t thresh16,
                   float drop_scale, float* din, void* dg, const float* dz, const float* stats, const float* zpool,
                   const float* attn_w, const float* attn_b, int64_t B, float* d_attn, float* scratch,
                   int64_t T, int64_t Bp, int64_t half_stride, na_stream_t stream);
int na_lstm_bwd_x3_dx(int64_t layer, const void* act_in, const void* h, const float* cstate, const float* dh_in,
                      const void* packed_x3, const void* zeros, const unsigned char* in_mask, uint64_t seed, int64_t thresh16,
                      float drop_scale, float* din, const float* dz, const float* stats, const float* zpool,
                      const float* attn_w, const float* attn_b, int64_t B, float* dx, const float* dz_inv_scale,
                      int64_t T, int64_t Bp, int64_t half_stride, na_stream_t stream);
int na_lstm_wgrad_x3(int64_t layer, const void* dg, const void* act_in, const void* h, const void* zeros,
                     float* dw_ih, float* dw_hh, float* db, float* scratch, int64_t T, int64_t Bp, int64_t half_stride,
                     na_stream_t stream);

/* ---- wide decoders (H = 96 / 144 / 192, BASELINE configs[4]): TRAINING on the tensor cores, 16-bit tier -----------
 * Replaces torch autograd of lstm_eeg_model.py:32-39 with hidden_size > 48 (SURVEY a15, config 5) for the serial part of a
 * layer; everything parallel over time (input projection, din, weight gradients) is a plain GEMM done by the caller.
 * Per-thread vectors use the wide tile layout WTL [T][NT][H/48][3][P][128][16 B] (NT = Bp / 128; thread = window row x 16-unit
 * group g of 48-unit task k; gates / d(gates): E = 64 fp16 in accumulator column order (u/4)*16 + gate*4 + u%4;
 * h: 16 fp16; c, dh: 16 fp32).
 *   na_lstm_wide_fwd_train  gx = in . W_ih^T + b (WTL, fp16) -> activated gates, h, c for every step.
 *                           w_image: [H/48][H/16][2][192][8] fp16 = W_hh rows of a task (accumulator column order) x K16 slices.
 *   na_lstm_wide_bwd        gates, c, dh_in (WTL) -> dg (WTL) with dh_rec = dG . W_hh carried through the steps.
 *                           w_image: [H/48][12][2][H][8] fp16 = W_hh^T, K = the task's 192 gate columns.
 *                           workspace: na_wide_train_ws_floats(H) floats (running d(cell), L2-resident).
 */
int64_t na_wide_train_ws_floats(int64_t H);
int na_lstm_wide_fwd_train(const void* gx, const void* w_image, void* gates, void* h, float* c, int64_t T, int64_t Bp,
                           int64_t H, na_stream_t stream);
int na_lstm_wide_bwd(const void* gates, const float* c, const float* dh_in, const void* w_image, void* dg, float* workspace,
                     int64_t T, int64_t Bp, int64_t H, na_stream_t stream);

/* ---- phase-coupling preprocessing filter (SURVEY 8(f) rank 1), OPT-IN ---------------------------------------------
 * Replaces, for batches of windows, Utilities/preprocessor.py:21-36 -> MindsAI/mindsai_filter_python/core.py:14-48 (the
 * step in front of the decoder on every live window): analytic signal per channel (Hilbert transform), pairwise
 * sum_t sin^2(phase_i - phase_j), diagonal renormalisation (EPS = 1e-12), M = (I + lambd P^T P)^-1, y = M x.
 * x, y fp32 [B][625][8] (batch-first windows as the reference stores them: samples x channels); arithmetic in float64.
 * twiddle = exp(-2 pi i k / 625), k = 0..624, as 1250 doubles (re, im); status: one int, set to 1 if a matrix was singular.
 * The method is third-party (MindsApplied, patent pending; the reference implementation is Polyform-Noncommercial):
 * written from the published mathematics, never enabled by default (preprocess_gpu.PhaseCouplingFilterGPU).
 */
int na_phase_coupling_filter(const float* x, float* y, const double* twiddle, double lambd, int* status,
                             int64_t B, int64_t T, int64_t C, na_stream_t stream);

/* ---- optimizer step (train step of SURVEY 8(d): "Adam lr 1e-3 in torch") --------------------------------------------
 * torch.optim.Adam's update (no amsgrad) for a whole list of fp32 tensors in ONE launch.  table (device): n_tensors x
 * {param ptr, grad ptr, exp_avg ptr, exp_avg_sq ptr, numel} as int64; grad_scale: optional device scalar multiplied into every
 * gradient (NULL = 1); bias_correction{1,2} = 1 - beta^step, computed by the caller.
 */
int na_adam_multi(const int64_t* table, int64_t n_tensors, int64_t max_numel, float lr, float beta1, float beta2, float eps,
                  float weight_decay, float bias_correction1, float bias_correction2, const float* grad_scale,
                  na_stream_t stream);

/* ---- K5: trial averaging -----------------------------------------------------------------
 * Replaces tester.py:54,89,97 (and :90,98 for the chunk): fp32 zeros, += in trial order
 * r = 0..R-1, then one IEEE division by R.   in [R][N] -> out [N].
 */
int na_trial_mean_f32(const float* in, float* out, int64_t R, int64_t N, na_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NEUROALPHA_H_ */
