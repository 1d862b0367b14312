/*
 * cmwg_b200 -- C ABI of the B200-native flow hot path of constant-memory-waveglow.
 *
 * The reference (yoyololicon/constant-memory-waveglow) is pure PyTorch and has no FFI of its own;
 * each entry point below replaces the stock-library kernels that one reference call site
 * dispatches to.  The reference file:line each one stands in for is cited (paths relative to the
 * reference repository root).  The Python host side (constant_memory_waveglow_b200/*.py) binds
 * these with ctypes and mirrors the reference's nn.Module / autograd.Function surface.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless stated otherwise;
 *   - every function returns CMWG_OK (0) or a negative error code and never throws;
 *     cmwg_last_error() returns a thread-local, NUL-terminated description of the last failure;
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued, never synchronised;
 *   - "NCL" = (batch, channel, time) with time contiguous, the layout PyTorch's Conv1d uses;
 *     *_bstride arguments are the batch stride in elements so channel-slices of a larger tensor
 *     can be passed without a copy;
 *   - "slab" = the internal channel-last layout [batch][time][channel] used between WN layers.
 */
#ifndef CMWG_B200_H
#define CMWG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CMWG_OK 0
#define CMWG_ERR_ARG (-1)
#define CMWG_ERR_CUDA (-2)
#define CMWG_ERR_UNSUPPORTED (-3)

#define CMWG_MAX_DEPTH 16

/* precision of the WN GEMM operands (accumulation, flow state, coupling and log-det are fp32) */
#define CMWG_PREC_FP32 0 /* exact: CUDA-core FFMA engine                                   */
#define CMWG_PREC_BF16 1 /* tcgen05 kind::f16, bf16 operands, fp32 accumulate in TMEM       */
#define CMWG_PREC_FP16 2 /* tcgen05 kind::f16, fp16 operands (TF32's mantissa); the backward     */
                         /* runs on a power-of-two multiple of the cotangent chosen on the device */

const char* cmwg_last_error(void);
int cmwg_version(void);
/* cumulative number of kernels this library has launched in this process */
unsigned long long cmwg_launch_count(void);
void cmwg_reset_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Invertible 1x1 convolution  (model/efficient_modules.py:17-54, 215-279)
 * ------------------------------------------------------------------------------------------- */

/* LU of a c x c fp32 matrix on the device (c <= 64): w_inv = W^-1, *logdet = log(det W), NaN when
 * det W <= 0 exactly like Tensor.logdet().  Replaces weight.squeeze().logdet() / .inverse()
 * (model/efficient_modules.py:39,52-53,221,235,254-256,272). */
int cmwg_small_inverse_logdet(const float* w, int c, float* w_inv, float* logdet, void* stream);

/* z[b,:,t] = M x[b,:,t] with M = W (transpose_w = 0) or W^T (transpose_w = 1); W is c x c row
 * major.  Replaces F.conv1d(x, weight) with kernel size 1
 * (model/efficient_modules.py:40,53,223,237,239,256,269,273). */
int cmwg_conv1x1_apply(const float* w, int transpose_w, const float* x, long long x_bstride, float* z,
                       long long z_bstride, int B, int C, int T, void* stream);

/* dm[o][i] = sum_{b,t} dz[b,o,t] * x[b,i,t]   (model/efficient_modules.py:240-241,274-275).
 * Deterministic two-pass reduction; `workspace` must hold cmwg_conv1x1_wgrad_workspace(B,C,T) bytes. */
size_t cmwg_conv1x1_wgrad_workspace(int B, int C, int T);
int cmwg_conv1x1_wgrad(const float* dz, long long dz_bstride, const float* x, long long x_bstride, int B, int C,
                       int T, float* dm, void* workspace, void* stream);

/* dW from dm (model/efficient_modules.py:242 and :276-277):
 *   inverse_mode = 0:  dW = dm + W^-T * (*dlogdet) * T
 *   inverse_mode = 1:  dW = -W^-T dm W^-T - W^-T * (*dlogdet) * T
 * w_inv is the c x c inverse; dlogdet points at one device float. */
int cmwg_conv1x1_dw_finalize(const float* dm, const float* w_inv, const float* dlogdet, int c, int T,
                             int inverse_mode, float* dw, void* stream);

/* The whole of Conv1x1Func.backward / InvConv1x1Func.backward (model/efficient_modules.py:229-244, 262-279) in two launches
 * for even C <= 8 (any other shape runs the separate entry points above, same arithmetic).  With M = W (inverse_mode 0) or
 * W^-1 (1) the forward call was out = M in:
 *   restored (B, C, T; may be NULL) <- in = M^-1 out       the freed input, re-materialised
 *   din      (B, C, T)             <- M^T dout
 *   dw       (C, C; may be NULL)   <- dm + W^-T dlogdet T   resp.  -W^-T dm W^-T - W^-T dlogdet T,  dm = sum dout in^T
 * w_inv = W^-1 as cmwg_small_inverse_logdet returned it in the forward pass; dlogdet: one device float (NULL = 0);
 * workspace: cmwg_conv1x1_backward_workspace(B, C, T) bytes (only needed with dw). */
size_t cmwg_conv1x1_backward_workspace(int B, int C, int T);
int cmwg_conv1x1_backward(const float* w, const float* w_inv, int inverse_mode, const float* out, long long out_bstride,
                          const float* dout, long long dout_bstride, const float* dlogdet, int B, int C, int T,
                          float* restored, long long restored_bstride, float* din, long long din_bstride, float* dw,
                          void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Affine coupling  (model/efficient_modules.py:57-212)
 * `lst` is the WN output, NCL (B, 2*cin, T): channels [0,cin) = log_s, [cin,2cin) = t.
 * ------------------------------------------------------------------------------------------- */

/* inverse = 0 (:105-111): z = cat(xa, xb*exp(log_s)+t)
 * inverse = 1 (:163-169): z = cat(xa, (xb-t)/exp(log_s)); neg_log_s (B,cin,T contiguous, may be
 * NULL) receives -log_s. */
int cmwg_coupling_apply(const float* x, long long x_bstride, const float* lst, float* z, long long z_bstride,
                        float* neg_log_s, int B, int cin, int T, int inverse, void* stream);

/* cmwg_coupling_apply for a padded batch with per-item lengths (lengths_dev: B device ints, in columns of T): the same
 * values at columns t < lengths_dev[b]; z (both halves) and neg_log_s are written as 0 at t >= lengths_dev[b]. */
int cmwg_coupling_apply_varlen(const float* x, long long x_bstride, const float* lst, float* z, long long z_bstride,
                               float* neg_log_s, int B, int cin, int T, const int* lengths_dev, int inverse, void* stream);

/* The elementwise half of AffineCouplingFunc.backward (:132-148, inverse = 0) and of
 * InvAffineCouplingFunc.backward (:190-207, inverse = 1).  Given the saved OUTPUT `out` of the
 * forward call, the recomputed `lst`, and the incoming cotangents (dout for the tensor output,
 * dls for the returned +-log_s), it
 *   - re-materialises the forward call's INPUT into `restored` (B, 2cin, T contiguous),
 *   - writes the cotangent of the WN output into `dlst` (B, 2cin, T contiguous),
 *   - writes din[:, cin:] (the 'b' half of the input gradient) and copies dout[:, :cin] into
 *     din[:, :cin] (the WN backward later ACCUMULATES its dxa into that half). */
int cmwg_coupling_bwd(const float* out, long long out_bstride, const float* lst, const float* dout,
                      long long dout_bstride, const float* dls, long long dls_bstride, float* restored, float* dlst,
                      float* din, int B, int cin, int T, int inverse, void* stream);

/* ---------------------------------------------------------------------------------------------
 * WN transform  (model/waveglow.py:13-105), weight norm (utils.py:9-16)
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int in_channels;   /* cin: channels of xa and of each of log_s / t  (WN in_channels)   */
  int aux_channels;  /* conditioning channels                                              */
  int dil_channels;  /* Cd (gate channels; W produces 2*Cd)                                */
  int res_channels;  /* Cr                                                                 */
  int skip_channels; /* Cs                                                                 */
  int depth;         /* number of NonCausalLayers, dilation 2^i                            */
  int radix;         /* kernel size of W (odd)                                             */
  int has_bias;      /* bias=True in the reference constructor                             */
  int precision;     /* CMWG_PREC_*                                                        */
  /* 2-D WN of WaveFlow (model/waveflow.py:14-151).  height <= 1: the 1-D WN above.  height = H > 1: activations
   * are (B, C, H, T) images, W is a radix x radix Conv2d with dilation (h_dilation[i], 2^i), causal in the
   * height dimension (top padding 2*h_dilation, :42,57) and 'same' in time; the conditioning has no height
   * dimension (V(y).unsqueeze(2), :131).  x / lst / dx are then NCL tensors over the FLATTENED (h, t) axis and
   * the `T` argument of every entry point is the WIDTH of one line. */
  int height;
  int h_dilation[CMWG_MAX_DEPTH];
} cmwg_wn_config;

/* One convolution's parameters.  With weight norm attached: g = weight_g (out,1,1), v = weight_v;
 * after remove_weight_norms (or for `end`, which never has weight norm): g = NULL, v = weight. */
typedef struct {
  const float* g;
  const float* v;
  const float* bias; /* NULL when has_bias == 0 */
} cmwg_conv_param;

typedef struct {
  cmwg_conv_param V;     /* (2*Cd*depth, aux, 1)                   model/waveglow.py:70-72 */
  cmwg_conv_param start; /* (Cr, cin, 1)                           model/waveglow.py:74-75 */
  cmwg_conv_param W[CMWG_MAX_DEPTH];   /* (2*Cd, Cr, radix)        model/waveglow.py:29-30 */
  cmwg_conv_param W_o[CMWG_MAX_DEPTH]; /* (Cr+Cs | Cs, Cd, 1)      model/waveglow.py:33-38 */
  cmwg_conv_param end;   /* (2*cin, Cs, 1), never weight-normed    model/waveglow.py:92    */
} cmwg_wn_params;

/* gradient destinations, same shapes as the parameters; any pointer may be NULL (skipped) */
typedef struct {
  float* g;
  float* v;
  float* bias;
} cmwg_conv_grad;

typedef struct {
  cmwg_conv_grad V, start, W[CMWG_MAX_DEPTH], W_o[CMWG_MAX_DEPTH], end;
} cmwg_wn_grads;

/* Is the tcgen05 engine usable for this configuration (channel counts multiples of 64, ...)?
 * Returns 1/0.  When 0, precision must be CMWG_PREC_FP32. */
int cmwg_wn_tc_supported(const cmwg_wn_config* cfg);

/* Padded channel count of the slab-layout conditioning tensor for this config/precision. */
int cmwg_wn_aux_padded(const cmwg_wn_config* cfg);

/* y (B, aux, T) fp32 with arbitrary element strides -> slab [B][T][aux_padded] in the operand type
 * of cfg->precision (zero padded).  Done once per conditioning tensor and shared by all flows.
 * Replaces nothing in the reference (its V conv reads y directly, model/waveglow.py:100); it is the
 * layout change that lets V be folded into the dilated-conv GEMM as extra K rows.
 * The PADDING columns [aux, aux_padded) of the slab belong to the library afterwards: cmwg_wn_forward and
 * cmwg_wn_backward keep the taps of xa there when they fold the start conv into layer 0 (DESIGN 3.9), although they take
 * the slab as `const void*` (its conditioning columns are never written).  One slab must therefore not be used by
 * concurrent calls on different streams; sequential calls (the flows of one model) may share it. */
int cmwg_cond_pack(const cmwg_wn_config* cfg, const float* y, long long y_bstride, long long y_cstride,
                   long long y_tstride, int B, int T, void* ycl, void* stream);
/* dy (B, aux, T) contiguous fp32 <- slab gradient [B][T][aux_padded] fp32 */
int cmwg_cond_unpack_grad(const cmwg_wn_config* cfg, const float* dycl, int B, int T, float* dy, void* stream);

/* Effective weights (g*v/||v||, utils.py:14-16 -> torch weight_norm) packed for the GEMM engines. */
size_t cmwg_wn_packed_bytes(const cmwg_wn_config* cfg);
int cmwg_wn_pack(const cmwg_wn_config* cfg, const cmwg_wn_params* params, void* packed, void* stream);

size_t cmwg_wn_workspace_bytes(const cmwg_wn_config* cfg, int B, int T);
/* host-side listing of the single-kernel WN forward (backward = 0) / backward chain (1) task lists, for the dependency-order
 * tests: entry i -> out[4i..4i+3] = (type, layer, row tile, N tile); *total entries, *lag row-tile slots */
int cmwg_mega_task_list(int backward, int depth, int B, int T, int* out, int cap, int* total, int* lag);
/* host-side split-K plan of a batched weight-gradient launch (for the plan's tests): `tiles` output tiles of `bn` columns
 * whose K runs over B batch items x T time steps -> number of splits (DESIGN 3.9: rounds x K per round, minimised) */
int cmwg_wgrad_plan_splits(int tiles, int bn, int B, int T);
/* tools only: 0 = TMA descriptor encodes so far (cache misses), 1 = descriptor cache clears */
unsigned long long cmwg_debug_counter(int which);
/* tools only: cycle accumulators [CTA][18 warps][16] of the last single-kernel WN forward launched with CMWG_MEGA_CLK=1 */
int cmwg_mega_clk_read(long long* host, int n);
/* bytes of per-layer activations kept between cmwg_wn_forward(save != NULL) and cmwg_wn_backward */
size_t cmwg_wn_saved_bytes(const cmwg_wn_config* cfg, int B, int T);

/* Inference over a padded batch with per-item lengths: item b of (x, ycl, lst) holds lengths_host[b] valid time steps of T,
 * 1 <= lengths_host[b] <= T.  lst[b, :, t] for t < lengths_host[b] is bit-identical to cmwg_wn_forward on that item alone
 * with T = lengths_host[b]; lst at t >= lengths_host[b] is unspecified (the single-kernel forward does not compute row tiles
 * that hold no valid step).  lengths_host plans the work on the host; lengths_dev is a device int[B] holding the SAME values,
 * uploaded by the caller (the library never allocates or copies it).  workspace: cmwg_wn_varlen_workspace_bytes(cfg, B, T).
 * No `saved` (training on per-item lengths is not supported).  Returns CMWG_ERR_ARG for a length outside [1, T] and
 * CMWG_ERR_UNSUPPORTED for the 2-D WN (height > 1). */
size_t cmwg_wn_varlen_workspace_bytes(const cmwg_wn_config* cfg, int B, int T);
int cmwg_wn_forward_varlen(const cmwg_wn_config* cfg, const void* packed, const float* x, long long x_bstride,
                           const void* ycl, int B, int T, const int* lengths_host, const int* lengths_dev, void* workspace,
                           float* lst, void* stream);
/* host-side listing of the single-kernel WN forward's task list for per-item lengths (host array `lengths`): out / total / lag as
 * cmwg_mega_task_list(0, ...); *row_tiles = sum_b ceil(lengths[b] / 256) compacted row tiles and tiles[3 rt .. 3 rt + 2] =
 * (item, tile within the item, tiles of the item) for rt < min(*row_tiles, tiles_cap) */
int cmwg_mega_task_list_varlen(int depth, int B, int T, const int* lengths, int* out, int cap, int* total, int* lag, int* tiles,
                               int tiles_cap, int* row_tiles);

/* (log_s, t) = WN(xa, y)   (model/waveglow.py:98-105 with NonCausalLayer.forward :41-46 and
 * fused_gate :13-15).  xa = first cin channels of x (NCL, batch stride x_bstride);
 * lst (B, 2cin, T) contiguous.  `saved` = NULL for inference, else a buffer of
 * cmwg_wn_saved_bytes() that cmwg_wn_backward consumes. */
int cmwg_wn_forward(const cmwg_wn_config* cfg, const void* packed, const float* x, long long x_bstride,
                    const void* ycl, int B, int T, void* workspace, void* saved, float* lst, void* stream);

/* Row-recurrent evaluation of the 2-D WN (cfg->height = H > 1), the engine of WaveFlow's inverse
 * (model/waveflow.py:53-67 NonCausalLayer2D.reverse_mode_forward, :137-151 WN2D.reverse_mode_forward, :243-258 the
 * per-row loop).  Computes lst for lines [line_begin, line_begin + line_count) only.  `state`
 * (cmwg_wn_line_state_bytes) keeps every layer's input for ALL lines -- the reference's rolling per-layer
 * `buffer_list` -- so a tap at line h - k*h_dilation reads what an earlier call left there; lines must therefore be
 * generated in increasing order, and lines above 0 read as zeros exactly like the reference's F.pad (:57).
 * x / lst are the same full-height tensors cmwg_wn_forward takes; only the window's lines are read / written. */
size_t cmwg_wn_line_state_bytes(const cmwg_wn_config* cfg, int B, int T);
int cmwg_wn_forward_lines(const cmwg_wn_config* cfg, const void* packed, const float* x, long long x_bstride,
                          const void* ycl, int B, int T, int line_begin, int line_count, void* workspace, void* state,
                          float* lst, void* stream);

/* Gradient of WN given dlst (B, 2cin, T): the autograd.grad call of
 * model/efficient_modules.py:139-144 / :198-203 for F = WN.
 *   dxa: ACCUMULATED (+=) into dx (NCL, batch stride dx_bstride, first cin channels);
 *   dycl: NULL or slab fp32 [B][T][aux_padded], OVERWRITTEN with the conditioning gradient;
 *   grads: weight gradients in the reference's parameterisation (weight_g / weight_v or weight),
 *          OVERWRITTEN. */
int cmwg_wn_backward(const cmwg_wn_config* cfg, const cmwg_wn_params* params, const void* packed,
                     const float* x, long long x_bstride, const void* ycl, int B, int T, void* workspace,
                     const void* saved, const float* dlst, float* dx, long long dx_bstride, float* dycl,
                     const cmwg_wn_grads* grads, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Conditioning upsampler (model/waveglow.py:126-130, 210-212): depthwise ConvTranspose1d with
 * weight norm and bias.  h (B, C, F) -> y (B, C, (F-1)*stride - 2*pad + K).
 * ------------------------------------------------------------------------------------------- */
int cmwg_upsample_fwd(const float* h, const float* g, const float* v, const float* bias, int B, int C, int F,
                      int K, int stride, int pad, float* y, void* stream);
/* dy (B, C, Tout) with element strides -> dg (C), dv (C,K), dbias (C); g == NULL => dv is d(weight) */
size_t cmwg_upsample_bwd_workspace(int B, int C, int K);
int cmwg_upsample_bwd(const float* h, const float* g, const float* v, const float* dy, long long dy_bstride,
                      long long dy_cstride, int B, int C, int F, int K, int stride, int pad, int Tvalid, float* dg,
                      float* dv, float* dbias, void* workspace, void* stream);
/* Gradient w.r.t. the upsampler INPUT (needed when the conditioning itself is trainable, e.g. the embedding
 * tables of WSRGlow, model/wsrglow.py:27-31,52-53):  dh[b,c,f] = sum_k w_eff[c,k] dy[b,c,f*stride-pad+k]. */
int cmwg_upsample_bwd_input(const float* g, const float* v, const float* dy, long long dy_bstride,
                            long long dy_cstride, int B, int C, int F, int K, int stride, int pad, int Tvalid,
                            float* dh, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Mel-spectrogram conditioner (model/condition.py:7-19; called at model/lightning.py:54 and inference.py:31):
 * ReflectionPad1d((n_fft/2 - hop/2, n_fft/2 + hop/2)) -> STFT(n_fft, hop, window, center=False) -> |.|^power ->
 * mel filterbank -> (+ eps) -> log, fused in one kernel.
 *   x (B, T) with batch stride x_bstride -> out (B, n_mels, frames), frames = cmwg_melspec_frames(T, n_fft, hop).
 *   window (n_fft); fbt (n_mels, n_fft/2 + 1) row major = the TRANSPOSE of torchaudio's mel_scale.fb, so a warp
 *   reads consecutive bins of one band; fb_lo / fb_hi (n_mels) int32: band m is non-zero only on bins
 *   [fb_lo[m], fb_hi[m]).  n_fft: power of two in [128, 4096].
 *   power_is_one: 0 -> power 2 (the default), 1 -> magnitude; take_log = 0 returns the mel powers (+ eps).
 * ------------------------------------------------------------------------------------------- */
int cmwg_melspec_frames(int T, int n_fft, int hop);
int cmwg_melspec_fwd(const float* x, long long x_bstride, int B, int T, const float* window, const float* fbt,
                     const int* fb_lo, const int* fb_hi, int n_fft, int hop, int n_mels, int power_is_one, float eps,
                     int take_log, float* out, void* stream);
/* The same transform over a zero-padded batch with per-item lengths, a free left pad and a choice of log; serves MelSpec
 * with lengths and TacotronSTFT.mel_spectrogram (Tacotron2's layers.py / stft.py: reflect pad n_fft/2, |STFT|, mel,
 * log(clamp(., 1e-5))).  Item b is framed over its own len_b samples (len_b = lengths[b], or T when both length pointers
 * are NULL) with reflection at its own end: frame f starts at sample f * hop - pad_left, and item b has len_b / hop + 1
 * frames; out (B, n_mels, T / hop + 1) holds 0 in the frames after them.  Nothing past len_b is read, so every item equals
 * its own call (B = 1, T = len_b) bit for bit.
 *   pad_left: n_fft/2 - hop/2 for MelSpec, n_fft/2 for Tacotron2; lengths in (max(pad_left, n_fft - pad_left), T].
 *   log_mode: 0 -> v, 1 -> log(v + eps) (then equal to cmwg_melspec_fwd bit for bit when pad_left = n_fft/2 - hop/2),
 *   2 -> log(max(v, eps)); v the mel value.  eps finite and >= 0.  Other arguments as cmwg_melspec_fwd.
 *   CMWG_ERR_ARG for a bad length, log_mode, eps or n_fft. */
int cmwg_melspec_fwd_varlen(const float* x, long long x_bstride, int B, int T, const int* lengths_host,
                            const int* lengths_dev, const float* window, const float* fbt, const int* fb_lo,
                            const int* fb_hi, int n_fft, int hop, int n_mels, int pad_left, int power_is_one,
                            int log_mode, float eps, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Denoiser of synthesised audio: bias-spectrum subtraction, the `Denoiser` of NVIDIA's WaveGlow (denoiser.py, mode 'zeros',
 * used by its inference.py --denoiser_strength).  With w the window (n_fft floats; a window shorter than n_fft zero-padded and
 * centred, as torch.stft does), STFT(x) = torch.stft(x, n_fft, hop, window=w, center=True, pad_mode="reflect",
 * onesided=True): len / hop + 1 frames of n_fft/2 + 1 bins.  n_fft: power of two in [128, 4096]; 1 <= hop <= n_fft/2; the
 * window's squared overlap-add must not vanish (true for a Hann window of win_length >= 2 hop).  Lengths: n_fft/2 < len <= T
 * (reflect padding needs more samples than the pad).  Deterministic; the caller owns all memory.
 * ------------------------------------------------------------------------------------------- */
/* mag (n_fft/2 + 1 floats) <- |STFT(x)[:, frame]| of one signal x (T floats), 0 <= frame <= T / hop.  The denoiser's bias
 * spectrum is this at frame 0 of the model's output for an all-zero mel spectrogram. */
int cmwg_stft_frame_magnitude(const float* x, int T, const float* window, int n_fft, int hop, int frame, float* mag,
                              void* stream);
/* bytes of the workspace of cmwg_denoise: B * (T / hop + 1) * n_fft floats (the windowed time-domain frames) */
size_t cmwg_denoise_workspace_bytes(int B, int T, int n_fft, int hop);
/* out (B, T) contiguous <- per item b, over its first len_b samples (len_b = lengths[b], or T when both length pointers are
 * NULL): S = STFT(x_b), M = max(|S| - strength * bias_mag[:, None], 0), out_b = torch.istft(M * S / |S|, n_fft, hop, w,
 * center=True, length=len_b), with the term 0 where |S| = 0; out[b, t] = 0 for t >= len_b.  Each item's output is
 * bit-identical to a call on that item alone.  x: (B, T) at batch stride x_bstride; bias_mag: n_fft/2 + 1 floats;
 * strength >= 0.  lengths_host (host) and lengths_dev (device) hold the same B ints, or are both NULL.  workspace:
 * cmwg_denoise_workspace_bytes(B, T, n_fft, hop) bytes.  Bad sizes, lengths or strength: CMWG_ERR_ARG. */
int cmwg_denoise(const float* x, long long x_bstride, int B, int T, const int* lengths_host, const int* lengths_dev,
                 const float* window, const float* bias_mag, float strength, int n_fft, int hop, void* workspace, float* out,
                 void* stream);

/* ---------------------------------------------------------------------------------------------
 * Band-limited resampling: torchaudio.functional.resample(x, orig, new, lowpass_filter_width, rolloff, resampling_method,
 * beta) per item, with the kernel of torchaudio/functional/functional.py `_get_sinc_resample_kernel` (windowed sinc at
 * t = ((i - w) / O - j / N) * base, clamped to [-lpw, lpw]) applied as `_apply_sinc_resample_kernel` does (zero padding by
 * w on the left, conv1d with stride O, output cut to ceil(N * len / O) samples), O = orig / gcd, N = new / gcd.
 * Only the taps inside the window's support (|t| < lpw) are evaluated: table (L, N) fp32 holds, in row m and column j, tap
 * first[j] + m of torchaudio's phase j (0 past the phase's span), first (N ints) the index of its first kept tap; w is
 * torchaudio's `width`.  The host builds both (resample.py `resample_table`).
 *   y (B, T_out), T_out = ceil(N * T / O) (64-bit arithmetic), at batch stride y_bstride <- per item b, over its first
 *   len_b samples (len_b = lengths[b], or T when both length pointers are NULL; 1 <= len_b <= T):
 *   y[b, kN + j] = sum_m table[m][j] * x[b, kO + first[j] + m - w] for kN + j < ceil(N len_b / O), x read as 0 outside
 *   [0, len_b); y[b, n] = 0 after that.  Summed in ascending m with fmaf, without atomics: deterministic, and each item is
 *   bit-identical to a call on that item alone.  x: (B, T) at batch stride x_bstride.  lengths_host (host) and lengths_dev
 *   (device) hold the same B ints, or are both NULL.  Nothing is allocated.  Bad sizes or lengths: CMWG_ERR_ARG. */
int cmwg_resample(const float* x, long long x_bstride, int B, int T, const int* lengths_host, const int* lengths_dev,
                  const float* table, const int* first, int O, int N, int L, int w, float* y, long long y_bstride, int T_out,
                  void* stream);

/* ---------------------------------------------------------------------------------------------
 * Spectral distances between (reference, estimate) pairs: log-spectral distance, log-mel L1 and mel-cepstral distortion on
 * Tacotron2's STFT and mel (the framing of cmwg_melspec_fwd_varlen with pad_left = n_fft/2 and power_is_one = 1).  Per item
 * b, over the first len_b samples of both signals (len_b = lengths[b], or T when both length pointers are NULL;
 * n_fft/2 < len_b <= T), with S, S^ the STFTs (reflect padding at len_b, len_b / hop + 1 frames, n_fft/2 + 1 bins) and per
 * frame P = |S|^2, m = ln max(mel @ |S|, 1e-5), c = D m:
 *   out[b][0] = mean_f sqrt(mean_k (log10 max(P, 1e-10) - log10 max(P^, 1e-10))^2)          (LSD)
 *   out[b][1] = mean_f mean_j |m_j - m^_j|                                                  (log-mel L1)
 *   out[b][2] = mean_f (10 / ln 10) sqrt(2 sum_{d=1}^{n_cep-1} (c_d - c^_d)^2)                (MCD, c0 excluded)
 * window (n_fft), fbt / fb_lo / fb_hi as for cmwg_melspec_fwd; dct (n_cep, n_mels) row major, the orthonormal DCT-II;
 * 2 <= n_cep <= n_mels.  ref, est: (B, T) at batch stride bstride; out (B, 3) contiguous.  workspace:
 * cmwg_spectral_distance_workspace_bytes(B, T, n_fft, hop) bytes (the per-frame terms).  Summed in a fixed order without
 * atomics: deterministic, and each item equals a call on that item alone bit for bit.  Nothing is allocated.
 * n_fft other than a power of two in [128, 4096]: CMWG_ERR_UNSUPPORTED; bad sizes or lengths: CMWG_ERR_ARG. */
size_t cmwg_spectral_distance_workspace_bytes(int B, int T, int n_fft, int hop);
int cmwg_spectral_distance(const float* ref, const float* est, long long bstride, int B, int T, const int* lengths_host,
                           const int* lengths_dev, const float* window, const float* fbt, const int* fb_lo,
                           const int* fb_hi, const float* dct, int n_fft, int hop, int n_mels, int n_cep, void* workspace,
                           float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * WSRGlow conditioning front end (model/wsrglow.py:37-50, `_get_cond`), one kernel:
 *   c (B, Tc) fp32 low-rate signal, CLIPPED TO [-1, 1] IN PLACE like the reference's c.clip_(-1, 1) (:38);
 *   out (B, 8E + 9 + 9P, Tc/8) fp32 NCL = cat(mu-law code embedding rows (emb: n_codes x E, :39), the 9 magnitudes of
 *   STFT(reflect_pad(c, 4), n_fft 16, hop 8, window, center=False) (:40-47), phase-code embedding rows (aemb: n_phase x P,
 *   index ((angle/pi + 1) * 0.5 * (n_phase - 1)) truncated, :15-17,48-49)).  window: 16 floats.
 *   codes (B, Tc) / phase_codes (B, 9, Tc/8) int32: the table indices used (NULL: not wanted); the backward pass scatters
 *   the cotangent into the two tables with them.
 * ------------------------------------------------------------------------------------------- */
int cmwg_wsrglow_cond(float* c, int B, int Tc, const float* emb, int E, int n_codes, const float* aemb, int P, int n_phase,
                      const float* window, float* out, int* codes, int* phase_codes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Location-variable convolution + gate of MelGlow's WN_LVC (model/melglow.py:52-92, NonCausalLayerLVC.forward, the F.conv1d
 * with groups = batch * frames at :81-82 and the fused_gate at :85):
 *   z[b, oc, t] = sum_{ic, k} w[b, t / span, oc, ic, k] * x[b, ic, t + (k - radix/2) * dilation]   (zero padding), span = T / frames
 *   g[b, c, t]  = tanh(z[b, c, t]) * sigmoid(z[b, Cd + c, t])
 * x (B, Cr, T), w (B, frames, 2Cd, Cr, radix), g (B, Cd, T), all fp32 contiguous.  One CTA per (frame, batch item).
 * Backward: dg (B, Cd, T) -> dx (B, Cr, T), dw (like w), with dz (B, 2Cd, T) as scratch; deterministic.
 * ------------------------------------------------------------------------------------------- */
int cmwg_lvc_gate_forward(const float* x, const float* w, int B, int T, int frames, int Cd, int Cr, int radix, int dilation,
                          float* g, void* stream);
int cmwg_lvc_gate_backward(const float* x, const float* w, const float* dg, int B, int T, int frames, int Cd, int Cr,
                           int radix, int dilation, float* dz, float* dx, float* dw, void* stream);

/* ---------------------------------------------------------------------------------------------
 * WaveFlow glue (model/waveflow.py:154-265).  Images are (B, H, W) fp32 contiguous, H = n_group lines;
 * lst = (B, 2, (H-1)*W) is the 2-D WN's output for input lines 0..H-2 (log_s, then t).
 * ------------------------------------------------------------------------------------------- */
/* With y = cat(x0, xout) in unflipped line order (y[0] = in[0]):
 *   inverse = 0 (:203-206):  y[j] = in[j] * exp(log_s[j-1]) + t[j-1]
 *   inverse = 1 (:253):      y[j] = (in[j] - t[j-1]) / exp(log_s[j-1])
 * for j in [line_begin, line_begin + line_count).  in_flip / out_flip address line H-1-j instead of j: the
 * height flips of :211 (x = cat(xout.flip(2), x0)) and :230 (z = z.flip(2)).  lst may be NULL when only line 0
 * is requested. */
int cmwg_waveflow_affine(const float* in, int in_flip, const float* lst, float* out, int out_flip, int B, int H, int W,
                         int line_begin, int line_count, int inverse, void* stream);
/* One flow of WaveFlow's synthesis direction (:237-259): x[0] = z'[0]; for i = 1..H-1: (log_s, t) = WN2D row
 * i-1 given rows < i (cmwg_wn_forward_lines), x[i] = (z'[i] - t) / exp(log_s), where z' = z read with the height
 * flip when in_flip != 0.  cfg->height = H-1 (the lines the WN sees); z, x (B, H, W); lst (B, 2, (H-1)*W) is left
 * filled with every row's (log_s, t) so the caller can form logdet (:255-258); workspace / state as for
 * cmwg_wn_forward_lines.  The whole row loop is enqueued by this one call (no host round trips). */
int cmwg_waveflow_inverse_flow(const cmwg_wn_config* cfg, const void* packed, const float* z, int in_flip,
                               const void* ycl, int B, int W, void* workspace, void* state, float* lst, float* x,
                               void* stream);
/* Backward of the inverse = 0 transform (autograd of :203-211): dout is the cotangent of the (optionally flipped)
 * output image, dlogdet (B floats, may be NULL) the cotangent of log_s.sum((1,2,3)) (:208).  Writes dx (B, H, W):
 * the direct path only -- the WN backward ACCUMULATES its input gradient into lines 0..H-2 afterwards -- and
 * dlst (B, 2, (H-1)*W). */
int cmwg_waveflow_affine_bwd(const float* x, const float* lst, const float* dout, int out_flip, const float* dlogdet,
                             float* dx, float* dlst, int B, int H, int W, void* stream);

/* Conditioning upsampler (:169-175, 263-265): ReplicationPad1d((0, rpad)) -> DENSE ConvTranspose1d(C, C, K, stride,
 * pad) with weight norm over dim 0 of the (in, out, K) weight (per INPUT channel; g == NULL: v is the plain
 * weight) -> LeakyReLU(slope).  h (B, C, F) -> y (B, C, (F+rpad-1)*stride - 2*pad + K).
 * workspace: cmwg_upsample_dense_workspace(C, K) bytes. */
size_t cmwg_upsample_dense_workspace(int C, int K);
int cmwg_upsample_dense_fwd(const float* h, const float* g, const float* v, const float* bias, int B, int C, int F,
                            int K, int stride, int pad, int rpad, float slope, float* y, void* workspace, void* stream);
/* y = the forward output (its sign selects the LeakyReLU slope), dy its cotangent (contiguous).
 * dg (C) / dbias (C) may be NULL; dv (C, C, K). */
int cmwg_upsample_dense_bwd(const float* h, const float* g, const float* v, const float* y, const float* dy, int B,
                            int C, int F, int K, int stride, int pad, int rpad, float slope, float* dg, float* dv,
                            float* dbias, void* workspace, void* stream);

/* Conditioning of NVIDIA's WaveGlow (NVIDIA/waveglow glow.py): ConvTranspose1d(C, C, taps * hop, stride = hop) with
 * bias, no weight norm, then unfolded by n_group, computed as one tcgen05 GEMM that writes the 16-bit WN conditioning
 * slab (the layout cmwg_cond_pack writes, C * n_group channels) directly:
 *   slab[b][t][c] = up[b, c / n_group, n_group t + c % n_group],
 *   up[b, o, hop q + r] = bias[o] + sum_{j < taps} sum_i w[i, o, r + hop j] * mel[b, i, q - j]   (mel = 0 outside [0, F)).
 * w is the (C, C, taps * hop) fp32 weight; `packed` (cmwg_nvidia_upsample_packed_bytes) is its GEMM operand, written by
 * cmwg_nvidia_upsample_pack once per weight version.  mel (B, C, F) fp32 with unit frame stride; T squeezed steps per
 * item (any T >= 0: frames past F contribute nothing, rows past T are not written); precision CMWG_PREC_FP16 / _BF16.
 * C * n_group must be a multiple of 64 (else CMWG_ERR_UNSUPPORTED) and n_group must divide hop.
 * workspace: cmwg_nvidia_upsample_workspace_bytes(B, T, C, hop, taps, n_group) bytes. */
size_t cmwg_nvidia_upsample_packed_bytes(int C, int hop, int taps);
int cmwg_nvidia_upsample_pack(const float* w, int C, int hop, int taps, int n_group, int precision, void* packed,
                              void* stream);
size_t cmwg_nvidia_upsample_workspace_bytes(int B, int T, int C, int hop, int taps, int n_group);
int cmwg_nvidia_upsample_slab(const void* packed, const float* bias, const float* mel, long long mel_bstride,
                              long long mel_cstride, int B, int C, int F, int hop, int taps, int n_group, int T,
                              int precision, void* slab, void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Model glue (model/waveglow.py:153,179; model/loss.py:10-15)
 * ------------------------------------------------------------------------------------------- */
/* squeeze: x (B, T) -> out (B, n_group, T/n_group);  unsqueeze is the inverse permutation */
int cmwg_squeeze(const float* x, float* out, int B, int T, int n_group, int inverse, void* stream);

/* loss = mean_b(0.5*sum_t z^2/sigma^2 - logdet_b) / (mean ? T : 1); also dz = dloss/dz (may be NULL).
 * Deterministic. workspace >= (B + 1) floats. */
int cmwg_nll_loss(const float* z, const float* logdet, int B, int T, float sigma, int elementwise_mean,
                  float* loss, float* dz, void* workspace, void* stream);

/* per-batch sum over (channel, time) of an NCL tensor: the log_s.sum((1,2)) of model/waveglow.py:175 */
int cmwg_sum_per_batch(const float* a, long long a_bstride, int B, int N, float* out, int accumulate, float scale,
                       void* stream);

/* One flow's log-det bookkeeping, `logdet = logdet + log_det_W + log_s.sum((1, 2))` (model/waveglow.py:175,199), in one
 * launch: out[b] = prev[b] + *log_det_w + sum over (channel, time) of a[b];  prev (B floats) and log_det_w (one device
 * float) may be NULL (= 0); out may alias prev.  Deterministic. */
int cmwg_logdet_accumulate(const float* a, long long a_bstride, int B, int N, const float* prev, const float* log_det_w,
                           float* out, void* stream);

/* Per-item lengths: out[b] = prev[b] + *log_det_w * len_b + sum over channels c < C and columns t < len_b of a[b, c, t],
 * len_b = lengths_dev[b] (device ints).  a: (C, T) rows per item at batch stride a_bstride.  log_det_w here is the log-det
 * of ONE column (the 1x1 conv's log|det W|), scaled by each item's own length.  The padded columns are not read. */
int cmwg_logdet_accumulate_varlen(const float* a, long long a_bstride, int B, int C, int T, const int* lengths_dev,
                                  const float* prev, const float* log_det_w, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Per-kernel-class device timing (CUDA events recorded on the launching stream around each GEMM
 * launch).  Off by default; bench.py turns it on for its roofline leg.
 * ------------------------------------------------------------------------------------------- */
#define CMWG_KCLASS_GATE 0    /* dilated conv + conditioning GEMM with fused gate epilogue */
#define CMWG_KCLASS_RESSKIP 1 /* W_o GEMM with residual/skip epilogue                      */
#define CMWG_KCLASS_DGATE 2   /* W_o^T GEMM with gate-backward epilogue                    */
#define CMWG_KCLASS_DX 3      /* transposed dilated conv GEMM                              */
#define CMWG_KCLASS_DCOND 4   /* conditioning gradient GEMM                                */
#define CMWG_KCLASS_WGRAD 5   /* weight-gradient GEMMs                                     */
#define CMWG_KCLASS_FWDFUSED 6 /* whole-WN forward task kernel (all gate, residual and skip GEMM tiles of one WN) */
#define CMWG_KCLASS_BWDFUSED 7 /* dgate + dx GEMM tiles of all layers of one WN backward (task kernel)             */
#define CMWG_KCLASS_COUNT 8
/* on != 0: start recording (drops earlier records); on == 0: stop */
int cmwg_profile_enable(int on);
/* waits for the recorded events; fills ms[CMWG_KCLASS_COUNT], launches[CMWG_KCLASS_COUNT]; clears records */
int cmwg_profile_collect(double* ms, long long* launches);

/* ---------------------------------------------------------------------------------------------
 * Self-test hooks used by tests/: a plain GEMM through each engine.
 *   D[m][n] = sum_k A[m][k] * Bm[n][k]      (A: M x K, Bm: N x K, both row major, 16-bit operands)
 * ------------------------------------------------------------------------------------------- */
int cmwg_selftest_tc_gemm(const void* a, const void* b, float* d, int M, int N, int K, int is_fp16, int variant,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CMWG_B200_H */
