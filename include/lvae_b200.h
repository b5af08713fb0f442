/* lvae_b200.h -- C ABI of liblvae_b200.so (hand-written sm_100a kernels for the Ladder VAE hot path).
 *
 * The reference (addtt/ladder-vae-pytorch) has no FFI: its "operators" are PyTorch nn.Modules
 * whose kernels are ATen/cuDNN library calls.  Each entry point below names the reference code
 * (file:line under the reference tree) whose GPU work it replaces; INTEGRATION.md shows the
 * ctypes stub a reference maintainer would add at that spot.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless noted; the caller (PyTorch) owns all memory;
 *   - activations are NHWC: (B, H, W, C) contiguous; `dtype` 0 = float32, 1 = bfloat16;
 *     images handed in by the user (`x` of the likelihoods, pad source) are NCHW float32;
 *   - `stream` is the cudaStream_t to launch on; kernels never allocate or synchronise, so
 *     every call can be captured into a CUDA graph;
 *   - return 0 on success, non-zero on error; lvae_last_error() gives the message
 *     (bad arguments are rejected before any launch).
 */
#ifndef LVAE_B200_H
#define LVAE_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef void* lvae_stream_t; /* cudaStream_t */

/* ---- plumbing ---- */
const char* lvae_last_error(void);
int lvae_abi_version(void);
unsigned long long lvae_launch_count(void); /* kernels launched by this library so far */
void lvae_reset_launch_count(void);
int lvae_device_check(void); /* 0 iff the current device is sm_10x */
/* programmatic dependent launch for every kernel of the library (default on): a kernel's prologue overlaps
 * the tail of its predecessor; all kernels call griddepcontrol.wait before touching upstream results */
void lvae_set_pdl(int enabled);
int lvae_get_pdl(void);

/* ---- convolutions: nn.Conv2d / nn.ConvTranspose2d forward, dgrad, wgrad ----
 * replaces cuDNN behind lib/nn.py:83-87 (3x3 residual convs), lib/nn.py:118 (1x1 gate conv),
 * lib/stochastic.py:25-27 (conv_in_p / conv_in_q / conv_out), models/lvae_layers.py:263-276
 * (strided / transposed resampling), models/lvae_layers.py:350,359 (1x1 merge over cat(x, x2)),
 * models/lvae.py:75 (5x5 stem), lib/likelihoods.py:55,199 (heads).
 *   y[b,oy,ox,n] = ( sum_{ky,kx,c} in[b,iy,ix,c] * wp[(ky*kw+kx)*(C1+C2)+c][n] + bias[n] ) * out_scale[b,n] + res
 *   mode 0: iy = oy*stride - pad + ky          (Conv2d forward, ConvTranspose2d dgrad)
 *   mode 1: iy = (oy + pad - ky) / stride      (Conv2d dgrad, ConvTranspose2d forward)
 * `in` is the channel concatenation of x (C1) and x2 (C2, may be NULL/0); in_scale (B,C1+C2) and
 * out_scale (B,N) are per-sample channel scales (Dropout2d, lib/nn.py:62,76,89) or NULL. */
int lvae_conv2d_gather(const void* x, const void* x2, const void* wp, const float* bias, const float* in_scale,
                       const float* out_scale, const void* res, void* y, int B, int Hi, int Wi, int C1, int C2,
                       int Ho, int Wo, int N, int ldw, int kh, int kw, int stride, int pad, int mode, int dtype,
                       lvae_stream_t stream);
/* dw[o][i][ky][kx] += sum dz[b,oy,ox,o] * u[b,oy*stride-pad+ky,ox*stride-pad+kx,i]; dbias[o] += sum dz.
 * dw is the torch parameter layout (O,I,kh,kw) fp32; for ConvTranspose2d pass (u=dy, dz=x). */
int lvae_conv2d_wgrad(const void* u, const void* u2, const void* dz, const float* in_scale, const float* out_scale,
                      float* dw, float* dbias, int B, int Hi, int Wi, int C1, int C2, int Ho, int Wo, int O, int kh,
                      int kw, int stride, int pad, int dtype, lvae_stream_t stream);
/* bf16 tensor-core path (TMA -> tcgen05.mma -> TMEM) for the stride-1 "same" convs with a multiple of 64 (at most
 * 256) channels per input tensor, two inputs of equal width: x, x2 (B,H,W,Cin) bf16; wp = lvae_pack_weights mode 2 (forward) / 3 (dgrad, flip = 1);
 * y (B,H,W,N) bf16 or fp32 (out_f32); y2 != NULL splits the N output columns at nsplit (dgrad of the
 * two-input merge conv).  H, W powers of two, W <= 128, N <= 256, ksize 1 or 3. */
int lvae_conv2d_tc(const void* x, const void* x2, const void* wp, const float* bias, const float* out_scale,
                   const void* res, void* y, void* y2, int nsplit, int B, int H, int W, int Cin, int N, int ksize,
                   int flip, int out_f32, lvae_stream_t stream);
/* bf16 tensor-core weight gradient for the same convolutions (reduction over pixels, MN-major operands,
 * two filter taps per M = 128 MMA, bias gradient from an all-ones operand block): x, x2 (B,H,W,64) bf16,
 * dy (B,H,W,N) bf16 with N in {64,128} (already multiplied by the Dropout2d mask); dw (N,I,k,k) fp32 +=,
 * dbias [N] += or NULL; ws = lvae_wgrad_tc_workspace(...) floats of scratch (one packed gradient, see below).
 * I_real: input channels of dw (0 = 64 per input, at most that); N_real: rows of dw (0 = N, at most N);
 * dy carries dyC channels (0 = N), of which channels [dy_c0, dy_c0 + N) are used (dy_c0 a multiple of 64). */
int lvae_conv2d_wgrad_tc(const void* x, const void* x2, const void* dy, float* dw, float* dbias, float* ws, int B,
                         int H, int W, int N, int ksize, int I_real, int N_real, int dyC, int dy_c0, lvae_stream_t stream);
long long lvae_wgrad_tc_workspace(int B, int H, int W, int N, int ksize, int two_inputs);
/* The same over a 64-channel window of wider inputs: x, x2 (B,H,W,xC) bf16 (xC a multiple of 64 up to 256; 0 = 64), of
 * which channels [x_c0, x_c0 + 64) are read (x_c0 a multiple of 64).  dw (N_real, I_real, k, k) with I_real = xC per input
 * (0) or fewer; this launch adds input channels s * xC + x_c0 + [0, 64) of input s.  Every launch also adds the bias
 * gradient, so a caller splitting one conv over several X windows passes dbias to one of them per dY window. */
int lvae_conv2d_wgrad_tc_ex(const void* x, const void* x2, const void* dy, float* dw, float* dbias, float* ws, int B,
                            int H, int W, int N, int ksize, int I_real, int N_real, int dyC, int dy_c0, int xC, int x_c0,
                            lvae_stream_t stream);
/* The same gradient in two steps, for callers that batch the re-layout (engine.py: one unpack launch per training step
 * instead of one per convolution; replaces the per-parameter `.grad` accumulation of loss.backward(),
 * experiment_manager.py:78-80 / boilr's training loop).  lvae_conv2d_wgrad_tc_acc ADDS the gradient into the packed
 * buffer gp (lvae_wgrad_tc_packed_size floats: [pair][128 rows = two (tap, input-block) row blocks of 64 ci][N]) with TMA
 * reduce-stores from every CTA; lvae_wgrad_unpack_batched adds n packed buffers into their (O,I,kh,kw) gradients
 * (descriptors of lvae_wgrad_unpack_desc_size bytes each, built on the host by lvae_wgrad_unpack_desc and copied to
 * device memory; clear bit 0: also zero gp for the next step; bit 1: overwrite dw / dbias instead of adding, for callers
 * that know nothing else contributed to them). */
long long lvae_wgrad_tc_packed_size(int N, int ksize, int two_inputs);
int lvae_conv2d_wgrad_tc_acc(const void* x, const void* x2, const void* dy, float* gp, int B, int H, int W, int N,
                             int ksize, int dyC, int dy_c0, lvae_stream_t stream);
/* Weight gradient of the stride-2 3x3 64 -> 64 resampling convolutions (models/lvae_layers.py:261-276) on the same kernel:
 * the tap-shifted operand xs (B,2Hg,2Wg,64) bf16 is read through an element-strided tensor map, c (B,Hg,Wg,64) bf16 lives
 * on the small grid.  Conv2d(stride 2, pad 1): xs = input, c = dY (masked), dw (Cout,Cin,3,3), dbias = column sums of dY.
 * ConvTranspose2d(stride 2, pad 1, output_padding 1): xs = dY (masked), c = input, dw (Cin,Cout,3,3), dbias must be NULL
 * (its bias gradient sums the LARGE grid: lvae_colsum).  _acc adds into a packed buffer of
 * lvae_wgrad_tc_packed_size(64, 3, 0) floats (unpack descriptor: N = 64, ksize = 3, one input); the one-call form
 * takes such a buffer as scratch (ws) and adds into dw / dbias. */
int lvae_conv2d_wgrad_tc_s2_acc(const void* xs, const void* c, float* gp, int B, int Hg, int Wg, lvae_stream_t stream);
int lvae_conv2d_wgrad_tc_s2(const void* xs, const void* c, float* dw, float* dbias, float* ws, int B, int Hg, int Wg,
                            lvae_stream_t stream);
int lvae_wgrad_unpack_desc_size(void);
int lvae_wgrad_unpack_desc(void* desc_host, const float* gp, float* dw, float* dbias, int N, int ksize, int two_inputs,
                           int I_real, int N_real, int clear);
int lvae_wgrad_unpack_batched(const void* desc_dev, int n, int max_n_real, lvae_stream_t stream);
/* Same with per-channel reductions fused into the epilogue (bf16 output, N == 64, no residual / split):
 *   stats_acc  [2*64] += sum / sum-of-squares of the output as stored (the next BatchNorm's statistics),
 *   bnb_*      BatchNorm-backward sums over this data-gradient output dy: bnb_acc [2*64] += sum(g), sum(g*xhat) with
 *              xhat = (bnb_x - mean)*rstd, g = dy * act'(xhat*gamma + beta); bnb_save = [mean | rstd]. */
typedef struct {
  double* stats_acc;
  const void* bnb_x;
  const float* bnb_save;
  const float* bnb_gamma;
  const float* bnb_beta;
  double* bnb_acc;
  int bnb_act;
  /* gated residual (lib/nn.py:121-126 GateLayer2d + the residual add of :99) in the epilogue of its 1x1 conv (N = 128):
   * gate_out (M,64) bf16 = act(h[:, :64]) * sigmoid(h[:, 64:]) + gate_x; h itself still goes to y (saved for backward);
   * stats_acc, when set, then accumulates the statistics of gate_out (the next block's first BatchNorm) */
  const void* gate_x;
  void* gate_out;
  int gate_act;
  int gate_skip_h;      /* eval mode: do not store h (y may then be NULL): nothing runs backward */
  /* eval-mode BatchNorm2d + activation of the CONSUMER (lib/nn.py:84-85 in eval mode) folded into this conv (N == 64, no other
   * fusion): y = act((conv + bias) * s + beta - mean * s), s = gamma * rsqrt(var + eps), from the running statistics.  For
   * no_grad callers only (the IW evaluator): the pre-BatchNorm tensor is never materialised.  fold_gamma NULL = off. */
  const float* fold_gamma;
  const float* fold_beta;
  const float* fold_mean;
  const float* fold_var;
  float fold_eps;
  int fold_act;
  /* with fold_*: the eval-mode BatchNorm2d + activation in FRONT of the conv (lib/nn.py:78-81 in eval mode) applied to the
   * operand tile in shared memory on its way to the tensor cores (same activation as fold_act): x may then be the raw block
   * input.  Single 64-channel input, 3x3, W % 8 == 0, H % 16 == 0.  pre_gamma NULL = off. */
  const float* pre_gamma;
  const float* pre_beta;
  const float* pre_mean;
  const float* pre_var;
  float pre_eps;
} LvaeConvFuse;
int lvae_conv2d_tc_ex(const void* x, const void* x2, const void* wp, const float* bias, const float* out_scale,
                      const void* res, void* y, void* y2, int nsplit, int B, int H, int W, int Cin, int N, int ksize,
                      int flip, int out_f32, const LvaeConvFuse* fuse, lvae_stream_t stream);
/* How lvae_conv2d_tc[_ex] holds the weights of a shape, decided by the code the launch uses (pure host, no CUDA call):
 * 0 = rejected, 1 = resident (all k-blocks stay in shared memory; the fused epilogues and halo tiles need this),
 * 2 = streamed (each pipeline stage carries its k-block's weight tile next to the activation box; plain epilogues). */
int lvae_conv2d_tc_plan(int Cin, int N, int ksize, int two_inputs, int H, int W, int out_f32);
/* The tail of a gated residual block as one launch (gated blocks on the bf16 path whose shapes it serves; the others run
 * conv2 and the gate conv as two launches):
 *   c2 = (conv3x3(a2) + bias2) * scale2      second 3x3 convolution of lib/nn.py:83-87 with its Dropout2d mask (B,64) or NULL
 *   h  = conv1x1(c2) + bias_g  (128 ch)      GateLayer2d's convolution, lib/nn.py:118
 *   out = act(h[:, :64]) * sigmoid(h[:, 64:]) + x_res          lib/nn.py:121-126 and the residual add :99
 * The 1x1 GEMM reads the bf16 tile that the 3x3 epilogue stages in shared memory for its TMA store (csrc/conv_gate_tcgen05.cu).
 * a2, x_res, c2, out: (B,H,W,64) bf16; h: (B,H,W,128) bf16; c2 and h both NULL in eval mode.  w2p: nine packed [64][64]
 * blocks, wgp: one packed [128][64] block (lvae_pack_weights mode 2).  stats_acc: 8-way striped (8,2,64) doubles, += the
 * per-channel sum / sum of squares of out, or NULL.  H, W powers of two, W <= 128. */
int lvae_conv_gate_tc(const void* a2, const void* w2p, const float* bias2, const float* scale2, const void* wgp,
                      const float* bias_g, const void* x_res, void* c2, void* h, void* out, double* stats_acc, int B, int H,
                      int W, int gate_act, lvae_stream_t stream);
/* Stride-2 3x3 convolutions 64 -> 64 on the same tcgen05 kernel (the down / up-sampling pre_convs of
 * models/lvae_layers.py:261-276).  kind 0 "gather": y (B,Hg,Wg,N) from x (B,2Hg,2Wg,64) = Conv2d(stride 2, pad 1) forward
 * and ConvTranspose2d(stride 2, pad 1, output_padding 1) input gradient (TMA traverses x with element stride 2).  kind 1
 * "transposed": y (B,2Hg,2Wg,N) from x (B,Hg,Wg,64) = ConvTranspose2d forward and Conv2d(stride 2) input gradient, as four
 * launches, one per output parity class (1 + 2 + 2 + 4 filter taps), each storing through a tensor map that steps two
 * output pixels.  wp: nine packed [64][64] blocks, block t = tap (t/3, t%3), rows = output channel (lvae_pack_weights
 * mode 2 / 3).  bias, out_scale (B,N) optional.  Hg, Wg powers of two, Wg <= 64. */
int lvae_conv2d_tc_s2(const void* x, const void* wp, const float* bias, const float* out_scale, void* y, int B, int Hg,
                      int Wg, int N, int kind, lvae_stream_t stream);
/* Narrow-output 3x3 "same" convolution, 64 bf16 channels -> N <= 4 (the Bernoulli head's parameter_net,
 * lib/likelihoods.py:61: 64 -> 1): bandwidth-bound, 8 lanes per pixel.  w: torch (N,64,3,3) fp32; y (B,H,W,N) fp32 / bf16. */
int lvae_conv3x3_narrow(const void* x, const float* w, const float* bias, void* y, int B, int H, int W, int N, int out_f32,
                        lvae_stream_t stream);
/* The same with the input given as a WINDOW of a larger (B,Hs,Ws,64) bf16 tensor (N == 1 only): x points at the window's first
 * pixel, row_pitch / img_pitch are the elements between consecutive rows / images (0 = dense).  The centred crop in front of the
 * likelihood (models/lvae.py:143, boilr crop_img_tensor) then needs no pass of its own. */
int lvae_conv3x3_narrow_ex(const void* x, const float* w, const float* bias, void* y, int B, int H, int W, int N, int out_f32,
                           int row_pitch, long long img_pitch, lvae_stream_t stream);
/* profiling aid: CTA 0 of subsequent lvae_conv2d_tc launches records clock64 stamps per tile into dev_buf (NULL = off) */
void lvae_conv2d_tc_debug(long long* dev_buf);
/* the same for lvae_conv_gate_tc (16 stamps per tile: epilogue phases in slots 0..6, MMA warp in 8..10) */
void lvae_conv_gate_tc_debug(long long* dev_buf);
/* y = x * scale[b,c] (Dropout2d mask on a gradient tensor ahead of the TMA-fed dgrad) */
int lvae_channel_scale(const void* x, const float* scale, void* y, int B, int HW, int C, int dtype,
                       lvae_stream_t stream);
/* Re-layout torch (O,I,kh,kw) weights into GEMM rows; descs_dev = device array of n LvaePackDesc
 * {const float* src; void* dst; int O, I, taps, mode, ld, dtype} (see csrc/conv_generic.cu). */
int lvae_pack_weights(const void* descs_dev, int n, lvae_stream_t stream);
int lvae_pack_desc_size(void);
/* out[c] += sum_{b,hw} dy[b,hw,c] * scale[b,c]  (ConvTranspose2d bias gradient) */
int lvae_colsum(const void* dy, const float* scale, float* out, int B, int HW, int C, int dtype, lvae_stream_t stream);

/* ---- BatchNorm2d (+ nonlinearity) : lib/nn.py:60,67,81 + models/lvae.py:64-69 ----
 * act: 0 none, 1 relu, 2 leaky_relu(0.01), 3 elu, 4 selu.  acc = 8 stripes x 2*C doubles ([stripe][sum|sumsq][C];
 * producers add into stripe blockIdx % 8 to cut atomic contention, consumers sum the stripes), zero on entry,
 * left zero on exit by the unfused calls.  Train mode: stats -> finalize (also updates running_mean/var and
 * num_batches_tracked on the device) -> bn_act_fwd.  Eval mode: eval_prepare -> bn_act_fwd. */
int lvae_bn_stats(const void* x, double* acc, long long P, int C, int dtype, lvae_stream_t stream);
int lvae_bn_finalize(double* acc, float* save_mean, float* save_rstd, float* running_mean, float* running_var,
                     long long* num_batches_tracked, long long P, int C, float momentum, float eps,
                     lvae_stream_t stream);
int lvae_bn_eval_prepare(const float* running_mean, const float* running_var, float* save_mean, float* save_rstd,
                         int C, float eps, lvae_stream_t stream);
/* y = act(((x-mean)*rstd)*gamma+beta); mean == NULL -> plain activation */
int lvae_bn_act_fwd(const void* x, void* y, const float* mean, const float* rstd, const float* gamma,
                    const float* beta, long long P, int C, int act, int dtype_in, int dtype_out,
                    lvae_stream_t stream);
/* dx, dgamma += , dbeta += ; training = 1 uses batch-statistics backward */
int lvae_bn_act_bwd(const void* dy, const void* x, void* dx, const float* mean, const float* rstd,
                    const float* gamma, const float* beta, double* acc, float* dgamma, float* dbeta, long long P,
                    int C, int act, int training, int dtype, lvae_stream_t stream);

/* Fused variants for the whole-residual-block schedule: forward derives mean / rstd in-kernel from the
 * statistics accumulator (training) or the running statistics (eval), writes save = [mean | rstd] and
 * updates the running statistics; backward = reduce + apply, the apply pass also emitting dgamma / dbeta,
 * an optional Dropout2d mask on dx (post_scale (B,C)) and an optional residual add.  Accumulators are
 * not cleared (the caller zeroes its BatchNorm scratch arena once per forward). */
int lvae_bn_act_fwd2(const void* x, void* y, const double* acc, const float* gamma, const float* beta, float* save,
                     float* running_mean, float* running_var, long long* num_batches_tracked, long long P, int C,
                     int act, int training, float momentum, float eps, int dtype_in, int dtype_out,
                     lvae_stream_t stream);
int lvae_bn_act_bwd2(const void* dy, const void* x, void* dx, const float* save, const float* gamma,
                     const float* beta, double* acc, float* dgamma, float* dbeta, const float* post_scale,
                     const void* add, long long P, int hw, int C, int act, int training, int dtype,
                     int skip_reduce, lvae_stream_t stream);
/* The same apply pass (statistics sums already in acc) that also runs the gate backward (lib/nn.py:121-126) of the residual block
 * that PRODUCED x -- the next block of the backward pass, whose output gradient is exactly this dx: gate_dh (P,2C) =
 * gate'(dx, gate_h).  bf16 only.  One launch and one re-read of dx less per pair of adjacent gated blocks. */
int lvae_bn_act_bwd2_gate(const void* dy, const void* x, void* dx, const float* save, const float* gamma, const float* beta,
                          double* acc, float* dgamma, float* dbeta, const float* post_scale, const void* add,
                          const void* gate_h, void* gate_dh, long long P, int hw, int C, int act, int gate_act, int training,
                          lvae_stream_t stream);

/* ---- GateLayer2d product + residual: lib/nn.py:121-126 and :99 ----
 * h (P,2C): out = act(h[:, :C]) * sigmoid(h[:, C:]) + res */
int lvae_gate_fwd(const void* h, const void* res, void* out, long long P, int C, int act, int dtype,
                  lvae_stream_t stream);
/* same, also accumulating per-channel sum / sum-of-squares of `out` into acc (2C doubles) */
int lvae_gate_fwd_stats(const void* h, const void* res, void* out, double* acc, long long P, int C, int act,
                        int dtype, lvae_stream_t stream);
int lvae_gate_bwd(const void* dout, const void* h, void* dh, long long P, int C, int act, int dtype,
                  lvae_stream_t stream);

/* ---- boilr helpers used inside the model: Interpolate(scale=2) (models/lvae.py:144),
 *      pad_img_tensor / crop_img_tensor (models/lvae.py:176,185,324,357) ---- */
int lvae_upsample2x_fwd(const void* x, void* y, int B, int H, int W, int C, int dtype, lvae_stream_t stream);
int lvae_upsample2x_bwd(const void* dy, void* dx, int B, int H, int W, int C, int dtype, lvae_stream_t stream);
int lvae_copy_window(const void* src, void* dst, int B, int C, int Hs, int Ws, int Hd, int Wd, int sy0, int sx0,
                     int dy0, int dx0, int h, int w, int src_nchw, int dst_nchw, int src_dtype, int dst_dtype,
                     lvae_stream_t stream);

/* ---- randomness: device-resident Philox state {uint64 seed, uint64 offset} ---- */
int lvae_dropout_masks(float* masks, long long n, float p, const void* rng_state, unsigned long long stream_id,
                       lvae_stream_t stream); /* nn.Dropout2d masks for every site of a step, lib/nn.py:62,76,89 */
int lvae_rng_advance(void* rng_state, unsigned long long inc, lvae_stream_t stream);
int lvae_sum_batch(const float* x, float* out, int B, long long n, int accumulate, lvae_stream_t stream);

/* ---- NormalStochasticBlock2d core: lib/stochastic.py:45-96 and kl_normal_mc :209-226 ----
 * q, p: (B,hw,2Z) fp32 rows [mu | logvar]; p_broadcast = 1 when p has batch 1 (learned top prior,
 * models/lvae_layers.py:131-136).  z = mu_q + exp(lv_q/2)*eps with eps given, or Philox when eps == NULL;
 * forced != NULL -> z = forced; use_mode -> z = mu.  q == NULL -> sample from p (generation).
 * Outputs: z (B,hw,Z) [+ optional bf16 copy with row pitch z_bf16_pitch >= Z, zero padded], kl_sample (B) (MC log q - log p, or analytic),
 * kl_spatial (B,hw) (always analytic), logp (B), logq (B). */
int lvae_stoch_fwd(const float* q, const float* p, int p_broadcast, const float* eps, const float* forced,
                   const void* rng_state, unsigned long long stream_id, float* z, void* z_bf16, int z_bf16_pitch, float* kl_sample,
                   float* kl_spatial, float* logp, float* logq, int B, int hw, int Z, int use_mode, int analytical,
                   void* ws, lvae_stream_t stream);
/* ws: NULL (one CTA per sample) or a device workspace of lvae_stoch_ws_bytes(B) bytes, zeroed once by the caller and used
 * with this one batch size, that lets the kernel split a sample over several CTAs (their per-sample sums are combined in
 * a fixed order: deterministic). */
long long lvae_stoch_ws_bytes(int B);
/* z_kind: 1 reparameterised sample, 2 mode, 0 forced latent.  dq, dp: (B,hw,2Z). */
int lvae_stoch_bwd(const float* q, const float* p, int p_broadcast, const float* z, const float* g_z,
                   const float* g_kl, const float* g_logp, const float* g_logq, const float* g_kls, float* dq,
                   float* dp, int B, int hw, int Z, int analytical, int z_kind, lvae_stream_t stream);
/* The same with optional bf16 copies of dq / dp ((B,hw,2Z), round to nearest even; NULL = none): the operands of the tensor-core
 * data / weight gradients of conv_in_q / conv_in_p (lib/stochastic.py:25-26), which then need no conversion pass. */
int lvae_stoch_bwd_ex(const float* q, const float* p, int p_broadcast, const float* z, const float* g_z,
                      const float* g_kl, const float* g_logp, const float* g_logq, const float* g_kls, float* dq,
                      float* dp, void* dq_bf16, void* dp_bf16, int B, int hw, int Z, int analytical, int z_kind,
                      lvae_stream_t stream);
/* Free bits + KL bookkeeping of LadderVAE.forward (models/lvae.py:192-198; boilr free_bits_kl) and the log p(z) total of
 * topdown_pass (:301-302) in one launch over the (L,B) matrices whose rows the L stochastic kernels wrote:
 * kl_sep (B), scalars[3] = {kl, kl_loss, logp}, kl_avg_layerwise (L), coef (L,B) = d kl_loss / d kl (kept for the backward). */
int lvae_kl_bookkeeping(const float* kl_rows, const float* logp_rows, int L, int B, float free_bits, float* kl_sep,
                        float* scalars, float* kl_avg_layerwise, float* coef, lvae_stream_t stream);
/* g_scalars: device float[3], upstream gradients of {kl, kl_loss, logp}; g_kl_sep (B) / g_kl_avg (L) / g_logp_rows optional */
int lvae_kl_bookkeeping_bwd(const float* coef, const float* g_scalars, const float* g_kl_sep, const float* g_kl_avg, int L,
                            int B, float* g_kl_rows, float* g_logp_rows, lvae_stream_t stream);

/* ---- likelihoods: lib/likelihoods.py ----
 * Bernoulli (:51-78, log_bernoulli :385-388): logits (B,hw,C) NHWC, x (B,C,hw) NCHW. */
int lvae_bernoulli_fwd(const float* logits, const float* x, float* prob, float* ll, int B, int hw, int C,
                       lvae_stream_t stream);
int lvae_bernoulli_bwd(const float* prob, const float* x, const float* g_ll, const float* g_prob, float* dlogits,
                       int B, int hw, int C, lvae_stream_t stream);
int lvae_bernoulli_sample(const float* prob, float* out_nchw, int B, int hw, int C, const void* rng_state,
                          unsigned long long stream_id, lvae_stream_t stream);
/* 10-component discretized mixture of logistics (:183-230, discretized_mix_logistic_loss :291-382):
 * l (B,hw,100) NHWC, x (B,3,hw) NCHW in [0,1]; ll (B) must be zero on entry (fwd accumulates). */
int lvae_dmol_fwd(const float* l, const float* x, float* ll, int B, int hw, lvae_stream_t stream);
/* dl: fp32 (B,hw,100); or dl_bf16_128 != NULL: bf16 (B,hw,128) zero-padded, ready for the tcgen05 dgrad / wgrad of the head */
int lvae_dmol_bwd(const float* l, const float* x, const float* g_ll, float* dl, void* dl_bf16_128, int B, int hw,
                  lvae_stream_t stream);
/* sample_from_discretized_mix_logistic (lib/stochastic.py:141-206) + rescale/clamp (likelihoods.py:221-225) */
int lvae_dmol_sample(const float* l, float* out_nchw, int B, int hw, const void* rng_state,
                     unsigned long long stream_id, lvae_stream_t stream);

/* ---- step glue: experiment/experiment_manager.py:78-80 (Adamax), :346-350 (L2 norm) ---- */
/* hyper_dev: NULL, or a device float[2] = {lr, weight_decay} that overrides the by-value arguments (a captured CUDA graph
 * then follows learning-rate schedules without a recapture). */
int lvae_adamax_step(float* p, const float* g, float* exp_avg, float* exp_inf, long long n, float lr, float beta1,
                     float beta2, float eps, float weight_decay, long long* step_count_dev, float grad_scale,
                     const float* hyper_dev, lvae_stream_t stream);
int lvae_l2_norm(const float* p, long long n, double* acc, float* out, lvae_stream_t stream);
/* lvae_adamax_step followed by lvae_l2_norm of the updated parameters, in one pass over the arena (l2_acc: device double scratch,
 * zero on entry, cleared on exit; l2_out[0] = sqrt(sum p^2)). */
int lvae_adamax_step_l2(float* p, const float* g, float* exp_avg, float* exp_inf, long long n, float lr, float beta1,
                        float beta2, float eps, float weight_decay, long long* step_count_dev, float grad_scale,
                        const float* hyper_dev, double* l2_acc, float* l2_out, lvae_stream_t stream);

/* ---- importance-weighted bound (boilr test_procedure, call site evaluate.py:30) ----
 * state (B,2) = running (max, sum exp) of elbo = ll - kl over samples; combine merges R ranks' states. */
int lvae_iw_lse_update(const float* ll, const float* kl, float* state, int B, int first, lvae_stream_t stream);
int lvae_iw_lse_combine(const float* states, float* out, int R, int B, int K_total, lvae_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LVAE_B200_H */
