/* seg2eye_b200 -- C ABI of the B200-native (sm_100a) SPADE+Style G/D training-step kernels.
 *
 * The reference (mcbuehler/Seg2Eye) has no FFI of its own: its hot path is a chain of stock
 * torch.nn calls.  Every entry point below therefore names the reference call site(s) whose
 * arithmetic it replaces (paths relative to the reference checkout).  The Python host in
 * seg2eye_b200/ binds these symbols with ctypes (see INTEGRATION.md) and mirrors the
 * reference's models.networks / Pix2PixModel / Pix2PixTrainer interface on top.
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless stated otherwise; nothing is allocated inside.
 *   - Activations are bf16, NHWC ("pixels x channels"); statistics, losses, master weights,
 *     gradients of weights and optimizer state are fp32 (BASELINE.md section 5).
 *   - `stream` is a cudaStream_t passed as void*.  Calls are asynchronous and re-entrant per stream.
 *   - Return value: 0 = OK, negative = error (s2e_last_error() gives the message).
 */
#ifndef SEG2EYE_B200_H_
#define SEG2EYE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define S2E_OK 0
#define S2E_ERR_ARG (-1)
#define S2E_ERR_CUDA (-2)
#define S2E_ERR_UNSUPPORTED (-3)

#define S2E_ACT_NONE 0
#define S2E_ACT_LRELU 1 /* leaky_relu(., 0.2) */
#define S2E_ACT_RELU 2

#define S2E_IMPL_TC 0   /* tcgen05 + TMEM + TMA implicit GEMM (product path) */
#define S2E_IMPL_SIMT 1 /* CUDA-core kernel: tiny / MMA-unfriendly layers and on-device cross-check */

#define S2E_MAX_TAPS 16

const char* s2e_last_error(void);
int s2e_abi_version(void);
/* debug knobs (bring-up only): key 0 = swap LBO/SBO in MN-major UMMA descriptors, key 1 = force SIMT,
 * key 2 = keep thin-channel layers on the generic SIMT kernel, key 3 = forward epilogue timing experiments (bit 0: skip
 * the TMA store), key 5 = 1: weight gradients with an N side < 256 go back to the one-tap-per-CTA kernel (default: several
 * taps per CTA; 2: these issue one MMA per tap even where the taps could share one), key 6: bit 0 = 3x3 / stride-1 convolutions with an N tile <= 128 take the halo-tile forward kernel, bit 1 =
 * its A descriptors carry an explicit base offset, bit 2 = never fall back to single 128-pixel tiles on small maps, bit 3 = layers with Cout <= 128 keep pixels on the M side
 * (no swapped-operand mode), key 7 = 1: single-output-channel layers with a wide input (PatchGAN head) skip the tiled head kernel.
 * The Python binding sets them from S2E_DEBUG="key=value,...". */
int s2e_debug_set(int key, int value);

/* ------------------------------------------------------------------------------------------
 * Integer path (bit-exact).  pix2pix_model.py:138-152 (one-hot scatter_), normalization.py:97 and
 * generator.py:72 (F.interpolate nearest: src = min(floor(dst * float(in)/float(out)), in-1)).
 * ------------------------------------------------------------------------------------------ */
int s2e_onehot_nchw(const int64_t* label, int B, int H, int W, int nc, float* out_nchw, void* stream);
/* nearest-resize an NCHW fp32 map (one-hot or soft) to (Hd,Wd) and emit NHWC bf16 with Cpad >= C channels. */
int s2e_seg_nearest_nhwc(const float* seg_nchw, int B, int C, int Hs, int Ws, int Hd, int Wd, int Cpad,
                         void* out_nhwc_bf16, void* stream);

/* nearest-resize + 3x3 im2col (zero padded) of a thin map (9*C <= 62) into 64 bf16 channels per pixel: channel
 * (r*3+s)*C + c, zeros up to channel 61 and a CONSTANT ONE in channels 62 and 63.  SPADE's mlp_shared
 * (normalization.py:85-88,98) then runs as a K=64 GEMM on the tensor-core kernels.  The matching weight layout is
 * [Cout][64] with the conv bias split into two bf16 columns (63: bf16(b), 62: bf16(b - bf16(b)); s2e_pack_weight_multi,
 * im2col3x3 job with `bias`), so the bias add rides in the GEMM at ~fp32 precision, and the adjoint (unpack of the fp32
 * weight gradient) returns the bias gradient from column 63. */
int s2e_seg_im2col3x3(const float* seg_nchw, int B, int C, int Hs, int Ws, int Hd, int Wd, void* out_nhwc64_bf16,
                      void* stream);
int s2e_pack_weight_im2col3x3(const float* w_oihw, int Cout, int C, void* out_bf16, void* stream); /* columns 62, 63 = 0 */
int s2e_unpack_wgrad_im2col3x3(const float* dwp, int Cout, int C, float* dw_oihw, float* db /* nullable */,
                               void* stream);

/* layout / precision boundary of the module API (NCHW fp32 <-> NHWC bf16) */
int s2e_nchw_f32_to_nhwc_bf16(const float* x, int B, int C, int H, int W, void* y, void* stream);
int s2e_nhwc_bf16_to_nchw_f32(const void* x, int B, int C, int H, int W, float* y, void* stream);

/* ------------------------------------------------------------------------------------------
 * Convolution as a stride-1 "tap convolution":
 *     y[b,ho,wo,:] = act( scale * sum_t  x[b, ho+dy[t], wo+dx[t], :] . Wp[t] + bias )
 * with zero fill outside the input.  Replaces every nn.Conv2d on the path: normalization.py:85-89
 * (mlp_shared/gamma/beta), architecture.py:24-27 (conv_0/1/s), generator.py:30,48 (fc, conv_img),
 * encoder.py:23-38, discriminator.py:84-96.  Stride-2 convolutions are expressed on a
 * space-to-depth input (s2e_space_to_depth) so one kernel family serves all geometries; the data
 * gradient is the same operator with negated taps and transposed weights.
 * Wp is bf16 [ntaps][Cout][Cin] (s2e_pack_weight).  `scale` is a device scalar (1/sigma of the
 * spectral norm, normalization.py:26 / architecture.py:31-34) or NULL.
 * impl = S2E_IMPL_TC requires Cin % 64 == 0 and Cout % 8 == 0; tile = tile_w*tile_h*tile_b <= 128 pixels.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int B, Hi, Wi, Cin;
  int Ho, Wo, Cout;
  int ntaps;
  int tap_dy[S2E_MAX_TAPS];
  int tap_dx[S2E_MAX_TAPS];
  int act;
  int tile_w, tile_h, tile_b; /* TC forward tile (<=128 px); 0 = choose inside */
  int ktile_w, ktile_h, ktile_b; /* TC wgrad pixel tile (multiple of 16, <=64 px); 0 = choose inside */
  const void* relu_mask;         /* optional bf16 tensor shaped like y: y is zeroed where mask <= 0 (fused ReLU backward
                                    when the operator computes the data gradient of a layer whose input came from a ReLU) */
  const void* residual;          /* optional bf16 tensor shaped like y, added after the activation: the `x_s + dx` of
                                    architecture.py:44 fused into conv_1's epilogue (tcgen05 path only) */
  int bias_n;                    /* number of valid bias entries, 0 = Cout (a channel-padded output, see DESIGN.md) */
  int in_act;                    /* activation applied to x as it is loaded (forward and weight gradient): the
                                    F.leaky_relu(x, 2e-1) in front of conv_img, generator.py:97-98.  CUDA-core kernels only */
  float mask_slope;              /* with relu_mask: where mask <= 0 the output is multiplied by this instead of zeroed
                                    (LeakyReLU backward fused into a data gradient).  CUDA-core kernels only */
  /* Fused SPADE+Style modulation for inference / no-grad forwards (normalization.py:91-105,161-192): the convolution is
   * the gamma|beta convolution (Cout = 2*spade_C, spade_C in {64, 128}) and instead of gamma|beta the kernel writes
   *   y[B][Ho][Wo][spade_C] = act( 0.5 * [ (x*ka + kb) * (1 + gamma) + beta + x*kc + s1 ] )
   * spade_x: the block input x (bf16 NHWC, spade_C channels; at half resolution when spade_up != 0, see s2e_spade_style_fwd);
   * spade_par: float [B][4][spade_C] = ka (rstd), kb (-mean*rstd), kc (1 + s0), s1 (s2e_spade_params).  tcgen05 path only */
  const void* spade_x;
  const float* spade_par;
  int spade_C, spade_act, spade_up;
  void* spade_gamma_out;         /* training (nullable): gamma alone, bf16 [B][Ho][Wo][spade_C] -- all that backward needs
                                    of gamma|beta (s2e_spade_style_bwd with gb_stride = spade_C) */
  void* spade_mask_out;          /* training (nullable): the activation bit mask of s2e_spade_style_fwd */
  int spade_plain;               /* != 0: plain SPADE (normalization.py:91-105 without the ApplyStyle half): the epilogue writes
                                    act(norm(x) (1 + gamma) + beta) -- no style term, no factor 1/2 (s2e_spade_params with
                                    style == NULL zeroes the style rows of `spade_par`) */
  /* image head (generator.py:97-99 conv_img -> tanh, 64 -> 1 channel, 3x3; CUDA-core tile kernel only): */
  float* img_out;                /* != NULL: tanh(conv) is written here as fp32 (B,1,H,W); `y` is not written */
  const float* img_target;       /* nullable: the target image, same shape */
  float* img_sums;               /* with img_target: [0] += sum |tanh(conv) - target|, [1] += sum (.)^2 (caller zeroes): the
                                    reductions of the L1 / L2 image losses (pix2pix_model.py:197-208) ride in this kernel */
} s2e_conv_t;

int s2e_tapconv_fwd(const s2e_conv_t* d, const void* x, const void* wp, const float* bias, const float* scale,
                    void* y, int impl, void* stream);
/* dWp[t][co][ci] += sum_pixels dy[p,co] * x[p+tap_t,ci]   (fp32, atomically accumulated; caller zeroes) */
int s2e_tapconv_wgrad(const s2e_conv_t* d, const void* x, const void* dy, float* dwp, int impl, void* stream);

/* PatchGAN logit head (discriminator.py:38 / :96 in the stock layout: nn.Conv2d(8*ndf, 1, kernel_size=4, stride=1,
 * padding=2), the last block of NLayerDiscriminator) in tap-channel form, y[p] = sum_t D[p + tap_t][t] with
 * D[q][t] = x[q] . W[t]: the wide input is read once, not once per tap.
 *   s2e_head_dots    D[P][16] fp32 (taps >= ntaps: 0) from x [P][Cin] bf16 and the tap-major weight copy wp [ntaps][Cin] bf16
 *   s2e_head_gather  y [B][Ho][Wo][1] bf16 = act(scale * sum_t D[...] + bias); geometry, taps and act from the descriptor.
 *                    gan_sums (nullable, 6 floats, caller-zeroed): the batch is [fake ; real] (pix2pix_model.py:328-338) and the
 *                    kernel adds, per half h, [3h] += sum y, [3h+1] += sum min(y-1, 0), [3h+2] += sum min(-y-1, 0): the reductions of
 *                    GANLoss's hinge / Wasserstein terms (loss.py:58-83) fused into the epilogue that produces the logits
 *   s2e_head_scatter G [B][Hi][Wi][64] bf16, G[q][t] = dy[q - tap_t] (0 outside the output / for t >= ntaps): the data and
 *                    weight gradients are then the 1x1 tap convolutions dx = G . W (64 -> Cin) and dW = G^T . x. */
int s2e_head_dots(const void* x_bf16, const void* wp_bf16, long long P, int Cin, int ntaps, float* D, void* stream);
int s2e_head_gather(const s2e_conv_t* d, const float* D, const float* bias, const float* scale, void* y_bf16, float* gan_sums,
                    void* stream);
int s2e_head_scatter(const s2e_conv_t* d, const void* dy_bf16, void* G_bf16, void* stream);
/* s2e_head_gather that also adds sign_sums[0] += sum sign(y) over the half b >= B/2 (the real logits of a [fake ; real]
 * batch; y as rounded to bf16, sign(0) = 0): the statistic of --ada_target.  sign_sums: one caller-zeroed float; B even and
 * B/2 * Ho * Wo < 2^24, so the fp32 sum of +-1 is exact whatever the order of the atomics. */
int s2e_head_gather_signs(const s2e_conv_t* d, const float* D, const float* bias, const float* scale, void* y_bf16,
                          float* gan_sums, float* sign_sums, void* stream);

/* OIHW fp32 master weight -> bf16 tap-major.  stride 1: taps (r,s) row-major, offset (r-pad, s-pad).
 * stride 2: space-to-depth taps (a,b), a in [floor(-pad/2), floor((k-1-pad)/2)], channel (i*2+j)*Cin+ci,
 * r = 2a+i+pad.  transposed=1 emits [t][Cin'][Cout] (data-gradient operand).
 * Several OIHW tensors can be packed side by side along Cout (the fused gamma|beta GEMM): the packed tensor has
 * Cout_total output channels and this call fills [co_offset, co_offset+Cout). */
int s2e_pack_weight(const float* w_oihw, int Cout, int Cin, int kh, int kw, int stride, int pad, int transposed,
                    int Cout_total, int co_offset, int cin_pad, void* out_bf16, void* stream);
/* cin_pad (0 = none): the activations carry cin_pad >= Cin channels (extra ones zero), e.g. the 5-channel D input
 * stored with 16 channels so that discriminator.py:84's first conv also runs on the tensor-core path. */
int s2e_packed_taps(int kh, int kw, int stride, int pad, int* ntaps, int* dy, int* dx); /* host helper */
/* Several s2e_pack_weight / s2e_pack_weight_im2col3x3 calls in one launch (all the packed copies that an optimizer
 * step invalidated).  `jobs` is a HOST array; im2col3x3 != 0 selects the [Cout][64] layout (then only w, out, Cout,
 * Cin are read). */
typedef struct {
  const float* w_oihw;
  const float* bias; /* im2col3x3 jobs only (nullable): written to columns 62 | 63 */
  void* out_bf16;
  int Cout, Cin, kh, kw, stride, pad, transposed, Cout_total, co_offset, cin_pad, im2col3x3;
} s2e_pack_job_t;
int s2e_pack_weight_multi(const s2e_pack_job_t* jobs, int n_jobs, void* stream);
/* tap-major fp32 weight gradient -> OIHW, with the spectral-norm chain rule when u != NULL:
 * dW_orig = inv_sigma * (G - inv_sigma * <G, W_orig> u v^T).  `dot` is a 1-float device scratch. */
int s2e_unpack_wgrad(const float* dwp, int Cout, int Cin, int kh, int kw, int stride, int pad, int Cout_total,
                     int co_offset, int cin_pad, const float* w_orig, const float* u, const float* v,
                     const float* inv_sigma, float* dot, float* dw_oihw, int accumulate, void* stream);
/* torch.nn.utils.spectral_norm power iteration (one step) on W viewed as (rows, cols):
 * v <- normalize(W^T u), u <- normalize(W v), inv_sigma <- 1 / (u . W v); eps 1e-12. scratch: rows + cols + ceil(rows/64)*cols floats
 * (fixed-order partial sums: the iteration is bitwise reproducible).
 * update = 0 (module in eval mode): u, v are left untouched and only inv_sigma is produced. */
int s2e_spectral_power_iter(const float* w, int rows, int cols, float* u, float* v, float* inv_sigma, float* scratch,
                            int update, float* u_copy, float* v_copy, void* stream); /* *_copy: optional snapshots */
/* The same iteration for a whole table of independent layers (all spectral-normed convolutions of one network, as
 * generator.py / discriminator.py / encoder.py build them) in four launches per iteration instead of four per layer.
 * `jobs` is a HOST array.  n_iters > 1 repeats the iteration (the reference calls netE once per sample,
 * pix2pix_model.py:285, so its u / v advance B times per step): iteration i writes inv_sigma[i] and, when given,
 * u_copy + i*rows / v_copy + i*cols.  Arithmetic per layer is identical to s2e_spectral_power_iter (which is this
 * call with one job). */
typedef struct {
  const float* w;
  float* u;
  float* v;
  float* inv_sigma;
  float* scratch;
  float* u_copy;
  float* v_copy;
  int rows, cols;
} s2e_sn_job_t;
int s2e_spectral_power_iter_multi(const s2e_sn_job_t* jobs, int n_jobs, int update, int n_iters, void* stream);

/* [B,H,W,C] -> [B,ceil(H/2),ceil(W/2),4C] with channel (i*2+j)*C+c = x[2h+i, 2w+j, c] (zero beyond the edge),
 * and its adjoint (gradient) */
int s2e_space_to_depth(const void* x, int B, int H, int W, int C, void* y, void* stream);
int s2e_depth_to_space(const void* dy, int B, int H, int W, int C, void* dx, void* stream);

/* ------------------------------------------------------------------------------------------
 * SPADE+Style normalisation / modulation (normalization.py:91-105,161-169,184-192):
 *   out = act( 0.5 * [ (x-mean)*rstd*(1+gamma) + beta  +  x*(1+s0) + s1 ] )
 * x [B,HW,C] bf16, gb [B,HW,2C] bf16 (gamma | beta), style [B,2C] fp32 (s0 | s1).  mean/rstd are per
 * channel (param-free BatchNorm2d, training mode) or per (sample, channel) (InstanceNorm2d).
 * ------------------------------------------------------------------------------------------ */
/* acc: double [G][3][C] (G = per_sample ? B : 1), written inside: rows sum (x - p), sum (x - p)^2 and the pivot p[c] = the
 * group's first pixel.  Shifted moments: E[x^2] - E[x]^2 from fp32 partial sums cancels badly for channels whose mean is
 * large against their spread.  Plain sum = row 0 + n * row 2. */
int s2e_norm_stats(const void* x, int B, int HW, int C, int per_sample, double* acc, void* stream);
/* mean/rstd float [G][C]; running_* may be NULL; biased var for rstd, unbiased for running_var.
 * count = number of elements behind `acc`; count_unbiased (0 = count) = number of elements the normalised tensor has
 * -- they differ when the statistics of a nearest-2x up-sampled tensor are taken from its 4x smaller source. */
int s2e_norm_finalize(const double* acc, int G, int C, double count, double count_unbiased, float eps, float* mean,
                      float* rstd, float* running_mean, float* running_var, float momentum,
                      int64_t* num_batches_tracked, void* stream);
/* Batch statistics shared by several ranks (SyncBatchNorm, normalization.py:72-78 rejects `syncbatch`; the reference SPADE
 * model's default --norm_G spectralspadesyncbatch3x3 takes them from the vendored sync_batchnorm, batchnorm.py:102-105,
 * which all-reduces raw sums).  records: double [world][3C + 1], rank r's acc of s2e_norm_stats (G = 1) followed by its
 * element count n_r (0 for an empty shard).  Combined in rank order with Chan's pairwise update of (mean, M2), never
 * through raw moments; acc receives the result in the acc format (pivot = global mean, sum (x - p) = 0, sum (x - p)^2 =
 * M2), count (one double) the total element count. */
int s2e_norm_merge(const double* records, int world, int C, double* acc, double* count, void* stream);
/* s2e_norm_finalize (G = 1) with the element count read from the device (`count` of s2e_norm_merge); the unbiased
 * running_var correction uses count * unbiased_factor (4 when the statistics come from a nearest-2x up-sampling's source). */
int s2e_norm_finalize_merged(const double* acc, const double* count, int C, double unbiased_factor, float eps, float* mean,
                             float* rstd, float* running_mean, float* running_var, float momentum,
                             int64_t* num_batches_tracked, void* stream);
/* act_mask (nullable): one BIT per element, [B*HW][C/8] bytes, bit j of byte (p, c/8) = (out[p][c+j] > 0); all the
 * backward pass needs to know about `out` (read instead of it: 0.125 B/element instead of 2). */
/* up_w != 0: x is the [B][H/2][W/2][C] tensor whose nearest-2x up-sampling (generator.py:50) is the block input; up_w = W
 * of the up-sampled map.  The up-sampled copy is never materialised; mean / rstd of the two are identical.  In backward
 * dx is then the gradient w.r.t. the HALF-RESOLUTION x itself, [B][HW/4][C]: the kernel adds the four output pixels of
 * every source pixel on the spot (the adjoint of the up-sampling), the full-resolution gradient is never written.
 * style == NULL selects plain SPADE: out = act(norm(x) (1 + gamma) + beta), no style term, no factor 1/2 (dstyle must
 * be NULL then). */
/* per-(sample, channel) constants of the fused variant (s2e_conv_t.spade_par): par[b][0..3][c] = rstd, -mean*rstd,
 * 1 + style[b][c], style[b][C + c]; mean / rstd are [G][C] with G = per_sample ? B : 1 */
int s2e_spade_params(const float* mean, const float* rstd, const float* style, int B, int C, int per_sample, float* par,
                     void* stream);
int s2e_spade_style_fwd(const void* x, const void* gb, const float* style, const float* mean, const float* rstd,
                        int B, int HW, int C, int per_sample, int act, void* out, uint8_t* act_mask, int up_w,
                        void* stream);
/* backward: racc = scratch of B*5*C doubles + B*2*C floats + 2*C + 1 doubles, zeroed inside. `act_mask` = the forward pass's mask (may be
 * NULL when act == NONE).  chsum (nullable, float [3][C]) receives the per-channel sums over the batch of dgamma, dbeta
 * and dx -- the bias gradients of the gamma|beta convolution (normalization.py:88-89) and of the convolution that
 * produced x (architecture.py:24) -- which the statistics pass yields for free.  dx_accumulate != 0 adds into dx
 * (two SPADE+Style blocks that share their input, norm_0 / norm_s of architecture.py:51-58, write ONE gradient buffer);
 * the third row of chsum then covers this call's contribution only.  per_sample: bit 0 = statistics per sample
 * (InstanceNorm), bit 1 = the statistics are constants (BatchNorm in eval mode, running statistics): dx has no
 * mean / projection terms (chsum's third row is not meaningful then). */
int s2e_spade_style_bwd(const void* dout, const uint8_t* act_mask, const void* x, const void* gb, const float* style,
                        const float* mean, const float* rstd, int B, int HW, int C, int per_sample, int act,
                        double* racc, void* dx, int dx_accumulate, void* dgb, float* dstyle, float* chsum, int up_w,
                        int gb_stride /* channels per pixel of `gb`: 0 = 2C (gamma|beta); C when only gamma was kept */,
                        void* stream);
/* s2e_spade_style_bwd in two halves, so that ranks sharing batch statistics can add their per-channel sums in between
 * (normalization.py:75 with SyncBatchNorm: the statistics, hence their gradient terms, span the global batch).
 * reduce: the raw-moment pass and the fold; dstyle and chsum as above (chsum's third row relies on the normalisation
 * part of dx summing to zero, which under shared statistics holds over the global batch only: a rank's value is off by
 * its share, and the shares cancel when the bias gradients are summed across ranks).  For batch statistics (bit 0 of
 * per_sample clear) sums = double [2][C] + 1: S1 = sum dxhat, S2 = sum dxhat * xhat per channel and this call's element
 * count B*HW; per-sample statistics keep theirs in racc.  racc = scratch of B*5*C doubles + B*2*C floats.
 * apply: dx / dgamma|dbeta from racc and sums, whose S1, S2 and count may have been summed over ranks (m1 = S1 / count,
 * m2 = S2 / count).  Running the two back to back is s2e_spade_style_bwd, bit for bit. */
int s2e_spade_style_bwd_reduce(const void* dout, const uint8_t* act_mask, const void* x, const void* gb, const float* style,
                               const float* mean, const float* rstd, int B, int HW, int C, int per_sample, int act,
                               double* racc, double* sums, float* dstyle, float* chsum, int up_w, int gb_stride,
                               void* stream);
int s2e_spade_style_bwd_apply(const void* dout, const uint8_t* act_mask, const void* x, const void* gb, const float* style,
                              const float* mean, const float* rstd, int B, int HW, int C, int per_sample, int act,
                              const double* racc, const double* sums, void* dx, int dx_accumulate, void* dgb, int up_w,
                              int gb_stride, void* stream);

/* InstanceNorm2d(affine=False)+optional LeakyReLU on NHWC bf16 (normalization.py:41; discriminator.py:88-92;
 * encoder.py:23-38).  in_scale (nullable): one factor per `group` consecutive images, applied to x implicitly. */
/* pair_l1 (nullable, one float, caller-zeroed): the batch is the [fake ; real] pair of a discriminator feature map and the apply
 * pass also adds sum |y[b] - y[b + B/2]| (bf16 values) to it: the feature-matching reduction of pix2pix_model.py:233-241. */
int s2e_instnorm_fwd(const void* x, int B, int HW, int C, int act, float eps, const float* in_scale, int group,
                     double* acc, float* mean, float* rstd, void* y, float* pair_l1, void* stream);
/* Batched style encoder (pix2pix_model.py:285 calls netE once per sample, so sample b sees its own 1/sigma_b):
 * the convolution runs unscaled, in_scale[n / group] folds 1/sigma_b into the InstanceNorm statistics, and the
 * spectral chain-rule term  dW_orig -= sum_b c_b u_b v_b^T,  c_b = (eps/is_b) sum_{n in b, c} S2[n,c] rstd'[n,c]^2
 * (S2 = sum_hw g*xhat, the second accumulator of s2e_instnorm_bwd) is produced here.  coef: B floats scratch. */
int s2e_sn_in_correction(const double* racc, const float* rstd, const float* inv_sigma, int Bn, int group, int C,
                         float eps, const float* U, const float* V, int K, float* coef, float* dw, void* stream);
/* y is unused (may be NULL): the sign the activation saw is that of fma(x, rstd, -mean * rstd), which backward recomputes */
int s2e_instnorm_bwd(const void* dy, const void* y, const void* x, const float* mean, const float* rstd, int B, int HW,
                     int C, int act, double* racc, void* dx, void* stream);

/* ------------------------------------------------------------------------------------------ elementwise */
int s2e_upsample2x_fwd(const void* x, int B, int H, int W, int C, void* y, void* stream);     /* generator.py:50 */
int s2e_upsample2x_bwd(const void* dy, int B, int H, int W, int C, void* dx, void* stream);
int s2e_add(const void* a, const void* b, long long n, void* y, void* stream);                /* architecture.py:52 */
int s2e_act_fwd(const void* x, long long n, int act, void* y, void* stream);                  /* generator.py:98 */
int s2e_act_bwd(const void* dy, const void* y, long long n, int act, void* dx, void* stream); /* mask from output sign */
/* F.avg_pool2d(3, stride 2, pad 1, count_include_pad=False) on NHWC bf16 (discriminator.py:46-49) */
int s2e_avgpool3s2_fwd(const void* x, int B, int H, int W, int C, void* y, void* stream);
int s2e_avgpool3s2_bwd(const void* dy, int B, int H, int W, int C, void* dx, void* stream);
/* F.interpolate(bilinear, align_corners=False) of single-channel-style NCHW fp32 planes -> bf16 (encoder.py:55) */
int s2e_bilinear_fwd(const float* x, int N, int Hs, int Ws, int Hd, int Wd, void* y_bf16, void* stream);
int s2e_bilinear_bwd(const void* dy_bf16, int N, int Hs, int Ws, int Hd, int Wd, float* dx, void* stream);
/* D input: cat([seg, fake],1) / cat([seg, real],1) / cat(.,0) as NHWC bf16 with Cpad channels (pix2pix_model.py:328-338) */
int s2e_make_d_input(const float* seg_nchw, const float* fake, const float* real, int B, int nc, int H, int W,
                     int Cpad, void* out, void* stream);
/* tanh on fp32 output of conv_img and its backward (generator.py:99) */
int s2e_tanh_fwd(const void* x_bf16, long long n, float* y, void* stream);
int s2e_tanh_bwd(const float* dy, const float* y, long long n, void* dx_bf16, void* stream);
/* gradient of the fake image w.r.t. the D input channel nc (first B samples) -> fp32 (B,1,H,W) */
int s2e_d_input_grad(const void* dxin, int B, int nc, int H, int W, int Cpad, float* dfake, void* stream);

/* Differentiable augmentation of the D input (--diff_augment, beyond the reference; DiffAugment, Zhao et al., NeurIPS
 * 2020: rand_brightness, rand_saturation, rand_contrast, rand_translation, rand_cutout, applied in that order).
 *
 * Parameters.  s2e_diffaug_draw writes one record of S2E_DIFFAUG_RECORD fp32 values per sample b < B,
 *     (u0, u1, tx, ty, ox, oy),
 * from Philox4x32-10 with key = (seed lo, seed hi) and counter = (n, ctr lo, ctr hi, blk), where state[0] = seed,
 * state[1] = ctr (both int64, device memory) and n = index_offset + b (the sample's global index, < 2^32).  Block
 * blk = 0 gives the words (r0, r1, r2, r3), block 1 gives (r4, r5, -, -).  A word r maps to
 *     a float in [0, 1):        (r >> 8) * 2^-24
 *     an integer in [0, n):     (r * n) >> 32        (64-bit product)
 * and   u0 = float(r0), u1 = float(r1),
 *       tx = int(r2, 2 sx + 1) - sx,  ty = int(r3, 2 sy + 1) - sy,   sx = (H + 4) / 8, sy = (W + 4) / 8  (= int(H/8 + 0.5)),
 *       ox = int(r4, H + 1 - cx % 2), oy = int(r5, W + 1 - cy % 2),  cx = (H + 1) / 2, cy = (W + 1) / 2  (= int(H/2 + 0.5)).
 * All six are drawn whatever the policy, so an op's parameters never depend on which other ops are on.  One launch
 * (one block); it reads ctr on the device and then sets state[1] = ctr + 1, so every replay of a captured CUDA graph
 * draws new parameters.
 *
 * Ops, per sample, on the H x W map (policy = OR of the S2E_DIFFAUG_* bits; row b of [fake ; real] and row B + b use
 * record b):
 *   COLOR (image channel only):  x'' = (x' - mean(x')) (u1 + 0.5) + mean(x'),  x' = x + (u0 - 0.5), the mean over the
 *       H x W pixels of that image (s2e_diffaug_means: fp32 values, fp64 sums).  Saturation is the identity on one
 *       channel and is not drawn.
 *   TRANSLATION (every channel):  out[i, j] = in[i + tx, j + ty], 0 where that index is outside the map.
 *   CUTOUT (every channel):  out[i, j] = 0 for ox - cx/2 <= i < ox - cx/2 + cx and oy - cy/2 <= j < oy - cy/2 + cy. */
#define S2E_DIFFAUG_COLOR 1
#define S2E_DIFFAUG_TRANSLATION 2
#define S2E_DIFFAUG_CUTOUT 4
#define S2E_DIFFAUG_ALL 7
#define S2E_DIFFAUG_RECORD 6
int s2e_diffaug_draw(int64_t* state, int B, long long index_offset, int H, int W, float* params_out, void* stream);
/* means_out[b] = mean(fake[b]), means_out[B + b] = mean(real[b]); fake, real fp32 (B,1,H,W) */
int s2e_diffaug_means(const float* fake, const float* real, int B, int H, int W, float* means_out, void* stream);
/* s2e_make_d_input with the policy applied while gathering (colour in fp32 on the image value, one rounding to bf16);
 * channels nc + 1 .. Cpad - 1 stay zero.  means: s2e_diffaug_means's output, needed with COLOR only. */
int s2e_make_d_input_aug(const float* seg_nchw, const float* fake, const float* real, int B, int nc, int H, int W,
                         int Cpad, const float* params, const float* means, int policy, void* out, void* stream);
/* adjoint of s2e_make_d_input_aug for the fake image: g'[i, j] = dxin[b, i - tx, j - ty, nc] (0 where that output pixel
 * does not exist or is cut out), then with COLOR dfake = c g' + (1 - c) mean(g'), c = u1 + 0.5 (brightness passes the
 * gradient unchanged).  scratch: B doubles (the per-sample sums of g'), needed with COLOR only; two launches with COLOR,
 * one without. */
int s2e_d_input_grad_aug(const void* dxin, int B, int nc, int H, int W, int Cpad, const float* params, int policy,
                         double* scratch, float* dfake, void* stream);

/* Per-sample gates of the ops (--diff_augment_p, --ada_target; ADA, Karras et al., NeurIPS 2020).
 * s2e_diffaug_draw_p writes params_out exactly as s2e_diffaug_draw does (and advances the counter by one, as it does), and
 * opmask_out[b] = the S2E_DIFFAUG_* bits whose gate passed, op k passing iff  (double)float(r_k) < *p  with the gate words
 *     COLOR: r6 = block 1, word 2     TRANSLATION: r7 = block 1, word 3     CUTOUT: r8 = block 2, word 0
 * of the same Philox counter (block 2 = counter (n, ctr lo, ctr hi, 2)).  p: one double in device memory, 0 <= p <= 1; at
 * p = 1 every gate passes, at p = 0 none does.
 * The _masked twins of s2e_make_d_input_aug / s2e_d_input_grad_aug apply policy & opmask[b] to sample b (rows b and B + b);
 * a sample whose colour gate is off passes its gradient through exactly.  With an empty mask they equal s2e_make_d_input /
 * s2e_d_input_grad, with a full mask the unmasked entry points, bit for bit. */
int s2e_diffaug_draw_p(int64_t* state, const double* p, int B, long long index_offset, int H, int W, float* params_out,
                       int* opmask_out, void* stream);
int s2e_make_d_input_aug_masked(const float* seg_nchw, const float* fake, const float* real, int B, int nc, int H, int W,
                                int Cpad, const float* params, const float* means, int policy, const int* opmask, void* out,
                                void* stream);
int s2e_d_input_grad_aug_masked(const void* dxin, int B, int nc, int H, int W, int Cpad, const float* params, int policy,
                                const int* opmask, double* scratch, float* dfake, void* stream);

/* Horizontal flip and geometric augmentation (--diff_augment xflip,geometric; ADA, Karras et al., NeurIPS 2020, the
 * "geometric" group without rotate90 and xint).  Canonical order: color -> xflip -> geometric -> translation -> cutout.
 *
 * Geometry.  Pixel units, x = column, y = row, centred: xc = j - (W-1)/2, yc = i - (H-1)/2.  Sample b has one inverse
 * 2x3 matrix M (rows b and B + b share it), mapping an output point to its source point:
 *     M = F . S(1/s) . R(-th1) . diag(1/a, a) . R(-th2) . T(-tx W, -ty H)        (ADA's G_inv order)
 * with R(t) = [[cos t, -sin t], [sin t, cos t]] and every factor whose gate is off the identity:
 *     F = diag(-1, 1) (mirror),  s = 2^(0.2 n0),  a = 2^(0.2 n1),  thk = pi (2 u - 1),  (tx, ty) = 0.125 (n2, n3),
 * composed in fp64 and rounded once to fp32 (m0 m1 m2 / m3 m4 m5 row-major, then two zero pads).
 *
 * Draw.  s2e_diffaug_draw_geom writes params_out and opmask bits COLOR / TRANSLATION / CUTOUT exactly as
 * s2e_diffaug_draw_p does, geom_out [B, S2E_DIFFAUG_GEOM_RECORD] fp32, and advances the counter by one.  Words of the
 * same Philox counter (block k = counter (n, ctr lo, ctr hi, k)); gates pass iff (double)unit(r) < q, unit as above:
 *     block 2, words 1..3: xflip gate (q = p), mirror coin (q = 0.5), scale gate (q = p)
 *     block 3, words 0..3: pre-rotation gate (q = p_rot), aniso gate (p), post-rotation gate (p_rot), xfrac gate (p)
 *     block 4: Box-Muller of words 0, 1 -> (n0, n1); th1 from word 2, th2 from word 3
 *     block 5: Box-Muller of words 0, 1 -> (n2, n3)
 * p_rot = 1 - sqrt(max(1 - p, 0)) (fp64).  Box-Muller in fp64: u = ((r0 >> 8) + 0.5) 2^-24, v likewise from r1,
 * n0 = sqrt(-2 ln u) cos(2 pi v), n1 = sqrt(-2 ln u) sin(2 pi v); |n| <= 5.9, so s and a lie in about [0.44, 2.3].
 * Every parameter is drawn whatever the gates.  opmask bit XFLIP: the mirror is applied (xflip gate and coin);
 * bit GEOMETRIC: some of the five geometric gates passed.
 *
 * Sampling (s2e_make_d_input_aug_geom; sample b applies policy & opmask[b], and M without F when the policy lacks XFLIP).
 * A sample with neither new bit takes s2e_make_d_input_aug_masked's path, bit for bit; XFLIP alone reads column
 * W-1-j exactly.  Otherwise an output pixel is first moved by cutout and translation to the warped-image position
 * (si, sj) as above (zero outside), then, in fp32 without contraction,
 *     X = ((m0 xc + m1 yc) + m2) + (W-1)/2,   Y = ((m3 xc + m4 yc) + m5) + (H-1)/2,   xc = sj - (W-1)/2, yc = si - (H-1)/2;
 * the image channel is sampled bilinearly at the taps floor(X) + {0, 1}, floor(Y) + {0, 1} (weights from the fp32
 * fractions), the label channels at the nearest tap floor(X + 0.5), floor(Y + 0.5) (labels stay one-hot); every tap
 * index k is folded into [0, n) by reflection, fold(k, n): m = 2(n-1), k' = k mod m, k' < n ? k' : m - k' (torch's
 * 'reflect', repeated).  Colour is applied to the sampled value, then one rounding to bf16.  Needs H, W >= 2.
 * Departures from ADA, deliberate: labels are sampled nearest, not warped alike, and there is no 2x oversampling with
 * wavelet filters.
 *
 * Adjoint (s2e_d_input_grad_aug_geom, the fake image): with h the gathered gradient of s2e_d_input_grad_aug at the
 * warped-image position, dfake = Warp^T(h) (mirror alone: h at column W-1-j), then colour's c dfake + (1 - c) sum(h)/HW.
 * Warp^T is a gather with a fixed summation order (deterministic, no atomics): each source pixel enumerates its mirror
 * images +-s + 2k(n-1) within the bounding box of M (output rect) widened by two pixels (the second tap, and margin for
 * the fp32 coordinates), scans the integer box of
 * M^-1 (image + [-1, 1]^2) widened by one pixel (fp64), and accepts a candidate only if the forward's fp32 taps land on it. */
#define S2E_DIFFAUG_XFLIP 8
#define S2E_DIFFAUG_GEOMETRIC 16
#define S2E_DIFFAUG_ALL_GEOM 31
#define S2E_DIFFAUG_GEOM_RECORD 8
int s2e_diffaug_draw_geom(int64_t* state, const double* p, int B, long long index_offset, int H, int W, float* params_out,
                          float* geom_out, int* opmask_out, void* stream);
int s2e_make_d_input_aug_geom(const float* seg_nchw, const float* fake, const float* real, int B, int nc, int H, int W,
                              int Cpad, const float* params, const float* means, int policy, const int* opmask,
                              const float* geom, void* out, void* stream);
int s2e_d_input_grad_aug_geom(const void* dxin, int B, int nc, int H, int W, int Cpad, const float* params, int policy,
                              const int* opmask, const float* geom, double* scratch, float* dfake, void* stream);
/* ADA's controller, one thread, device memory only (a replayed CUDA graph adapts).  step_stat: this D step's record
 * [S_0, N_0, ..., S_{D-1}, N_{D-1}, I] (D = num_D; S_i = sum sign(real logits of scale i), N_i = their number, I = the
 * number of real images; all-reduced over the ranks), acc: 2D + 2 doubles (the record's running sums, then the r of the last
 * completed interval), pos: the D steps accumulated so far.  It adds step_stat into acc and, when pos + 1 reaches interval,
 *     r = (1/D) sum_i acc[2i] / acc[2i+1],   p = min(max(p + sign(r - target) * acc[2D] / (kimg * 1000), 0), 1)   (fp64),
 * stores r in acc[2D + 1] and resets the sums and pos to 0. */
int s2e_ada_update(const double* step_stat, int num_D, double* acc, int* pos, double* p, double target, double kimg, int interval,
                   void* stream);

/* small fp32 linear layers: y = act(x W^T + b).  FC 16->2C (normalization.py:134-141), fc_mu/fc_var
 * (encoder.py:68-71).  in_nhwc_hw > 0: x is bf16 NHWC [M, hw, K/hw] flattened in NCHW order with LeakyReLU(0.2)
 * applied to the input first (encoder.py:64-67). */
int s2e_linear_fwd(const void* x, const float* w, const float* b, int M, int N, int K, int act, int in_nhwc_hw,
                   float* y, void* stream);
int s2e_linear_bwd(const float* dy, const float* y, const void* x, const float* w, int M, int N, int K, int act,
                   int in_nhwc_hw, void* dx, float* dw, float* db, void* stream);

/* ------------------------------------------------------------------------------------------ losses
 * Reductions write fp32 scalars: out[0] (+)= coef * sum(f(x)).  loss.py:58-83, pix2pix_model.py:193-241. */
#define S2E_RED_SUM 0        /* x            (hinge G: -mean(x))        */
#define S2E_RED_HINGE_REAL 1 /* min(x-1,0)                              */
#define S2E_RED_HINGE_FAKE 2 /* min(-x-1,0)                             */
#define S2E_RED_L1 3         /* |x-y|                                   */
#define S2E_RED_L2 4         /* (x-y)^2                                 */
#define S2E_RED_LS 5         /* (x-target)^2          gan_mode ls       (loss.py:63-65: mse_loss against the label) */
#define S2E_RED_BCE 6        /* BCE-with-logits(x, target)  gan_mode original (loss.py:59-62) */
#define S2E_RED_SIGN 7       /* sign(x), sign(0) = 0 (ADA's statistic; gradient 0): exact below 2^24 elements */
/* `target` is the constant label of the LS / BCE kinds (ignored by the others). */
int s2e_reduce_loss(const void* x, const void* y, long long n, int x_is_f32, int kind, float coef, float target,
                    float* out, int accumulate, void* stream);
/* dx (+)= gout[0] * coef * f'(x)   (dx same dtype as x) */
int s2e_reduce_loss_bwd(const void* x, const void* y, long long n, int x_is_f32, int kind, float coef, float target,
                        const float* gout, void* dx, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------ optimizer
 * torch.optim.Adam (pix2pix_model.py:105-108).  The step count, learning rate and bias corrections live in a 4-float
 * DEVICE array `state` = {step, lr, lr/(1-b1^step), sqrt(1-b2^step)} so that a whole training step can be replayed
 * from a CUDA graph: s2e_adam_prepare advances it once per optimizer step, s2e_adam_step applies it to one tensor. */
int s2e_adam_prepare(float* state, float beta1, float beta2, void* stream);
int s2e_adam_step(float* p, const float* g, float* m, float* v, long long n, const float* state, float beta1,
                  float beta2, float eps, float weight_decay, void* stream);
/* s2e_adam_step for a list of tensors in one launch per 48 tensors (multi-tensor apply; pix2pix_model.py:92-110 hands
 * ~200 tensors to torch.optim.Adam).  p/g/m/v/n are HOST arrays of n_tensors device pointers / element counts. */
int s2e_adam_multi(int n_tensors, float* const* p, const float* const* g, float* const* m, float* const* v,
                   const long long* n, const float* state, float beta1, float beta2, float eps, float weight_decay,
                   void* stream);
/* s2e_adam_multi plus an exponential moving average of the updated weights (--ema_decay, beyond the reference: the
 * optimizer_G step of pix2pix_model.py:92-110 also advances netG_ema / netE_ema).  `ema` is a HOST array of n_tensors
 * device pointers; after the Adam update of p, e <- fmaf(beta_t, e - p, p) in fp32 with
 * beta_t = min(ema_decay, (1 + t) / (10 + t)) and t = state[0], the step count s2e_adam_prepare just advanced.
 * 0 <= ema_decay < 1.  p, m, v come out bitwise equal to s2e_adam_multi's. */
int s2e_adam_multi_ema(int n_tensors, float* const* p, const float* const* g, float* const* m, float* const* v,
                       const long long* n, const float* state, float beta1, float beta2, float eps, float weight_decay,
                       float* const* ema, float ema_decay, void* stream);
/* dst[i] <- src[i] (nbytes[i] bytes, device memory, any dtype), one launch per 48 rows: the EMA nets take byte copies of
 * the live nets' buffers (spectral-norm u/v, BatchNorm running statistics) after every optimizer_G step.  dst/src/nbytes
 * are HOST arrays. */
int s2e_copy_multi(int n_rows, void* const* dst, const void* const* src, const long long* nbytes, void* stream);
int s2e_fill_f32(float* p, long long n, float value, void* stream);

/* ------------------------------------------------------------------------------------------
 * Validation / inference tail (SURVEY 8(f) row 2) and style aggregation.
 * ------------------------------------------------------------------------------------------ */
/* data/postprocessor.py:57-114 (ImageProcessor.to_255resized_imagebatch, called from util/tester.py:44-47): fp32 images in
 * [-1,1], (N,1,h,w) -> int32 (N,1,H,W) in [0,255]: cv2.resize(INTER_LINEAR) in float64, (x+1)*255/2, .int() -- bit-exact
 * integer result.  f32_path = 1: ImageProcessor.to_255imagebatch on the tensor itself (no resize, fp32 arithmetic;
 * models/networks/loss.py:143-144).  With `target` (int32, same shape as out) the per-image exact sum of squared
 * differences goes to sqsum (N x u64 scratch) and, if `score` != NULL, score[n] = sqrt(sqsum[n]) / (H*W)
 * (models/networks/loss.py:102-133 openEDSaccuracy / MSECalculator). */
int s2e_to255_resize(const float* x, int N, int h, int w, int H, int W, int f32_path, const int* target, int* out,
                     unsigned long long* sqsum, float* score, void* stream);
/* MSECalculator.calculate_mse_for_images (loss.py:113-133) on two int32 (N,1,H,W) batches already on the device */
int s2e_openeds_score(const int* produced, const int* target, int N, int H, int W, unsigned long long* sqsum, float* score,
                      void* stream);
/* Pix2PixModel._aggregate_tensor (pix2pix_model.py:271-278): mean (mode 0) | max (mode 1) over the ns style images:
 * x [G][ns][n] (fp32 or bf16) -> out [G][n] fp32; argmax (u8, max only) feeds the backward pass. */
int s2e_aggregate_fwd(const void* x, int x_is_f32, int G, int ns, long long n, int mode, float* out, uint8_t* argmax, void* stream);
int s2e_aggregate_bwd(const float* dout, const uint8_t* argmax, int x_is_f32, int G, int ns, long long n, int mode, void* dx,
                      void* stream);

/* ------------------------------------------------------------------------------------------
 * Device-side data layer (SURVEY 8(f) row 3): data/openeds_dataset.py:82-119 + data/base_dataset.py:50-80 ('fixed' mode) on
 * raw uint8 frames resident in HBM.  `flip` (nullable) = one byte per sample, != 0: horizontal flip after the resize.
 * ------------------------------------------------------------------------------------------ */
/* mask (N,H0,W0) u8 -> cv2.resize(INTER_NEAREST) to (h,w) -> flip -> int64 (N,1,h,w): the `label` entry of the data dict */
int s2e_label_nearest_flip(const uint8_t* mask, int N, int H0, int W0, int h, int w, const uint8_t* flip, int64_t* out,
                           void* stream);
/* one separable pass of PIL's 8-bit Image.resize (base_dataset.py:88-91): kk [out_size][ksize] 22-bit fixed-point taps and
 * bounds [out_size][2] = (first source index, tap count), computed on the host like Pillow's precompute_coeffs /
 * normalize_coeffs_8bpc.  horizontal != 0: (N,Hin,Win) -> (N,Hin,out_size); else -> (N,out_size,Win). */
int s2e_pil_resample_u8(const uint8_t* in, int N, int Hin, int Win, int out_size, int horizontal, const int* kk,
                        const int* bounds, int ksize, uint8_t* out, void* stream);
/* flip + transforms.ToTensor + Normalize((0.5,), (0.5,)): u8 (N,h,w) -> fp32 ((v / 255) - 0.5) / 0.5; image n uses
 * flip[n / images_per_flag] (the ns style images of a sample share its flag) */
int s2e_u8_flip_normalize(const uint8_t* in, int N, int images_per_flag, int h, int w, const uint8_t* flip, float* out,
                          void* stream);
/* `target_original` (openeds_dataset.py:112-116): the raw target frame, flipped, as int32 */
int s2e_u8_flip_to_i32(const uint8_t* in, int N, int h, int w, const uint8_t* flip, int* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEG2EYE_B200_H_ */
