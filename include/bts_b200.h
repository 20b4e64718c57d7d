/* bts_b200 -- C ABI of the B200-native BTS hot path (libbts_b200.so).
 *
 * This is the native boundary underneath the Python module surface `bts` (BtsModel / encoder / bts /
 * local_planar_guidance / reduction_1x1 / silog_loss, reference pytorch/bts.py).  The reference's only
 * native interface is the TensorFlow custom op (tensorflow/custom_layer/local_planar_guidance.h:22-49:
 * LocalPlanarGuidanceKernel / LocalPlanarGuidanceGradKernel functors taking raw float pointers + sizes);
 * bts_lpg_fwd / bts_lpg_bwd replace exactly those two functors (layout=BTS_LAYOUT_NHWC, tf_compat=1
 * reproduces the op bit-for-formula); every other entry point replaces an ATen/cuDNN call sequence of
 * pytorch/bts.py cited per function.
 *
 * Conventions (all entry points):
 *   - plain pointers are DEVICE pointers (fp32 unless noted); no torch / TF types.
 *   - asynchronous on the caller-supplied CUDA stream (void* == cudaStream_t); never allocates,
 *     never synchronises (the reference op calls d.synchronize() after each launch, .cu:91,170 -- we do not).
 *   - returns 0 on success, a negative BTS_E* on bad arguments, a positive cudaError_t on launch failure.
 *   - `*_h` variants take HOST pointers, do the H2D/D2H copies themselves and synchronise; they are the
 *     reference-facing plugin form used for end-to-end (e2e) measurements and by non-torch callers.
 */
#ifndef BTS_B200_H_
#define BTS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BTS_LAYOUT_NCHW 0 /* plane (B,4,h,w)  -- pytorch/bts.py:135-138 */
#define BTS_LAYOUT_NHWC 1 /* plane (B,h,w,4)  -- custom_layer/local_planar_guidance.cc:102-107 */

#define BTS_EINVAL (-1)   /* bad argument (null pointer, non-positive size, unsupported upratio) */
#define BTS_EALIGN (-2)   /* pointer not 16-byte aligned where the kernel needs it */

/* library / build identification: returns e.g. 100 for sm_100a; writes a short version string */
int bts_version(char *buf, int buflen);

/* ---- Local planar guidance --------------------------------------------------------------------
 * Forward  (pytorch/bts.py:132-146; custom_layer/local_planar_guidance.cu:33-72, .cc:74-115):
 *     depth[b,y,x] = n4 / ((n1*u(x) + n2*v(y)) + n3),  plane of patch (y/r, x/r),
 *     u(x) = ((x mod r) - (r-1)/2)/r  (bit-exact dyadic grid), v(y) likewise.
 * `focal` is unused by the reference in both implementations (SURVEY Q1) and is not a parameter.
 * Optional fused by-products of bts.forward (pytorch/bts.py:228-229,242-243,256); pass NULL to skip:
 *     scaled = depth / max_depth            (B,H,W)
 *     ds     = scaled[:, ::ds_stride, ::ds_stride]   (B,H/ds_stride,W/ds_stride)  nearest down-sample
 * `depth` itself may be NULL when only the by-products are wanted.  upratio r must be 1 or even. */
int bts_lpg_fwd(const float *plane, float *depth, int B, int h, int w, int r, int layout, void *stream);
int bts_lpg_fwd_fused(const float *plane, float *depth, float *scaled, float *ds, float max_depth,
                      int ds_stride, int B, int h, int w, int r, int layout, void *stream);

/* Backward (autograd of pytorch/bts.py:146; custom_layer/local_planar_guidance.cu:95-150, .cc:241-298):
 *     dplane[b,:,i,j] = sum over the r x r tile of (-dY*n4*u/den^2, -dY*n4*v/den^2, -dY*n4/den^2, dY/den)
 * tf_compat=1 drops n4 from the first three (the reference TF kernel's formula, SURVEY Q5).
 * Fused form: dY_total = d_depth + (d_scaled + scatter(d_ds)) / max_depth, any of the three may be NULL. */
int bts_lpg_bwd(const float *dy, const float *plane, float *dplane, int B, int h, int w, int r,
                int layout, int tf_compat, void *stream);
int bts_lpg_bwd_fused(const float *d_depth, const float *d_scaled, const float *d_ds, float max_depth,
                      int ds_stride, const float *plane, float *dplane, int B, int h, int w, int r,
                      int layout, int tf_compat, void *stream);

/* Host-pointer plugin form of the TF op pair (input (B,h,w,4) NHWC, output (B,h*r,w*r)); copies in/out
 * and synchronises.  Mirrors LocalPlanarGuidanceOp::Compute / LocalPlanarGuidanceGradOp::Compute
 * (custom_layer/local_planar_guidance.cc:190-229, 364-416). */
int bts_lpg_fwd_h(const float *plane_host, float *depth_host, int B, int h, int w, int r, int layout);
int bts_lpg_bwd_h(const float *dy_host, const float *plane_host, float *dplane_host, int B, int h, int w,
                  int r, int layout, int tf_compat);

/* ---- silog loss (pytorch/bts.py:41-48) ---------------------------------------------------------
 * mask: uint8/bool, n elements.  ws: >= 4 doubles of device workspace, zeroed by the call.
 * fwd:  d_i = ln est_i - ln gt_i over mask; loss = 10*sqrt(mean(d^2) - lambda*mean(d)^2)  -> loss[0]
 *       ws keeps (sum d, sum d^2, N) for the backward.
 * bwd:  dest_i = gout[0] * mask_i * (10/sqrt(S)) * (d_i - lambda*m1) / (N*est_i)   (SURVEY Appendix B) */
int bts_silog_fwd(const float *est, const float *gt, const uint8_t *mask, long long n, float lambda,
                  double *ws, float *loss, void *stream);
int bts_silog_bwd(const float *est, const float *gt, const uint8_t *mask, long long n, float lambda,
                  const double *ws, const float *gout, float *dest, void *stream);

/* ---- plane-coefficient head tail (pytorch/bts.py:112-120 + 223-229 per scale) -------------------
 * c3: (B,3,h,w) output of reduc.plane_params.  Computes theta=sig(c0)*pi/3, phi=sig(c1)*2pi,
 * dist=sig(c2)*max_depth, n=(sin th cos ph, sin th sin ph, cos th), n^=n/max(|n|,1e-12), plane=(n^,dist),
 * then LPG(r) -> scaled=(depth/max_depth) (B,H,W) and ds (optional, nearest down-sample by ds_stride).
 * plane_out (B,4,h,w) optional (saved for backward / inspection). */
int bts_plane_head_fwd(const float *c3, float *plane_out, float *scaled, float *ds, float max_depth,
                       int ds_stride, int B, int h, int w, int r, void *stream);
/* backward of the above: inputs d_scaled (B,H,W), d_ds (optional), c3; output dc3 (B,3,h,w) */
int bts_plane_head_bwd(const float *d_scaled, const float *d_ds, const float *c3, float *dc3,
                       float max_depth, int ds_stride, int B, int h, int w, int r, void *stream);

/* ---- tcgen05 implicit-GEMM convolution (pytorch/bts.py:51-80,153-194; torchvision dense/bottleneck layers) ----
 * NHWC activations, fp32 in / fp32 out, parity-grade 3xTF32 on the 5th-gen tensor cores (precision=0) or
 * single-pass TF32 (precision=1, labelled fast mode, not parity).
 *   out[p,co] = act( sum_{tap,ci} pre(x[p (+) tap, ci]) * w[co,ci,tap] )
 *   pre : x*pre_scale[ci]+pre_shift[ci] (folded BatchNorm; both NULL to skip), then ReLU if pre_relu;
 *         zero padding is applied after pre.  upsample2=1 folds a nearest x2 up-sample of the source in.
 *   act : 0 none, 1 ELU, 2 sigmoid.
 * x: source (B,Hs,Ws,*) with x_pixel_stride floats between pixels (a channel slice of a wider slab is fine);
 * out likewise with out_pixel_stride.  Weights must first be packed (split hi/lo, K-major, 128B-swizzled tiles):
 *   bts_conv_packed_floats(n_rows, k_channels, KH, KW) -> number of floats of the packed buffer
 *   bts_conv_pack_weights(w, strides of (co,ci,kh,kw) in floats, ..., transpose_flip, wpack)
 *       transpose_flip=0: forward operator (rows = Cout);  1: dgrad operator (rows = Cin, taps flipped) so that
 *       dX = bts_conv_fwd(dY, wpack_T, Cin<->Cout swapped, pad' = dil*(K-1) - pad).
 *   bts_conv_n_tile(Cout) -> the N tile the engine uses for that many output channels. */
int bts_conv_n_tile(int Cout);
long long bts_conv_packed_floats(int n_rows, int k_channels, int KH, int KW);
/* flags bit 0 = chunk-major K order (K channels % 32 == 0): k-block = (32-channel chunk, tap) with the taps innermost, so
 * that consecutive k-blocks re-read the same pixels' cache lines (hits in L1 instead of nine L2 reads per element); pass the
 * same flags to bts_conv_fwd_ex / bts_conv_fwd_bnbwd. */
int bts_conv_pack_weights(const float *w, long long s_co, long long s_ci, long long s_kh, long long s_kw,
                          int Cout, int Cin, int KH, int KW, int transpose_flip, int flags, float *wpack,
                          void *stream);
int bts_conv_fwd(const float *x, long long x_pixel_stride, int B, int Hs, int Ws, int upsample2, int Cin,
                 int KH, int KW, int stride, int pad, int dil, const float *wpack, int Cout,
                 const float *pre_scale, const float *pre_shift, int pre_relu, float *out,
                 long long out_pixel_stride, int act, int precision, void *stream);

/* bts_conv_fwd that also returns the BatchNorm batch statistics of its output: stat_sum[co] += sum_p out[p,co],
 * stat_sumsq[co] += sum_p out[p,co]^2 (fp64, accumulated with atomics -> zero them first; Cout <= 256, act must be 0).  Replaces a separate
 * bts_bn_stats pass over the tensor just written (torchvision _DenseLayer: conv1 -> norm2, conv2 -> every later norm1). */
int bts_conv_fwd_stats(const float *x, long long x_pixel_stride, int B, int Hs, int Ws, int upsample2, int Cin,
                       int KH, int KW, int stride, int pad, int dil, const float *wpack, int Cout,
                       const float *pre_scale, const float *pre_shift, int pre_relu, float *out,
                       long long out_pixel_stride, int act, int precision, double *stat_sum, double *stat_sumsq,
                       void *stream);

/* General form of bts_conv_fwd (replaces cuDNN's strided-dgrad and grouped-convolution paths behind the ResNet / ResNeXt
 * encoders, reference pytorch/bts.py:282-296 via torchvision.models.resnet):
 *   source_mode 0 plain | 1 nearest x2 up-sample folded in | 2 ZERO-STUFFED x2 source with an explicit out_h x out_w output:
 *       with the transposed, tap-flipped packed operator, stride = 1 and pad' = dil*(K-1) - pad this is the input gradient
 *       of a STRIDE-2 convolution whose input was out_h x out_w (x = dY of that layer);
 *   kwin > 0 block-diagonal ("grouped") operator packed by bts_conv_pack_weights_grouped: output channels
 *       [nt*kwin, (nt+1)*kwin) read input channels [nt*kwin, (nt+1)*kwin) only; Cin == Cout == the layer width;
 *   stat_sum / stat_sumsq as in bts_conv_fwd_stats (or both NULL). */
int bts_conv_fwd_ex(const float *x, long long x_pixel_stride, int B, int Hs, int Ws, int source_mode, int out_h, int out_w,
                    int kwin, int Cin, int KH, int KW, int stride, int pad, int dil, const float *wpack, int Cout,
                    const float *pre_scale, const float *pre_shift, int pre_relu, float *out, long long out_pixel_stride,
                    int act, int precision, double *stat_sum, double *stat_sumsq, int flags, void *stream);
/* Staging of the activation tiles of bts_conv_fwd*: 0 = the producer warps load them (LDG + hi/lo split in registers),
 * 1 = TMA im2col loads (cp.async.bulk.tensor -> UTMALDG.4D.IM2COL; zero padding by out-of-bounds fill) land the raw tile in
 * shared memory as the A_hi operand and the producers only derive A_lo in place -- used for stride-1, non-up-sampled layers
 * whose K channels are a multiple of 32 and whose rows are 16-byte aligned, every other layer keeps mode 0 automatically.
 * (2, 3: bring-up variants.)  Process-wide setting. */
int bts_conv_set_tma(int mode);
int bts_conv_get_tma(void);
/* MMA issue loops of the three tensor-core kernels: 1 (default) = whole-warp loop with one elected lane, one barrier per stage,
 * incrementally advanced descriptors; 0 = the round-1 single-lane loops, kept as a bring-up fallback.  Process-wide. */
int bts_conv_set_issue_mode(int lean);
/* activation-producer groups of the conv engine (4 warps each): 0 / 4 = four groups without register prefetch wherever the
 * operand ring has >= 4 stages (default), 2 = always two groups with one k-block of register prefetch (round-1 layout). */
int bts_conv_set_producer_groups(int groups);
/* Tuning / bring-up switches of the narrow-output wgrad (csrc/wgrad2_tc.cu).  set_tma(0): the producers load the operands
 * from global memory (round-1 path) instead of the TMA landing ring; set_min_pixels(n): smallest map (input pixels) routed to
 * this kernel (default 12000, n < 0 restores it; tests pass 0 to reach it with small shapes). */
int bts_wgrad2_set_tma(int on);
int bts_wgrad2_set_min_pixels(long long n);
int bts_wgrad2_set_min_kblocks(int n);
int bts_wgrad2_set_pointwise(int on);        /* 1 (default): 1x1 layers with 64 < Cout <= 256 use this kernel too */       /* fewest 16-pixel k-blocks per split-K CTA (default 8; n < 1 restores) */

/* dgrad (or any act-free conv) whose epilogue also reduces the BatchNorm(+ReLU)-backward sums of the layer in front of the
 * conv: the tile written is g = dL/d[relu](bn(x_bn)); S1[c] += sum_p g*mask, S2[c] += sum_p g*mask*xhat (zero them first),
 * mask = [bn(x)>0] when relu else 1, xhat = (x-mean)*invstd; bn_st = [4][Cout] scale|shift|mean|invstd.  Replaces the
 * bts_bn_bwd_reduce pass over (x, g); follow with bts_bn_bwd_coef + bts_bn_bwd_apply. */
int bts_conv_fwd_bnbwd(const float *x, long long x_pixel_stride, int B, int Hs, int Ws, int source_mode, int out_h, int out_w,
                       int kwin, int Cin, int KH, int KW, int stride, int pad, int dil, const float *wpack, int Cout,
                       float *out, long long out_pixel_stride, int precision, const float *x_bn, long long x_bn_stride,
                       const float *bn_st, int relu, double *S1, double *S2, int flags, void *stream);
int bts_bn_bwd_coef(const double *S1, const double *S2, long long M, int C, const float *scale, const float *mean,
                    const float *invstd, float *coef, void *stream);
/* grouped 3x3 (ResNeXt: 32 groups of cpg channels): w is (width, cpg, KH, KW).  bts_conv_group_window -> the diagonal block
 * width kwin the packed operator uses (128 when width % 128 == 0 and 128 % cpg == 0; 0 = not supported). */
int bts_conv_group_window(int width, int cpg);
long long bts_conv_packed_floats_grouped(int width, int cpg, int KH, int KW);
int bts_conv_pack_weights_grouped(const float *w, long long s_co, long long s_ci, long long s_kh, long long s_kw, int width,
                                  int cpg, int KH, int KW, int transpose_flip, int flags, float *wpack, void *stream);
int bts_conv_wgrad_grouped_plan(int B, int Hout, int Wout, int width, int cpg, int KH, int KW, int *splitK_out,
                                long long *workspace_floats);
int bts_conv_wgrad_grouped(const float *x, long long x_pixel_stride, int B, int Hs, int Ws, int width, int cpg, int KH, int KW,
                           int stride, int pad, int dil, const float *dy, long long dy_pixel_stride, float *workspace,
                           int splitK, float *dw, long long s_co, long long s_ci, long long s_kh, long long s_kw,
                           int precision, void *stream);

/* wgrad on the same engine: dW[co,ci,tap] = sum_p dY[p,co] * pre(x[p (+) tap, ci]), MN-major tcgen05 operands,
 * split-K partials in `workspace` reduced deterministically into dw (strides in floats).
 *   bts_conv_wgrad_plan(...) -> splitK and the workspace size (floats) the call needs. */
int bts_conv_wgrad_plan(int B, int Hout, int Wout, int Cin, int Cout, int KH, int KW, int stride, int *splitK_out,
                        long long *workspace_floats);
int bts_conv_wgrad(const float *x, long long x_pixel_stride, int B, int Hs, int Ws, int upsample2, int Cin,
                   int KH, int KW, int stride, int pad, int dil, const float *pre_scale, const float *pre_shift,
                   int pre_relu, const float *dy, long long dy_pixel_stride, int Cout, float *workspace, int splitK,
                   float *dw, long long s_co, long long s_ci, long long s_kh, long long s_kw, int precision,
                   void *stream);

/* ---- single-output-channel convolutions (get_depth 3x3 32->1 + sigmoid, bts.py:193-194; reduc1x1 final 1x1 8->1 +
 * sigmoid, bts.py:94-96) as HBM-bound CUDA-core kernels.  x NHWC, C in {8,16,32,64,128}, K in {1,3}, stride 1,
 * pad K/2.  w: the (1,C,K,K) parameter addressed by its (ci,kh,kw) strides.  act: 0 none, 2 sigmoid.
 * Backward entry points take dy and, when the forward applied the sigmoid, the saved output `sig` (else NULL):
 * the effective gradient is dy*sig*(1-sig).  wgrad needs bts_conv_c1_workspace_floats(C,K) floats of workspace. */
int bts_conv_c1_workspace_floats(int C, int K);
int bts_conv_c1_fwd(const float *x, long long x_pixel_stride, int B, int H, int W, int C, int K, const float *w,
                    long long s_ci, long long s_kh, long long s_kw, int act, float *y, void *stream);
int bts_conv_c1_dgrad(const float *dy, const float *sig, int B, int H, int W, int C, int K, const float *w,
                      long long s_ci, long long s_kh, long long s_kw, float *dx, long long dx_pixel_stride,
                      void *stream);
int bts_conv_c1_wgrad(const float *x, long long x_pixel_stride, const float *dy, const float *sig, int B, int H,
                      int W, int C, int K, float *workspace, float *dw, long long s_ci, long long s_kh,
                      long long s_kw, void *stream);

/* ---- train-mode BatchNorm pieces for fused BN -> ReLU -> conv chains (torchvision _DenseLayer norm1/relu1/conv1/
 * norm2/relu2/conv2; decoder BNs bts.py:154-182).  The normalisation is applied inside the consumer conv
 * (bts_conv_fwd pre_scale/pre_shift/pre_relu); these entry points provide the per-channel reductions and the
 * backward pass over NHWC tensors (explicit pixel strides -> channel slices of slabs work in place).
 *   bts_bn_stats            : sum / sum of squares per channel (fp64 accumulators, zeroed by the call)
 *   bts_bn_finalize         : -> scale = gamma*invstd, shift = beta - mean*scale, mean, invstd (+ running-stat update,
 *                             momentum m, unbiased variance; running_* may be NULL)
 *   bts_bn_fold             : the same four vectors from frozen running statistics (eval mode)
 *   bts_bn_relu_bwd_reduce  : S1 = sum g*[y>0], S2 = sum g*[y>0]*xhat (y = x*scale+shift) and the fp32 backward
 *                             coefficients coef[0:C] = k0, coef[C:2C] = k1 (dx = [y>0]*scale*g + k1*x + k0)
 *   bts_bn_relu_bwd_apply   : out (=|+=) [y>0]*scale*g + k1*x + k0   (coef == NULL: frozen statistics, k0 = k1 = 0) */
int bts_bn_stats(const float *x, long long x_pixel_stride, long long M, int C, double *sum, double *sumsq, void *stream);
int bts_bn_finalize(const double *sum, const double *sumsq, long long N, int C, const float *gamma, const float *beta,
                    float eps, float momentum, float *running_mean, float *running_var, float *scale, float *shift,
                    float *mean, float *invstd, void *stream);
int bts_bn_finalize_track(const double *sum, const double *sumsq, long long N, int C, const float *gamma, const float *beta,
                          float eps, float momentum, float *running_mean, float *running_var, long long *num_batches_tracked,
                          float *scale, float *shift, float *mean, float *invstd, void *stream);   /* + num_batches_tracked += 1 */
int bts_bn_fold(int C, const float *gamma, const float *beta, float eps, const float *running_mean,
                const float *running_var, float *scale, float *shift, float *mean, float *invstd, void *stream);
int bts_bn_relu_bwd_reduce(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride,
                           long long M, int C, const float *scale, const float *shift, const float *mean,
                           const float *invstd, double *S1, double *S2, float *coef, void *stream);
int bts_bn_relu_bwd_apply(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride,
                          long long M, int C, const float *scale, const float *shift, const float *coef, float *out,
                          long long out_pixel_stride, int accumulate, void *stream);

/* generalised forms with an explicit `relu` flag (relu=0: plain BatchNorm, as the decoder's bn5/bn4/bn4_2/bn3/bn2 which
 * feed a concat, bts.py:200-246; relu=2: ReLU6, mask 0 < y < 6 strictly, the MobileNetV2 BN + ReLU6); the *_relu_* entry
 * points above are these with relu=1. */
int bts_bn_bwd_reduce(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride, long long M,
                      int C, const float *scale, const float *shift, const float *mean, const float *invstd, int relu,
                      double *S1, double *S2, float *coef, void *stream);
int bts_bn_bwd_apply(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride, long long M,
                     int C, const float *scale, const float *shift, const float *coef, int relu, float *out,
                     long long out_pixel_stride, int accumulate, void *stream);

/* One-pass BatchNorm+ReLU backward into a concat gradient slab (the dense-block fan-out, torchvision densenet.py
 * _DenseLayer / _DenseBlock backward): out += [y>0]*scale*g in the same pass that reduces S1, S2; the per-channel affine
 * remainder k1*x + k0 is added into K0/K1 (fp64, K0 == K1 == NULL for frozen statistics) and applied later, once per
 * channel slice, by bts_bn_bwd_correct (out += K1*x + K0) -- before that slice's gradient is consumed. */
int bts_bn_relu_bwd_fused(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride, long long M,
                          int C, const float *scale, const float *shift, const float *mean, const float *invstd,
                          double *S1, double *S2, float *out, long long out_pixel_stride, double *K0, double *K1,
                          void *stream);
int bts_bn_bwd_correct(const float *x, long long x_pixel_stride, long long M, int C, const double *K0, const double *K1,
                       float *out, long long out_pixel_stride, void *stream);

/* ---- streaming NHWC glue kernels of the decoder / encoder transitions (csrc/elem.cu) ---------------------------
 * All take explicit pixel strides (floats) so channel slices of wider slabs are read / written in place.
 *   bts_bn_apply       out = x*scale + shift [, ReLU]   -- BatchNorm2d forward given (scale, shift) from bts_bn_finalize /
 *                      bts_bn_fold (decoder BNs bts.py:154-182; torchvision norm0 / norm5); relu: 0 none, 1 ReLU,
 *                      2 ReLU6 = clamp(., 0, 6) (MobileNetV2 Conv2dNormActivation)
 *   bts_elu_bwd        out = gy * (y > 0 ? 1 : y + 1)   -- backward of nn.ELU() through its saved OUTPUT y (bts.py:72,79,...)
 *   bts_upsample2_sum  out[b,y,x,:] = sum of g[b,2y..2y+1,2x..2x+1,:]  -- backward of F.interpolate(scale_factor=2,
 *                      mode='nearest') (bts.py:77); relu_src != NULL additionally gates by relu_src > 0 (torch.nn.ReLU in
 *                      front of upconv5, bts.py:198)
 *   bts_copy_channels  dst (=|+=) src over M pixels x C channels -- torch.cat along channels / its backward (bts.py:201-260)
 *   bts_zero_channels  dst[:, c0:c1] = 0                -- alignment padding channels of concat3 (225) / concat2 (161)
 *   bts_avgpool2_fwd/bwd  2x2 stride-2 average pooling of the DenseNet transitions (torchvision densenet.py `pool`) */
int bts_bn_apply(const float *x, long long x_pixel_stride, long long M, int C, const float *scale, const float *shift,
                 int relu, float *out, long long out_pixel_stride, void *stream);
int bts_elu_bwd(const float *gy, long long gy_pixel_stride, const float *y, long long y_pixel_stride, long long M, int C,
                float *out, long long out_pixel_stride, void *stream);
int bts_upsample2_sum(const float *g, long long g_pixel_stride, int B, int H, int W, int C, const float *relu_src,
                      long long relu_pixel_stride, float *out, long long out_pixel_stride, void *stream);
int bts_copy_channels(const float *src, long long src_pixel_stride, long long M, int C, float *dst,
                      long long dst_pixel_stride, int accumulate, void *stream);
int bts_zero_channels(float *dst, long long dst_pixel_stride, long long M, int c0, int c1, void *stream);
int bts_avgpool2_fwd(const float *x, long long x_pixel_stride, int B, int Hout, int Wout, int C, float *out,
                     long long out_pixel_stride, void *stream);
int bts_avgpool2_bwd(const float *g, long long g_pixel_stride, int B, int Hout, int Wout, int C, float *gx,
                     long long gx_pixel_stride, void *stream);

/* ---- weight gradient of the narrow 1x1 convolutions of the reduction heads (bts.py:83-108) on CUDA cores (csrc/pointwise.cu):
 * dW[co,ci] = sum_p dY[p,co]*x[p,ci] for Cin in {8,16,32,64}, Cout <= 32 -- HBM-bound, deterministic two-pass reduction.
 * workspace: bts_conv_pw_wgrad_workspace_floats(Cin, Cout) floats; dw addressed by its (co, ci) strides in floats. */
/* Forward / dgrad of the same narrow 1x1 layers on CUDA cores (HBM-bound): out[p, co] = act(sum_ci x[p, ci] * W[co, ci]),
 * Cin in {8,16,32,64}, Cout <= 64; (s_out, s_in) are the element strides of W[out, in] -- for dgrad pass the conv weight's
 * (s_ci, s_co) and dY as x.  act: 0 none, 1 ELU, 2 sigmoid.  Replaces the tensor engine for reduc1x1/2x2/4x4 (bts.py:83-108). */
int bts_conv_pw_fwd_eligible(int Cin, int Cout);
int bts_conv_pw_fwd(const float *x, long long x_pixel_stride, long long M, int Cin, const float *w, long long s_out,
                    long long s_in, int Cout, int act, float *out, long long out_pixel_stride, void *stream);
int bts_conv_pw_wgrad_eligible(int Cin, int Cout);
long long bts_conv_pw_wgrad_workspace_floats(int Cin, int Cout);
int bts_conv_pw_wgrad(const float *x, long long x_pixel_stride, const float *dy, long long dy_pixel_stride, long long M,
                      int Cin, int Cout, float *workspace, float *dw, long long s_co, long long s_ci, void *stream);

/* ResNet / ResNeXt encoder glue (torchvision.models.resnet behind reference pytorch/bts.py:282-296):
 *   bts_bn_add_relu   out = max(x*scale + shift + res, 0)            Bottleneck tail  relu(bn3(conv3(.)) + identity)
 *   bts_relu_bwd      out = gy * (y > 0)                             its backward (through the saved output y)
 *   bts_maxpool3s2_*  3x3 / stride 2 / pad 1 max-pool (the encoder stems' pool0 / maxpool), NHWC; forward records the
 *                     winning window position (uint8 per OUTPUT element, dense [B,Ho,Wo,C]) -> deterministic gather backward */
int bts_bn_add_relu(const float *x, long long x_pixel_stride, long long M, int C, const float *scale, const float *shift,
                    const float *res, long long res_pixel_stride, float *out, long long out_pixel_stride, void *stream);
/*   bts_bn_add        out = x*scale + shift + res                    MobileNetV2 InvertedResidual tail  x + bn3(conv3(.)) */
int bts_bn_add(const float *x, long long x_pixel_stride, long long M, int C, const float *scale, const float *shift,
               const float *res, long long res_pixel_stride, float *out, long long out_pixel_stride, void *stream);
int bts_relu_bwd(const float *gy, long long gy_pixel_stride, const float *y, long long y_pixel_stride, long long M, int C,
                 float *out, long long out_pixel_stride, void *stream);
int bts_maxpool3s2_fwd(const float *x, long long x_pixel_stride, int B, int H, int W, int C, float *out,
                       long long out_pixel_stride, unsigned char *argmax, void *stream);
int bts_maxpool3s2_bwd(const float *g, long long g_pixel_stride, const unsigned char *argmax, int B, int H, int W, int C,
                       float *gx, long long gx_pixel_stride, void *stream);

/* ---- depthwise 3x3 convolution, padding 1, stride 1 or 2, of the MobileNetV2 inverted residuals (torchvision
 * mobilenetv2.py behind reference pytorch/bts.py:298-300), csrc/dwconv.cu.  fp32 NHWC with explicit pixel strides
 * (multiples of 4, 16-byte aligned bases), C % 4 == 0; w = the contiguous (C,1,3,3) weight, read on every call.
 * Hout = (H-1)/stride + 1, likewise Wout.
 *   bts_dw_fwd   y = dw(act_in(x)); act_in(x) = clamp(x*pre_scale + pre_shift, 0, 6) when pre_* != NULL, else x
 *                (out-of-bounds taps are 0 after the activation).  Epilogue: sums != NULL -> sums[0][c] = sum y,
 *                sums[1][c] = sum y^2 (fp64 [2][C], deterministic two-pass reduction through `partials`);
 *                post_* != NULL -> y = clamp(y*post_scale + post_shift, 0, 6) (a folded eval-mode BN + ReLU6).
 *   bts_dw_dgrad gx (B,H,W,C) = d/dx of the plain depthwise conv given g (B,Hout,Wout,C); gather form, no atomics.
 *   bts_dw_wgrad dw[c*s_c + ky*s_kh + kx*s_kw] = sum_p g[p,c] * act_in(x)[p*stride + (ky-1, kx-1), c]; deterministic
 *                two-pass reduction through `partials`.
 * partials: bts_dw_partials(B, Hout, Wout, C, wgrad) doubles (wgrad = 0 for the forward statistics, 1 for bts_dw_wgrad). */
long long bts_dw_partials(int B, int Hout, int Wout, int C, int wgrad);
int bts_dw_fwd(const float *x, long long x_pixel_stride, int B, int H, int W, int C, int stride, const float *w,
               const float *pre_scale, const float *pre_shift, const float *post_scale, const float *post_shift, float *y,
               long long y_pixel_stride, double *partials, double *sums, void *stream);
int bts_dw_dgrad(const float *g, long long g_pixel_stride, int B, int H, int W, int C, int stride, const float *w, float *gx,
                 long long gx_pixel_stride, void *stream);
int bts_dw_wgrad(const float *x, long long x_pixel_stride, int B, int H, int W, int C, int stride, const float *pre_scale,
                 const float *pre_shift, const float *g, long long g_pixel_stride, double *partials, float *dw, long long s_c,
                 long long s_kh, long long s_kw, void *stream);

/* ---- optimizer step of the training loop (reference pytorch/bts_main.py:371-373 torch.optim.AdamW, two groups, eps 1e-3;
 * :456-460 poly LR) as ONE multi-tensor kernel, csrc/optim.cu.  ptrs: device int64 [4n] = param | grad | exp_avg | exp_avg_sq
 * addresses; numel: device int64 [n]; group: device int32 [n] -> index into the n_groups (<= 8) scalar sets;
 * chunk_tensor / chunk_off: device tables cutting every tensor into bts_adamw_chunk()-element pieces;
 * scalars: HOST float [7*n_groups], seven blocks of n_groups: 1-lr*wd | 1-beta1 | beta2 | 1-beta2 | sqrt(1-beta2^t) | eps |
 * -lr/(1-beta1^t).  Element arithmetic follows torch's _multi_tensor_adam operation by operation. */
int bts_adamw_chunk(void);
int bts_adamw_multi(const long long *ptrs, const long long *numel, const int *group, int n, const int *chunk_tensor,
                    const long long *chunk_off, int n_chunks, const float *scalars, int n_groups, void *stream);
/* every packed conv operator of a model in one launch: descs = device array of n 96-byte descriptors
 * {w, wpack, s_co, s_ci, s_kh, s_kw, start (int64 each), Cout, Cin, KH, KW, transpose_flip, n_tile, n_tiles, kwin, cpg, pad
 * (int32 each)}, start = prefix sum of packed_floats/2; total = their sum. */
int bts_conv_pack_weights_multi(const void *descs, int n, long long total, void *stream);

/* ---- data formats either side of the hot path (SURVEY 8f ranks 2-3), csrc/io.cu
 * bts_input_prep: the reference loader's per-sample transform after decoding (pytorch/bts_dataloader.py:128-140,202-235,
 *   244-249), fused: uint8 HWC frames [B,Hs,Ws,3] (+ optional uint16 depth [B,Hs,Ws]) -> crop -> flip -> gamma/brightness/
 *   colour augmentation + clip -> ImageNet normalisation -> fp32 NHWC image [B,H,W,(stride)] and depth/depth_div [B,H,W].
 *   params: device float [B][9] = y0, x0, flip, augment, gamma, brightness, colour r,g,b (the random draws stay on the host).
 * bts_eval_errors: online-eval clamps + masks + the nine metrics of one image (pytorch/bts_main.py:144-165,275-296):
 *   metrics_out[10] = silog, abs_rel, log10, rms, sq_rel, log_rms, d1, d2, d3, n_valid; crop rows [y0,y1) cols [x0,x1);
 *   workspace = 10 doubles.
 * bts_depth_to_u16: the 16-bit PNG wire format of pytorch/bts_test.py:179-185, uint16(depth * scale). */
int bts_input_prep(const unsigned char *img_u8, int Hs, int Ws, const unsigned short *depth_u16, float depth_div,
                   const float *params, int B, int H, int W, float *image_out, long long out_pixel_stride, float *depth_out,
                   void *stream);
int bts_eval_errors(const float *pred, const float *gt, int H, int W, float min_depth, float max_depth, int crop_y0,
                    int crop_y1, int crop_x0, int crop_x1, double *workspace, float *metrics_out, void *stream);
int bts_depth_to_u16(const float *depth, float scale, long long n, unsigned short *out, void *stream);

/* zero n floats on the stream (grad_focal output of the TF-op surface, integration/tf_op/bts_lpg_tf_op.cc) */
int bts_fill_zero_f32(float *p, long long n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BTS_B200_H_ */
