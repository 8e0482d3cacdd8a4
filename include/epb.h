/*
 * epb.h -- C ABI of libepb.so, the B200 (sm_100a) implementation of the
 * EpipolarPose training-loop hot path.
 *
 * The reference (mkocabas/EpipolarPose) has no FFI layer: its extension points
 * are Python call sites that reach cuDNN / ATen / numpy / OpenCV.  Each entry
 * point below replaces one of those library call sites; the comment on each
 * names the reference file:line whose arithmetic it reproduces.  The Python
 * mirror of the reference interface (epipolarpose_b200/lib/...) binds these
 * symbols with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *     the caller owns all memory; the library never allocates caller-visible
 *     memory and never synchronises the device;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - activations are NHWC float32 ("pixel rows"), row pitch == channel count;
 *     packed weights are [Cout][T][Cin] float32 (T = taps);
 *   - return value: 0 on success, negative EPB_E* otherwise; the message is
 *     available from epb_last_error() (thread local);
 *   - alignment: all float buffers 16-byte aligned, channel counts that feed
 *     the tensor-core path are multiples of 32.
 */
#ifndef EPB_H_
#define EPB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EPB_OK 0
#define EPB_EINVAL (-1)   /* bad argument / unsupported shape            */
#define EPB_ECUDA (-2)    /* a CUDA runtime / driver call failed          */
#define EPB_ENOGPU (-3)   /* no sm_100 device present                     */

#define EPB_MAX_TAPS 64

typedef void* epb_stream_t;

int epb_version(void);
const char* epb_last_error(void);
/* 0 if a compute-capability 10.x device is usable, EPB_ENOGPU otherwise */
int epb_device_check(void);

/* ------------------------------------------------------------------------
 * Convolution family (cuDNN call sites behind nn.Conv2d / nn.ConvTranspose2d:
 * lib/models/pose3d_resnet.py:12-15,55-60,99,116-122,132,171-178).
 *
 * One "tap-list implicit GEMM" geometry expresses forward convs, transposed
 * convs (one call per output phase), and both of their data gradients:
 *
 *   out[n, i*os+ph, j*os+pw, co] (+)= sum_t sum_ci
 *        f(in[n, i*is+dh[t], j*is+dw[t], ci]) * w[co][wt[t]][ci]   (+ bias[co])
 *
 * for i<Hp, j<Wp (the phase grid), out-of-range input pixels contribute 0.
 * f is identity, or the fused BatchNorm+ReLU of the producing layer
 * (relu(in*in_scale[ci] + in_shift[ci])) when in_scale != NULL.
 * ---------------------------------------------------------------------- */
typedef struct {
  int N, Hi, Wi, Cin;        /* input tensor  [N,Hi,Wi,Cin]                 */
  int Ho, Wo, Cout;          /* output tensor [N,Ho,Wo,Cout]                */
  int Hp, Wp;                /* phase grid (== Ho,Wo when os == 1)          */
  int os, ph, pw;            /* output stride and phase offset              */
  int is;                    /* input stride                                */
  int T;                     /* number of taps                              */
  int dh[EPB_MAX_TAPS];      /* input row offset per tap                    */
  int dw[EPB_MAX_TAPS];      /* input col offset per tap                    */
  int wt[EPB_MAX_TAPS];      /* index of the tap inside the packed weight   */
  int Tw;                    /* taps in the packed weight (row = Tw*Cin)    */
  int in_relu;               /* 1: relu after the input affine              */
  int accumulate;            /* 1: out += result (beta = 1)                 */
  int precision;             /* 0: fp32 SIMT, 1: tf32 (1 pass), 3: tf32x3   */
} epb_conv_geom;

/* out = conv(in) ; optional fused input BN+ReLU, bias, per-channel
 * statistics of the output (stats[0..Cout) += sum, stats[Cout..2Cout) +=
 * sum of squares, float64, caller zeroes).  Any of in_scale/in_shift/bias/
 * stats may be NULL. */
int epb_conv_fprop(const epb_conv_geom* g, const float* in, const float* w,
                   const float* in_scale, const float* in_shift,
                   const float* bias, float* out, double* stats,
                   epb_stream_t stream);

/* dw[co][wt[t]][ci] += sum_{n,i,j} dout[n,i*os+ph,j*os+pw,co] * f(in[...tap t...][ci])
 * (cuDNN wgrad).  dw must be zeroed by the caller before the first phase. */
int epb_conv_wgrad(const epb_conv_geom* g, const float* in, const float* dout,
                   const float* in_scale, const float* in_shift, float* dw,
                   epb_stream_t stream);

/* Weight layout conversion between the reference's state_dict layouts
 * (Conv2d [O][I][kh][kw], ConvTranspose2d [I][O][kh][kw]) and the packed GEMM
 * operand.  src is [A][B][kh*kw]; packed is [X][kh*kw][Ypad] with
 * (X,Y) = (A,B) when swap == 0 and (B,A) when swap == 1, zero padded to Ypad.
 *   Conv2d fprop: swap 0 (X=O,Y=I)      Conv2d dgrad:   swap 1 (X=I,Y=O)
 *   Deconv fprop: swap 1 (X=O,Y=I)      Deconv dgrad:   swap 0 (X=I,Y=O)
 * No spatial flip: the tap tables in epb_conv_geom index taps by the original
 * (r,s).  unpack != 0 runs the inverse map (packed gradient -> state_dict
 * layout; `src` is then the packed tensor). */
int epb_pack_weight(const float* src, float* dst, int A, int B, int kh, int kw,
                    int swap, int Ypad, int unpack, epb_stream_t stream);

/* The same conversion for MANY tensors in one launch (all layers of the network before
 * a forward pass; all weight gradients after a backward pass).  `jobs` is a DEVICE array
 * of njobs descriptors ordered by first_block; job j owns the blocks
 * [first_block_j, first_block_{j+1}) of 1024 packed elements each, total_blocks in all.
 * x_pitch is the distance in floats between consecutive X rows of the packed tensor
 * (kh*kw*Ypad when dense; larger when the packed tensor is a slice of a wider matrix,
 * as for the im2col form of the stem). */
typedef struct epb_pack_job {
  const float* src;
  float* dst;
  int A, B, T, swap, Ypad, unpack, x_pitch, reserved;
  long long first_block;
  long long reserved2;
} epb_pack_job;
int epb_pack_weight_batch(const epb_pack_job* jobs, int njobs, long long total_blocks,
                          epb_stream_t stream);

/* Patch matrix of a small-Cin convolution (the 7x7 stem, pose3d_resnet.py:99):
 * col[m][(r*kw+s)*C + c] = in[n, oh*stride-pad+r, ow*stride-pad+s, c] (0 outside
 * the image and for columns >= kh*kw*C), row pitch Kpad floats, so the layer
 * runs as a 1x1 conv on the tensor-core path.  `in` is NHWC with `pitch` floats
 * per pixel. */
int epb_im2col(const float* in, float* col, int N, int Hi, int Wi, int pitch,
               int C, int kh, int kw, int stride, int pad, int Ho, int Wo,
               int Kpad, epb_stream_t stream);

/* NCHW <-> NHWC float32 with channel padding (module boundary only:
 * pose3d_resnet.py:185 takes NCHW images, returns NCHW heatmaps). */
int epb_nchw_to_nhwc(const float* src, float* dst, int N, int C, int H, int W,
                     int Cpad, epb_stream_t stream);
int epb_nhwc_to_nchw(const float* src, float* dst, int N, int C, int H, int W,
                     int Cpad, epb_stream_t stream);

/* ------------------------------------------------------------------------
 * BatchNorm2d(momentum=0.1, eps=1e-5) training semantics (cuDNN BN call
 * sites: pose3d_resnet.py:24,56-63,101,134,179), ReLU, residual add, MaxPool.
 * ---------------------------------------------------------------------- */
/* per-channel sum / sum-of-squares of x[M][C] into stats[2C] (float64, +=) */
int epb_channel_stats(const float* x, int64_t M, int C, double* stats,
                      epb_stream_t stream);
/* stats -> (scale, shift, mean, invstd) and running-stat update (biased var
 * for normalisation, unbiased for running_var; pose3d_resnet.py:8). */
int epb_bn_finalize(const double* stats, int64_t M, int C, const float* gamma,
                    const float* beta, float eps, float momentum,
                    float* running_mean, float* running_var, float* scale,
                    float* shift, float* mean, float* invstd,
                    epb_stream_t stream);
/* eval mode: scale/shift from running statistics */
int epb_bn_eval_affine(int C, const float* gamma, const float* beta,
                       const float* running_mean, const float* running_var,
                       float eps, float* scale, float* shift,
                       epb_stream_t stream);
/* y = act(x*scale+shift [+ r*rscale+rshift | + r]) ; r may be NULL, rscale
 * NULL means identity residual (pose3d_resnet.py:44-45,85-86). */
int epb_bn_act(const float* x, const float* scale, const float* shift,
               const float* r, const float* rscale, const float* rshift,
               int relu, float* y, int64_t M, int C, epb_stream_t stream);
/* stem: y = maxpool3x3s2p1(relu(x*scale+shift)) (pose3d_resnet.py:187-189);
 * also records the argmax position (0..8) for the backward. */
int epb_bn_relu_maxpool(const float* x, const float* scale, const float* shift,
                        float* y, uint8_t* argidx, int N, int H, int W, int C,
                        epb_stream_t stream);
int epb_maxpool_bwd(const float* dy, const uint8_t* argidx, float* dx, int N,
                    int H, int W, int C, epb_stream_t stream);
/* BatchNorm(+ReLU) backward, two passes.
 *   g = dy * [mask]   where mask = (y_out > 0) if y_out != NULL, else
 *                     (x*scale+shift > 0) if relu, else 1
 * reduce: sums[0..C) += sum g ; sums[C..2C) += sum g * xhat   (float64)
 * apply : dx = gamma*invstd*(g - sum_g/M - xhat*sum_gx/M); dgamma, dbeta out */
int epb_bn_bwd_reduce(const float* dy, const float* x, const float* y_out,
                      const float* scale, const float* shift, const float* mean,
                      const float* invstd, int relu, int64_t M, int C,
                      double* sums, epb_stream_t stream);
int epb_bn_bwd_apply(const float* dy, const float* x, const float* y_out,
                     const float* scale, const float* shift, const float* mean,
                     const float* invstd, const float* gamma, int relu,
                     const double* sums, int64_t M, int C, float* dx,
                     float* dgamma, float* dbeta, epb_stream_t stream);
/* dx = a + b * [mask_src > 0] (residual gradient merge); mask_src may be NULL */
int epb_add_masked(const float* a, const float* b, const float* mask_src,
                   float* dx, int64_t n, epb_stream_t stream);
/* VOLUME=False head: y[n][c] = mean over HW (pose3d_resnet.py:125,208) */
int epb_avgpool(const float* x, float* y, int N, int HW, int C,
                epb_stream_t stream);
int epb_avgpool_bwd(const float* dy, float* dx, int N, int HW, int C,
                    int accumulate, epb_stream_t stream);
/* column sums of x[M][C] (bias gradients): out[c] = sum_m x[m][c] */
int epb_colsum(const float* x, int64_t M, int C, float* out,
               epb_stream_t stream);

/* ------------------------------------------------------------------------
 * Split-fp16 operand family ("f16x3"): the same conv / BatchNorm call sites as above
 * (pose3d_resnet.py:12-15,24,55-63,99,116-122,171-179), with every GEMM operand
 * materialised ONCE as two fp16 planes and fed to tcgen05 kind::f16 by TMA.
 *
 * A split tensor holds x as   x * s = hi + lo   (hi = fp16(x*s), lo = fp16(x*s - hi),
 * s a power of two), planes[0] = hi, planes[1] = lo, each [rows][C] fp16 (raw bits,
 * epb_half), C % 8 == 0; `sc` is a DEVICE float[2] = {s, 1/s}.  Three tensor passes
 * (lo*hi + hi*lo + hi*hi, fp32 accumulation) reproduce the fp32 product to ~2^-22.
 *
 * Single-pass layout ("f16"): `int planes` = 1 on the calls below selects [1][rows][C], the
 * hi plane alone (x*s ~= hi: 10 explicit mantissa bits, the TF32 operand class).  Producers
 * then write neither the lo plane nor its address range (the buffer may end after the hi
 * plane), readers read hi only, and the GEMMs issue one kind::f16 pass (hi*hi) per k-step.
 * Scales and bounds are those of the two-plane form.  planes = 2 is the layout above; the
 * plane count is a launch argument (the GEMMs build their TMA tensor maps from it).
 * ---------------------------------------------------------------------- */
typedef uint16_t epb_half;

/* Power-of-two scale of a post-activation split tensor from STATISTICS only (no pass over the
 * data): with stats[2C] the float64 (sum, sum of squares) of a conv output over M rows,
 *   |x*scale_c + shift_c| <= |scale_c*mean_c + shift_c| + |scale_c| * sqrt(M * var_c)
 * (no element lies further than sqrt(M) standard deviations from its mean), maximised over
 * the channels; a second group (the downsample BatchNorm of a residual block) and the bound
 * of a split residual (res_sc[2]) add.  sc[4] = {s, 1/s, bound, 0}, s the largest power of
 * two with s*bound <= 2^15, so the fp16 planes can neither overflow nor saturate. */
int epb_act_scale(const double* stats, const float* scale, const float* shift, int64_t M, int C,
                  const double* stats2, const float* scale2, const float* shift2,
                  const float* res_sc, float* sc, epb_stream_t stream);
/* epb_bn_finalize of one layer + epb_act_scale of its post-activation tensor in ONE launch
 * (train() forward of the split path: one single-CTA kernel per BatchNorm instead of two).
 * Group 1 = (stats, the scale / shift this call produces); group 2 / res_sc as epb_act_scale. */
int epb_bn_finalize_scale(const double* stats, int64_t M, int C, const float* gamma,
                          const float* beta, float eps, float momentum, float* running_mean,
                          float* running_var, float* scale, float* shift, float* mean,
                          float* invstd, const double* stats2, const float* scale2,
                          const float* shift2, const float* res_sc, float* sc, epb_stream_t stream);
/* y_split = act(x*scale+shift [+ residual]).  The residual is either fp32 rows `r`
 * (with optional affine rscale/rshift: the downsample BatchNorm) or a split tensor
 * `r_split` / `r_sc` (the identity path: the previous block's output), or absent. */
int epb_bn_act_split(const float* x, const float* scale, const float* shift,
                     const float* r, const float* rscale, const float* rshift,
                     const epb_half* r_split, const float* r_sc, int relu,
                     int64_t M, int C, epb_half* y, const float* y_sc,
                     uint8_t* mask_bits, int planes, epb_stream_t stream);
/* mask_bits (optional, [M*C/8] bytes): bit k of byte i = (pre-ReLU value of element 8*i+k > 0),
 * the ReLU mask the BatchNorm backward of the block reads (epb_bn_bwd_split). */
/* stem: maxpool3x3s2p1(relu(x*scale+shift)) -> split tensor + argmax slot (0..8) */
int epb_bn_relu_maxpool_split(const float* x, const float* scale, const float* shift,
                              epb_half* y, const float* y_sc, uint8_t* argidx, int N,
                              int H, int W, int C, int planes, epb_stream_t stream);
/* patch matrix of the 7x7 stem straight from the NCHW image (pose3d_resnet.py:99,185):
 * col[m][(r*kw+s)*C + c] = img[n][c][oh*stride-pad+r][ow*stride-pad+s], zero padded to
 * Kpad (% 64 == 0) columns, as a split tensor [planes][N*Ho*Wo][Kpad]. */
int epb_im2col_split(const float* img_nchw, epb_half* col, const float* col_sc, int N,
                     int C, int Hi, int Wi, int kh, int kw, int stride, int pad, int Ho,
                     int Wo, int Kpad, int planes, epb_stream_t stream);
/* fp32 tensors -> split tensors with a per-tensor power-of-two scale chosen from the
 * tensor's max |x| (largest scaled magnitude in [2^13, 2^14)); job j: src[n] ->
 * dst[planes][n], sc[2] written.  Blocks of 2048 elements, jobs ordered by first_block.
 * amax_ws: njobs uint32 of DEVICE scratch (zeroed by the call). */
typedef struct epb_split_job {
  const float* src;
  epb_half* dst;
  float* sc;
  long long n;
  long long first_block;
} epb_split_job;
int epb_split16_batch(const epb_split_job* jobs, int njobs, long long total_blocks,
                      uint32_t* amax_ws, int planes, epb_stream_t stream);

/* one tensor (n % 4 == 0), pointers as arguments: for tensors whose address is only known at
 * call time (the logit gradient autograd hands to the network's backward).  amax_ws: one
 * uint32 of DEVICE scratch. */
int epb_split16(const float* src, long long n, epb_half* dst, float* sc, uint32_t* amax_ws,
                int planes, epb_stream_t stream);

/* epb_conv_fprop on split operands: in [planes][N,Hi,Wi,Cin], w [planes][Cout][Tw*Cin] (the packed
 * operand of epb_pack_weight, split).  Cin % 64 == 0, Cout % 4 == 0.  CTA pairs
 * (tcgen05 cta_group::2, M = 256), A and B tiles by TMA (5-D / 3-D tensor maps; the
 * zero padding of the convolution is the TMA out-of-bounds fill), fp32 accumulators
 * in TMEM; out = acc / (s_in * s_w) (+ bias), optional accumulate / statistics as
 * epb_conv_fprop.  g->precision, g->in_relu are ignored (operands are post-activation).
 * planes 2: three kind::f16 passes; planes 1: one pass over the hi planes. */
int epb_conv16_fprop(const epb_conv_geom* g, const epb_half* in, const float* in_sc,
                     const epb_half* w, const float* w_sc, const float* bias,
                     float* out, double* stats, int planes, epb_stream_t stream);
/* epb_conv_wgrad on split operands (in as above, dout [planes][N,Ho,Wo,Cout]); both operands
 * MN-major by TMA, reduction over pixel tiles split across clusters and summed in a FIXED
 * order from `ws` (deterministic): dw[co][wt[t]][ci] += sum.  ws: >= ws_floats floats of
 * scratch (the call uses as many split partials as fit). */
int epb_conv16_wgrad(const epb_conv_geom* g, const epb_half* in, const float* in_sc,
                     const epb_half* dout, const float* dout_sc, float* dw, float* ws,
                     long long ws_floats, int planes, epb_stream_t stream);

/* BatchNorm(+ReLU) backward for the split path.  mask = (mask_hi > 0) when mask_hi != NULL
 * (hi plane of the block output, of either layout: only the hi plane is read), else (x*scale+shift > 0) if relu, else 1.
 * reduce: sums as epb_bn_bwd_reduce; maxes[0..C) = max |g|, maxes[C..2C) = max |xhat|
 *         (float, caller zeroes; used to bound |dz| for the scale of the split output).
 *         Two launches: per-CTA partials, then a fixed-order combine (deterministic).
 * apply : dz_split = gamma*invstd*(g - sum_g/M - xhat*sum_gx/M) with the power-of-two
 *         scale derived from the bound written to dz_sc[2]; if dy_masked != NULL the
 *         masked gradient g is also written there (may alias dy: the identity path of
 *         the residual block then accumulates into it). */
int epb_bn_bwd_reduce_mx(const float* dy, const float* x, const epb_half* mask_hi,
                         const float* scale, const float* shift, const float* mean,
                         const float* invstd, int relu, int64_t M, int C, double* sums,
                         float* maxes, epb_stream_t stream);
int epb_bn_bwd_apply_split(const float* dy, const float* x, const epb_half* mask_hi,
                           const float* scale, const float* shift, const float* mean,
                           const float* invstd, const float* gamma, int relu,
                           const double* sums, const float* maxes, int64_t M, int C,
                           epb_half* dz, float* dz_sc, float* dy_masked, float* dgamma,
                           float* dbeta, int planes, epb_stream_t stream);
/* Both passes in one call (what the engine uses): per-CTA partial reductions, a fixed-order
 * combine (no atomics: dgamma / dbeta / the scale of dz are run-to-run identical), apply.
 * Outputs as epb_bn_bwd_apply_split; the sums / maxes live in internal scratch of the stream.
 * mask_bits (instead of mask_hi; C % 8 == 0): the bit mask epb_bn_act_split wrote for the block
 * output, 1/8 byte per element instead of the 2-byte hi plane in both passes. */
int epb_bn_bwd_split(const float* dy, const float* x, const epb_half* mask_hi,
                     const uint8_t* mask_bits, const float* scale, const float* shift, const float* mean, const float* invstd,
                     const float* gamma, int relu, int64_t M, int C, epb_half* dz, float* dz_sc,
                     float* dy_masked, float* dgamma, float* dbeta, int planes, epb_stream_t stream);
/* VOLUME=False head on a split tensor: y[n][c] = mean over HW of x (fp32 out) */
int epb_avgpool_split(const epb_half* x, const float* x_sc, float* y, int N, int HW, int C,
                      int planes, epb_stream_t stream);

/* ------------------------------------------------------------------------
 * Soft-argmax (ATen softmax + 9 reductions: lib/core/integral_loss.py:49-86)
 * logits: volume per (n,j) of D*H*W float32.  layout 0 = NCHW contiguous
 * ([N][J*D][H][W]); layout 1 = NHWC ([N][H][W][J*D]).
 * coords: [N][J*3] float32 (x,y,z interleaved, in [-0.5,0.5)).
 * lse_ws: [N*J*2] float32 workspace written by fwd (max, sum) and consumed by
 * bwd so the backward is a single pass.
 * ---------------------------------------------------------------------- */
int epb_softargmax_fwd(const float* logits, int layout, int N, int J, int D,
                       int H, int W, float* coords, float* lse_ws,
                       epb_stream_t stream);
/* dlogits = p * (s - sum p s),  s = gx*x/W + gy*y/H + gz*z/D */
int epb_softargmax_bwd(const float* logits, int layout, int N, int J, int D,
                       int H, int W, const float* coords, const float* lse_ws,
                       const float* dcoords, float* dlogits,
                       epb_stream_t stream);
/* The same gradient written straight as the split operand of the final layer's backward
 * (channels_last logits only, D % 4 == 0, J*D/4 <= 1024): dlogits16 = planes [planes][N][H][W][J*D],
 * sc = {s, 1/s} with s from the hard bound max_nj p_max * (|gx|+|gy|+|gz|), and (optional)
 * dbias[J*D] = column sums of the gradient = the final layer's bias gradient, added in a fixed
 * order.  Replaces epb_softargmax_bwd + epb_split16 + epb_colsum of the fp32 form (the logit
 * gradient never exists in fp32: 1 read + 1 write of the volume instead of 4 + 2). */
int epb_softargmax_bwd_split(const float* logits, int N, int J, int D, int H, int W,
                             const float* coords, const float* lse_ws, const float* dcoords,
                             epb_half* dlogits16, float* sc, float* dbias, int planes,
                             epb_stream_t stream);

/* Fused joint-location loss (integral_loss.py:7-47): kind 0 = weighted MSE,
 * 1 = weighted L1, 2 = weighted SmoothL1(beta=1).  loss = sum(w*l(x-t))/div,
 * dx = dloss/dx.  norm != 0: x,t divided by their global L1 norms first
 * (integral_loss.py:9-11).  n = N*J*3 elements (single CTA; n is tiny). */
int epb_jointloss_fwd_bwd(const float* x, const float* t, const float* w, int n,
                          int kind, int norm, float div, float* loss, float* dx,
                          epb_stream_t stream);

/* Heat-map regression loss fused with the joint-location loss, ONE launch (the objective of
 * the VOLUME=False head, pose3d_resnet.py:202-212: 2-D heat-maps + depth branch; the
 * reference keeps only the config remnants of its heat-map loss, lib/core/config.py:32-34
 * LOSS.USE_TARGET_WEIGHT, so the arithmetic is torch.nn.functional.mse_loss on the
 * weighted maps plus integral_loss.py:7-47 on the joint vector):
 *   loss_hm = sum_{r,p} (wh[r] * (hm[r][p] - target[r][p]))^2 / (R*HW)   r = (n, j) map
 *   loss_jt = sum_i w[i] * l_kind(x[i] - t[i]) / div      (kind as epb_jointloss_fwd_bwd)
 *   loss[0] = loss_hm, loss[1] = loss_jt, loss[2] = hm_scale*loss_hm + jt_scale*loss_jt
 *   dhm = d loss[2] / d hm  [R][HW],   dx = d loss[2] / d x  [n]
 * hm, target: [R][HW] float32 contiguous; hm_weight [R] or NULL (ones); n may be 0 (heat-map
 * loss only; x, t, w, dx ignored); dhm / dx may be NULL (loss only).  Deterministic. */
int epb_heatmap_joint_loss(const float* hm, const float* target, const float* hm_weight,
                           int R, int HW, float hm_scale, const float* x, const float* t,
                           const float* w, int n, int kind, float div, float jt_scale,
                           float* loss, float* dhm, float* dx, epb_stream_t stream);

/* Hard argmax (numpy call site lib/core/inference.py:24-39).  hm [NJ][HW]
 * float32 contiguous.  idx: flat first-max index (int32), maxval float32,
 * preds [NJ][2] float32 = (idx%W, idx/W) * (max > 0). */
int epb_argmax2d(const float* hm, int NJ, int H, int W, int32_t* idx,
                 float* maxval, float* preds, epb_stream_t stream);

/* lib/core/inference.py:43-68 get_final_preds in one launch: the argmax above, the +-0.25 px
 * refinement toward the higher neighbour (:49-61, when post_process != 0) and transform_preds
 * (lib/utils/transforms.py:39-44) with the inverse affine of get_affine_transform(center,
 * scale, 0, (W, H), inv=1) (:47-79; cv2.getAffineTransform's 6x6 LU on the float32 point
 * triplets).  hm [N][J][H][W] float32; center, scale [N][2] float64 (scale in units of
 * 200 px, :57).  preds [N][J][2] float32 image coordinates, maxvals [N][J] (or NULL). */
int epb_final_preds(const float* hm, int N, int J, int H, int W, const double* center,
                    const double* scale, int post_process, float* preds, float* maxvals,
                    epb_stream_t stream);

/* ------------------------------------------------------------------------
 * Epipolar geometry in float64 (OpenCV/numpy call sites).
 * ---------------------------------------------------------------------- */
/* lib/core/integral_loss.py:196-205 + lib/utils/img_utils.py:141-155:
 * coords [B][J*3] f32 (soft-argmax output) -> image-frame keypoints
 * kps [B][J][4] f64 = (affine_inv(x,y), z*2000/.., 1).  box [B][6] f64 =
 * (c_x, c_y, width, height, scale, rot). */
int epb_patch_to_image(const float* coords, const double* box, int B, int J,
                       double patch_w, double patch_h, double rect3d_w,
                       double* kps, epb_stream_t stream);
/* lib/utils/triangulation.py: u1,u2 [NP][J][stride_u] f64 (first two entries
 * used), P1,P2 [NP][12] f64 row-major 3x4.  X [NP][J][3] f64, status [NP][J].
 * method 0: linear-eigen homogeneous DLT (:8-27, cv2.triangulatePoints);
 * method 1: linear LS (:34-97); method 2: iterative LS, 10 cumulative
 * re-weighting rounds, tol 3e-5 (:104-181); method 3: polynomial / optimal
 * (:184-220): F = [t]x R of the canonical pair, cv2.correctMatches
 * (Hartley-Sturm: degree-6 polynomial per match, roots by Laguerre iteration),
 * then method 0 on the corrected matches; when the correction is NaN for every
 * joint of a pair (F = 0: identical / degenerate cameras) F is re-estimated from
 * the matches with the normalised 8-point algorithm (cv2.findFundamentalMat(...,
 * FM_8POINT), :215-217) and the correction repeated.  method 4: always the
 * 8-point F (the fallback branch on its own). */
int epb_triangulate(const double* u1, const double* u2, int stride_u,
                    const double* P1, const double* P2, int NP, int J,
                    int method, double tol, double* X, int32_t* status,
                    epb_stream_t stream);
/* V-view homogeneous DLT (SURVEY 8(f) row 3; the reference only pairs two views,
 * triangulation.py:8-27): u [NT][V][J][stride_u] f64 (first two entries used), P [NT][V][12] f64,
 * 2 <= V <= 4 -> X [NT][J][3], status [NT][J] (max |coordinate| <= 1e16). */
int epb_triangulate_nview(const double* u, int stride_u, const double* P, int NT, int V, int J,
                          double* X, int32_t* status, epb_stream_t stream);
/* lib/utils/img_utils.py:212-243 + lib/utils/prep_h36m.py:170-204 +
 * integral_loss.py:170-177: X [B][J][3] world -> label,weight [B][J*3] f32.
 * cam [B][16] f64 = R(9) T(3) f(2) c(2); box as above. */
int epb_project_labels(const double* X, const double* cam, const double* box,
                       int B, int J, double patch_w, double patch_h,
                       double rect3d_w, float* label, float* weight,
                       epb_stream_t stream);

/* H36M evaluation protocol per sample (lib/dataset/h36m.py:168-378: CamBackProj
 * lib/utils/prep_h36m.py:85-89, compute_similarity_transform(..., compute_optimal_scale=True)
 * :108-168, root alignment, per-joint Euclidean errors).  float64.
 *   pred, gt  [S][J][3]  image-space joints (x px, y px, root-relative depth mm); gt already in
 *                        the order of pred (the H36M_TO_MPII permutation is a host gather)
 *   cam       [S][5]     fx, fy, cx, cy, pelvis depth (gt['fl'], gt['c_p'], gt['pelvis'][2])
 *   root                 root joint (6 with MPII_ORDER, else 0); j14mask: bit j set <=> joint j
 *                        belongs to the 14-joint subset; pck_thr = 150 (mm)
 *   metrics   [S][9]     means over joints of: e, e_align, e_norm, e (14), e_align (14),
 *                        e_norm (14), |dx|, |dy|, |dz|
 *   per_joint [S][J] (or NULL)  e per joint;   pck [S][J] int32 (or NULL)  e < pck_thr
 *   poses     [S][J][9] (or NULL)  root-aligned pred | align_pred | gt  (pred_to_save) */
int epb_h36m_eval(const double* pred, const double* gt, const double* cam, int S, int J,
                  int root, uint32_t j14mask, double pck_thr, double* metrics,
                  double* per_joint, int32_t* pck, double* poses, epb_stream_t stream);

/* Element-wise helpers of the refiner MLP (refiner/model.py:39-68,117-143): out = a + b (+ c when
 * c != NULL) -- the residual sums -- and nn.Dropout with an explicit keep mask:
 * out = mask ? x * scale : 0  (scale = 1 / (1 - p); the backward is the same call on the gradient). */
int epb_add3(const float* a, const float* b, const float* c, float* out, int64_t n, epb_stream_t stream);
int epb_mask_scale(const float* x, const uint8_t* mask, float scale, float* out, int64_t n,
                   epb_stream_t stream);

/* torch.nn.utils.clip_grad_norm_(parameters, max_norm) of the refiner loop (refiner/main.py:57)
 * over a list of gradient tensors, without a host round trip: epb_sumsq adds sum(x^2) of one
 * tensor to the DEVICE float64 scalar *total (caller zeroes); epb_clip_scale multiplies one
 * tensor by clamp(max_norm / (sqrt(*total) + 1e-6), max = 1). */
int epb_sumsq(const float* x, int64_t n, double* total, epb_stream_t stream);
int epb_clip_scale(float* x, int64_t n, const double* total, double max_norm, epb_stream_t stream);

/* ------------------------------------------------------------------------
 * Input pipeline (lib/utils/img_utils.py:246-298 get_single_patch_sample after the frame is
 * decoded, including the occluder paste of lib/utils/augmentation.py:61-114).
 * ---------------------------------------------------------------------- */
/* Crop + colour + normalisation of B frames in one launch, bit-exact against OpenCV:
 * generate_patch_image_cv (:114-127: gen_trans_from_patch_cv :72-105 with float32 point
 * triplets and cv2.getAffineTransform's 6x6 LU; cv2.warpAffine INTER_LINEAR, constant border 0,
 * fixed-point coordinates and weights as imgproc/imgwarp.cpp), BGR->RGB (:268), colour scale,
 * clip to [0,255], (x-mean)/std (:277-281).
 *   img_base            uint8 BGR frames (cv2.imread layout [H][W][3]) in one device buffer
 *   img_off  [B] int64  byte offset of frame b;  img_hwp [B][3] int32: H, W, row pitch in bytes
 *   box      [B][6] f64 c_x, c_y, bb_width, bb_height, scale, rot (degrees)
 *   flip     [B] int32 or NULL (horizontal mirror: img[:, ::-1, :], c_x = W - c_x - 1, :118-120)
 *   color    [B][3] f32 or NULL (ones): colour_scale per RGB channel
 *   mean_std_host [6] f64 HOST pointer (mean RGB, std RGB) or NULL (no normalisation)
 *   out      [B][3][patch_h][patch_w] f32;  trans [B][6] f64 or NULL: the image->patch affine */
int epb_patch_sample(const uint8_t* img_base, const int64_t* img_off, const int32_t* img_hwp,
                     const double* box, const int32_t* flip, const float* color,
                     const double* mean_std_host, int B, int patch_w, int patch_h, float* out,
                     double* trans, epb_stream_t stream);
/* The same with the synthetic-occlusion augmentation (img_utils.py:269-270, augmentation.py:
 * 61-114 occlude_with_objects / paste_over): after the crop and BGR->RGB, up to 7 RGBA occluders
 * per sample are alpha-blended IN ORDER into the uint8 patch -- float32 alpha*src + (1-alpha)*dst,
 * truncated to uint8, bit-exact against numpy -- before the colour scale / normalisation.  The
 * random draws and the cv2.resize of each occluder are host-side augmentation parameters:
 *   occ_base            uint8 RGBA occluder images (already resized), one device buffer
 *   occ_desc [B][7][5]  int64: byte offset, width, height, centre x, centre y (np.round'ed)
 *   occ_count [B]       int32: occluders of sample b (0..7); all three NULL = no occluders. */
int epb_patch_sample_occ(const uint8_t* img_base, const int64_t* img_off, const int32_t* img_hwp,
                         const double* box, const int32_t* flip, const float* color,
                         const double* mean_std_host, int B, int patch_w, int patch_h,
                         const uint8_t* occ_base, const int64_t* occ_desc, const int32_t* occ_count,
                         float* out, double* trans, epb_stream_t stream);
/* Joint half (:283-296 + lib/core/integral_loss.py:170-177): joints [B][J][3] f64 (x, y image px;
 * z mm) through trans [B][6] (from epb_patch_sample), z / (rect_3d_w*scale) * patch_w (or the
 * box width when depth_in_image), then x/pw - 0.5, y/ph - 0.5, z/pw -> label [B][J*3] f64. */
int epb_patch_joints(const double* joints, const double* box, const double* trans, int B, int J,
                     double patch_w, double patch_h, double rect_3d_w, int depth_in_image,
                     double* label, epb_stream_t stream);

/* ------------------------------------------------------------------------
 * Optimiser (torch.optim.Adam call site lib/utils/utils.py:56-60; betas
 * (0.9,0.999), eps 1e-8, no weight decay) over one flat parameter buffer.
 * step is the 1-based step count.  grad_scale multiplies the gradient first
 * (1/world_size after the NCCL sum).
 * ---------------------------------------------------------------------- */
int epb_adam_step(float* param, const float* grad, float* exp_avg,
                  float* exp_avg_sq, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int step,
                  float grad_scale, epb_stream_t stream);
int epb_sgd_step(float* param, const float* grad, float* momentum_buf, int64_t n,
                 float lr, float momentum, float weight_decay, int nesterov,
                 int first_step, float grad_scale, epb_stream_t stream);

/* Same updates with the hyper-parameters and the step count read from DEVICE
 * memory, so that a whole training step can be captured in a CUDA graph and
 * replayed while the LR schedule (scripts/train.py:107-109) keeps changing:
 * adam hyper = [lr, beta1, beta2, eps, weight_decay, grad_scale];
 * sgd  hyper = [lr, momentum, weight_decay, nesterov, grad_scale];
 * *step_dev is the 1-based step (the caller increments it before the call). */
int epb_adam_step_dev(float* param, const float* grad, float* exp_avg,
                      float* exp_avg_sq, int64_t n, const float* hyper,
                      const int* step_dev, epb_stream_t stream);
int epb_sgd_step_dev(float* param, const float* grad, float* momentum_buf,
                     int64_t n, const float* hyper, const int* step_dev,
                     epb_stream_t stream);

/* Profiling aid (never on a product path): with EPB_C16_PROBE & 32 in the environment, cluster 0 of
 * an epb_conv16_fprop launch records clock64() at its pipeline hand-overs; this copies the trace
 * ([role: producer, MMA issuer, epilogue per tile, epilogue per chunk][CTA rank][256] int64) to host memory after a device sync. */
int epb_debug_conv16_trace(long long* host_dst, int n);

#ifdef __cplusplus
}
#endif
#endif /* EPB_H_ */
