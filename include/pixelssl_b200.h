/*
 * pixelssl_b200 -- C ABI of the B200-native (sm_100a) hot path of PixelSSL's semantic-segmentation
 * SSL training step.  Plain pointers and sizes, no torch types.  Every pointer is a DEVICE pointer
 * unless the parameter name ends in `_host`.  `stream` is a cudaStream_t passed as void*.
 * Every entry point returns 0 on success or a cudaError_t / negative pxl error code; nothing is
 * ever computed on the host as a fallback.
 *
 * Each group cites the reference call site it replaces (paths relative to the PixelSSL tree).
 * Layouts: "NHWC" = channels innermost (torch channels_last), used for backbone activations;
 * "planar" = NCHW, used for the C=21 logit / probability maps exactly like the reference.
 * The reference-side binding is Python: see INTEGRATION.md (ctypes stub used by
 * pixelssl_b200/_lib.py).
 */
#ifndef PIXELSSL_B200_H
#define PIXELSSL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PXL_ERR_BAD_ARG   (-1)
#define PXL_ERR_UNSUPPORTED (-2)

/* library identity: returns the ABI version (bumped on signature changes) */
int pxl_abi_version(void);
/* number of kernel launches issued through this library since load / last reset (bench.py
 * reports it as gpu_launches) */
int64_t pxl_launch_count(void);
void pxl_reset_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Consistency loss: nn.MSELoss() on student vs detached teacher maps
 *   pixelssl/ssl_algorithm/ssl_mt.py:115,179-187 (logits), ssl_cutmix.py:212-215,
 *   ssl_gct.py:450, ssl_cct.py:484 (softmax maps)
 * loss_out[0] = loss_scale * mean((s - t)^2) over n elements (fp64 accumulation, deterministic
 * two-level reduction).  If grad_s != NULL also writes grad_s = loss_scale * 2 (s - t) / n
 * (the fused fwd+bwd form: 12 B/element algorithmic traffic; forward-only is 8 B/element).
 * workspace: >= pxl_mse_workspace_bytes() bytes, zero-initialised once (the kernel restores it).
 * ------------------------------------------------------------------------------------------- */
int64_t pxl_mse_workspace_bytes(void);
int pxl_mse_consistency(const float* s, const float* t, int64_t n, float loss_scale,
                        float* loss_out, float* grad_s, void* workspace, void* stream);
/* generic backward for a device-resident upstream scalar: grad_s = upstream[0]*scale*2(s-t)/n */
int pxl_mse_consistency_bwd(const float* s, const float* t, int64_t n, float loss_scale,
                            const float* upstream, float* grad_s, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Per-pixel cross-entropy: CommonSSEGCriterion.forward, task/sseg/criterion.py:24-38
 *   (nn.CrossEntropyLoss(ignore_index, reduction='none') on gt.long(), then mean over ALL H*W)
 * logits planar [n, C, H*W]; labels fp32 [n, H*W] holding integers; per_sample[n] receives
 * sum_pixels(ce)/HW (ignored pixels add 0 but count in the denominator).
 * grad_logits (nullable) = g * (softmax - onehot) / HW on valid pixels, 0 on ignored ones, with
 * g = upstream[i] if upstream != NULL else upstream_const (e.g. 1/lbs for the torch.mean that
 * follows at ssl_mt.py:160).  Labels outside [0, C) other than ignore_index -> PXL_ERR_BAD_ARG is
 * NOT detected on device; they are treated as ignored (documented deviation: torch asserts).
 * ------------------------------------------------------------------------------------------- */
int pxl_ce2d(const float* logits, const float* labels, int n, int C, int64_t HW, int ignore_index,
             float* per_sample, float* grad_logits, const float* upstream, float upstream_const,
             void* stream);

/* ---------------------------------------------------------------------------------------------
 * Channel softmax on planar maps: F.softmax(pred, dim=1), task/sseg/model.py:62,121;
 * task/sseg/func.py:216-220
 * ------------------------------------------------------------------------------------------- */
int pxl_softmax_planar(const float* logits, float* prob, int n, int C, int64_t HW, void* stream);
/* grad_logits = p * (g - sum_c g*p) */
int pxl_softmax_planar_bwd(const float* prob, const float* grad_prob, float* grad_logits,
                           int n, int C, int64_t HW, void* stream);
/* fused CutMix / GCT / CCT consistency: loss = loss_scale*mean((softmax(s_logits)-t_prob)^2);
 * optional prob_out (softmax of s), optional grad_logits (through the softmax).
 * ssl_cutmix.py:206-215 */
int pxl_softmax_mse(const float* s_logits, const float* t_prob, int n, int C, int64_t HW,
                    float loss_scale, float* loss_out, float* prob_out, float* grad_logits,
                    void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Bilinear resize, F.interpolate(mode='bilinear'): deeplab_v2.py:32, _pspnet.py:99-100,127,
 * ssl_gct.py:580, ssl_adv.py:488, ssl_cct.py:482.  Planar [n*C, h, w] -> [n*C, H, W].
 * in_nhwc != 0: the input is NHWC with channel stride ldc (e.g. the ASPP output padded to 32).
 * ------------------------------------------------------------------------------------------- */
int pxl_bilinear_fwd(const float* in, float* out, int n, int C, int h, int w, int H, int W,
                     int align_corners, int in_nhwc, int ldc, void* stream);
int pxl_bilinear_bwd(const float* grad_out, float* grad_in, int n, int C, int h, int w, int H, int W,
                     int align_corners, int in_nhwc, int ldc, void* stream);

/* ---------------------------------------------------------------------------------------------
 * CutMix: mask*a + (1-mask)*b, bit-exact with the reference's fp32 evaluation order
 *   ssl_cutmix.py:195,428.  a,b,out: [n, C, HW]; mask: [n, 1, HW] (broadcast over C).
 * Confidence: count of pixels with max_c p > thr (ssl_cutmix.py:200); count_out is int64[1].
 * ------------------------------------------------------------------------------------------- */
int pxl_cutmix_mix(const float* mask, const float* a, const float* b, float* out,
                   int n, int C, int64_t HW, void* stream);
int pxl_cutmix_confidence(const float* prob, int n, int C, int64_t HW, float thr,
                          unsigned long long* count_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * BatchNorm2d (training and eval), NHWC rows = N*H*W, C channels:
 *   _SynchronizedBatchNorm.forward, sync_batchnorm/batchnorm.py:48-78,113-125
 * stats: sums[0:C] = sum x, sums[C:2C] = sum x^2 as fp64 (atomically accumulated; caller zeroes).
 *   For N>1 GPUs the caller all-reduces `sums` (NCCL) between stats and finalize.
 * finalize: from sums & count -> mean, invstd (biased var; invstd = 1/sqrt(var+eps), or
 *   clamp(var,eps)^-1/2 when clamp_mode!=0 = the reference's multi-replica formula), updates
 *   running stats with the unbiased variance (momentum), writes scale=gamma*invstd,
 *   shift=beta-mean*scale.
 * apply: y = x*scale + shift (+ residual) (ReLU if relu!=0).
 * ------------------------------------------------------------------------------------------- */
int pxl_bn_stats(const float* x, int64_t rows, int C, double* sums, void* stream);
int pxl_bn_finalize(const double* sums, double count, int C, const float* gamma, const float* beta,
                    float* running_mean, float* running_var, float momentum, float eps,
                    int clamp_mode, float* mean, float* invstd, float* scale, float* shift,
                    void* stream);
/* eval mode: scale/shift from running stats */
int pxl_bn_eval_coeffs(int C, const float* gamma, const float* beta, const float* running_mean,
                       const float* running_var, float eps, float* scale, float* shift, void* stream);
int pxl_bn_apply(const float* x, const float* scale, const float* shift, const float* residual,
                 int relu, float* y, int64_t rows, int C, void* stream);
/* training forward in one launch: pxl_bn_finalize + pxl_bn_apply (sums already hold the batch totals). */
int pxl_bn_finalize_apply(const float* x, const double* sums, double count, const float* gamma,
                          const float* beta, float* running_mean, float* running_var, float momentum,
                          float eps, int clamp_mode, float* mean, float* invstd, float* scale, float* shift,
                          const float* residual, int relu, float* y, int64_t rows, int C, void* stream);
/* backward of y = relu?(bn(x) + residual?):
 *   reduce: dsums[0:C] = sum dz, dsums[C:2C] = sum dz*xhat with dz = dy * (y>0 if relu) (fp64;
 *   caller zeroes; all-reduced for N>1);  writes nothing else.
 *   dx:  dx = gamma*invstd*(dz - dsums0/count - xhat*dsums1/count); dres (nullable) = dz.
 *   dgamma += dsums1, dbeta += dsums0 are produced by pxl_bn_bwd_params.
 *   relu with y == NULL: the mask is recomputed as fmaf(x, scale, shift) > 0 (exactly what pxl_bn_apply
 *   evaluated; only valid without a residual) - saves reading y. */
int pxl_bn_bwd_reduce(const float* x, const float* y, const float* dy, const float* mean,
                      const float* invstd, int relu, int64_t rows, int C, double* dsums,
                      const float* scale, const float* shift, void* stream);
int pxl_bn_bwd_dx(const float* x, const float* y, const float* dy, const float* mean,
                  const float* invstd, const float* gamma, const double* dsums, double count,
                  int relu, float* dx, float* dres, int64_t rows, int C,
                  const float* scale, const float* shift, float* dgamma_acc, float* dbeta_acc, void* stream);
/* dgamma_acc / dbeta_acc (both or neither): dgamma_acc[c] += dsums[C+c], dbeta_acc[c] += dsums[c] by the same launch
 * (single-GPU path: dsums are the local sums; replaces pxl_bn_bwd_params + the optimizer-side accumulation). */
/* fp16-pair variants (csrc/h16_prep.cu) of the BatchNorm launches: the SAME pass that writes y (dx) also, or only
 * (y / dx NULL), writes it as the fp16 pair the next tcgen05 convolution reads, so the pair costs no extra trip
 * through HBM.  hi / lo: __half NHWC planes, lo nullable.  Forward: fixed scale `hscale`.  Backward: the reduce
 * launch leaves absmax(dz) in slot[2] (DEVICE float[4], zeroed), the dx launch derives the power-of-two scale from
 * it, max|gamma*invstd| and target_log2, and stores s / 1/s in slot[0] / slot[1].
 * relu_mask (nullable, rows*C/4 bytes): the forward launches store the sign bits of the result (bit k of byte i =
 * element 4i+k > 0); the backward launches then take the ReLU mask from it instead of re-reading the fp32 result
 * (0.25 B/element instead of 4). */
int pxl_bn_apply_h16(const float* x, const float* scale, const float* shift, const float* residual, int relu, float* y,
                     int64_t rows, int C, void* hi, void* lo, float hscale, void* relu_mask, void* stream);
int pxl_bn_finalize_apply_h16(const float* x, const double* sums, double count, const float* gamma, const float* beta,
                              float* running_mean, float* running_var, float momentum, float eps, int clamp_mode,
                              float* mean, float* invstd, float* scale, float* shift, const float* residual, int relu,
                              float* y, int64_t rows, int C, void* hi, void* lo, float hscale, void* relu_mask,
                              void* stream);
int pxl_bn_bwd_reduce_h16(const float* x, const float* y, const float* dy, const float* mean, const float* invstd,
                          int relu, int64_t rows, int C, double* dsums, const float* scale, const float* shift,
                          float* amax_slot, const void* relu_mask, void* stream);
int pxl_bn_bwd_dx_h16(const float* x, const float* y, const float* dy, const float* mean, const float* invstd,
                      const float* gamma, const double* dsums, double count, int relu, float* dx, float* dres,
                      int64_t rows, int C, const float* scale, const float* shift, float* dgamma_acc, float* dbeta_acc,
                      void* dhi, void* dlo, float* slot, int target_log2, const void* relu_mask, void* stream);
int pxl_bn_bwd_params(const double* dsums, int C, float* dgamma, float* dbeta, int accumulate,
                      void* stream);

/* ---------------------------------------------------------------------------------------------
 * MaxPool2d(3, stride 2, pad 1) on NHWC: resnet.py:72,125
 * ------------------------------------------------------------------------------------------- */
int pxl_maxpool3x3s2_fwd(const float* x, float* y, int N, int H, int W, int C, int OH, int OW,
                         void* stream);
int pxl_maxpool3x3s2_bwd(const float* x, const float* y, const float* dy, float* dx,
                         int N, int H, int W, int C, int OH, int OW, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Convolution, NHWC activations, weights [Cout][tap][Cin] (= torch channels_last OIHW storage),
 * arbitrary tap table (dy,dx per tap) so that a dilated 3x3 is 9 taps and the whole ASPP head
 * (deeplab_v2.py:71-85: 4 dilated 3x3 convs summed) is ONE 36-tap convolution.
 *   nn.Conv2d call sites: resnet.py:18-25,69,88-91 ; deeplab_v2.py:76,81-85 ; _pspnet.py:17,46,69,90
 *
 * geometry: out[n,oy,ox,co] = bias[co] + sum_t sum_ci in[n, (oy*mul + dy_t)/div, (ox*mul + dx_t)/div, ci]
 *                                                   * w[co][t][ci]
 *   (terms whose coordinate is not divisible by div or falls outside [0,H)x[0,W) are zero).
 *   forward conv: mul=stride, div=1, dy_t = r*dil - pad.   dgrad: mul=1, div=stride, taps negated,
 *   weights transposed to [Cin][tap][Cout] (pxl_conv_transpose_weights).
 * precision: 0 = fp32 FFMA (exact fp32 accumulate), 1 = tf32 tensor cores (tcgen05), 2 = 3xTF32
 *   error-compensated tcgen05.  Unsupported (shape, precision) combos return PXL_ERR_UNSUPPORTED.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int N, H, W, Cin;        /* input tensor  */
    int OH, OW, Cout;        /* output tensor */
    int ldo;                 /* output channel stride (>= Cout; 32 for the padded ASPP output) */
    int mul, div;            /* coordinate transform, see above */
    int ntaps;               /* <= PXL_MAX_TAPS */
    int precision;
} pxl_conv_geom;
#define PXL_MAX_TAPS 64
int pxl_conv_nhwc(const pxl_conv_geom* geom_host, const int* taps_dydx_host /* 2*ntaps ints */,
                  const float* in, const float* w, const float* bias /* nullable */,
                  float* out, void* stream);
/* dW[co][t][ci] += sum over output pixels of dy[n,oy,ox,co] * in[n, iy, ix, ci]   (accumulates) */
int pxl_conv_wgrad_nhwc(const pxl_conv_geom* geom_host, const int* taps_dydx_host,
                        const float* in, const float* dy, float* dw, void* stream);
/* tcgen05 path with explicit operands.  precision 1: in_lo / w_lo ignored (NULL).  precision 2
 * (3xTF32): in_hi/in_lo and w_hi/w_lo are the tf32 split of the fp32 tensors (pxl_split_tf32):
 * out = in_hi*w_hi + in_lo*w_hi + in_hi*w_lo accumulated in fp32 (TMEM).  Supports mul == div == 1
 * and Cin % 32 == 0; anything else returns PXL_ERR_UNSUPPORTED. */
int pxl_conv_tc_launch(const pxl_conv_geom* geom_host, const int* taps_dydx_host, const float* in_hi,
                       const float* in_lo, const float* w_hi, const float* w_lo, const float* bias,
                       float* out, void* stream);
/* Extended form used for strided convolutions:
 *  - geom.mul == 2 (stride-2 forward) is served by the TMA traversal stride;
 *  - stride-2 dgrad is decomposed by output parity into four stride-1 problems over dY: each launch
 *    passes the taps of one parity class (offsets already halved), `widx_host[t]` = index of tap t in
 *    the [rows][w_ntaps][Cin] weight tensor, and stores its OH x OW result at
 *    (oy*out_mul + out_offy, ox*out_mul + out_offx) of the out_H x out_W output image. */
typedef struct {
    int w_ntaps;             /* taps held by the weight tensor (>= geom.ntaps); 0 = geom.ntaps */
    const int* widx_host;    /* nullable: identity */
    int out_mul, out_offy, out_offx, out_H, out_W;   /* out_mul == 0 is read as "no output transform" */
    double* bn_stats;        /* nullable DEVICE pointer [2*Cout] fp64: the epilogue adds sum(y), sum(y^2) per
                              * output channel (the statistics pass of the BatchNorm that follows,
                              * sync_batchnorm/batchnorm.py:60-62) */
    float out_scale;         /* 0 is read as 1: the accumulator is multiplied by out_scale * (*out_scale_dev) before */
    const float* out_scale_dev;   /* bias / statistics / store (undoes the power-of-two scales of fp16 pairs); nullable */
    int out_accumulate;      /* != 0: out += result (TMA reduce-add epilogue; PXL_ERR_UNSUPPORTED where that epilogue is not used) */
} pxl_conv_tc_ext;
int pxl_conv_tc_launch_ex(const pxl_conv_geom* geom_host, const int* taps_dydx_host, const pxl_conv_tc_ext* ext_host,
                          const float* in_hi, const float* in_lo, const float* w_hi, const float* w_lo,
                          const float* bias, float* out, void* stream);
/* tcgen05 wgrad (accumulates into dw): both operands MN-major via TMA, split over the pixel range.  Every split
 * writes its tile into its own slot of the DEVICE workspace ws, and the slots are then added into dw in split order,
 * so dw is the same in every run.  ws holds at least pxl_conv_wgrad_workspace_floats(geom, taps) floats and must not
 * be used by another stream until this launch's work on `stream` is done.  Same precision / operand convention as
 * pxl_conv_tc_launch; needs mul == div == 1, Cin % 32 == 0 and ldo % 32 == 0. */
int64_t pxl_conv_wgrad_workspace_floats(const pxl_conv_geom* geom_host, const int* taps_dydx_host);
int pxl_conv_wgrad_tc_launch(const pxl_conv_geom* geom_host, const int* taps_dydx_host, const float* in_hi,
                             const float* in_lo, const float* dy_hi, const float* dy_lo, float* dw,
                             float* ws, int64_t ws_floats, void* stream);
/* ---- fp16 pairs: the operand format of the kind::f16 tcgen05 path (csrc/h16_prep.cu) -------------------------
 * x*s = hi + lo, hi = fp16(x*s), lo = fp16(x*s - hi), s a power of two.  precision 3 ("f16x3"): hi*hi + lo*hi +
 * hi*lo in fp32 (products good to ~2^-21: fp32-grade, like 3xTF32, at twice its MMA rate); precision 4 ("f16"):
 * hi*hi only (11-bit significands = the TF32 numerics of the reference's cuDNN path).  Same geometry contract as
 * pxl_conv_tc_launch_ex with Cin % 64 == 0 (wgrad: Cin % 64 == 0 and ldo % 64 == 0); operands are __half NHWC /
 * [Cout][taps][Cin] tensors; ext->out_scale(_dev) undo the operand scales.  These replace the same reference
 * calls as pxl_conv_nhwc (nn.Conv2d forward / backward, resnet.py:18-25). */
int pxl_conv_h16_launch(const pxl_conv_geom* geom_host, const int* taps_dydx_host, const pxl_conv_tc_ext* ext_host,
                        const void* in_hi, const void* in_lo, const void* w_hi, const void* w_lo,
                        const float* bias, float* out, void* stream);
int pxl_conv_wgrad_h16_launch(const pxl_conv_geom* geom_host, const int* taps_dydx_host, const void* in_hi,
                              const void* in_lo, const void* dy_hi, const void* dy_lo, float* dw, float out_scale,
                              const float* out_scale_dev, float* ws, int64_t ws_floats, void* stream);
/* x -> (hi, lo).  slot == NULL: fixed `scale`.  slot != NULL (DEVICE float[4], zeroed, then filled by
 * pxl_h16_absmax on the same stream): s = 2^(target_log2 - ceil(log2 absmax)); the kernel stores s in slot[0] and
 * 1/s in slot[1] (what out_scale_dev points at).  lo nullable; n % 4 == 0.  Out-of-range values saturate at
 * +-65504 and are counted (pxl_h16_status). */
int pxl_h16_split(const float* x, void* hi, void* lo, int64_t n, float scale, float* slot, int target_log2,
                  void* stream);
int pxl_h16_absmax(const float* x, int64_t n, float* slot, void* stream);
int* pxl_h16_sat_counter(void);      /* DEVICE int[4] the producers of fp16 pairs add saturation events to */
int pxl_h16_status(void);            /* number of threads that clipped a value since the last reset (synchronises) */
int pxl_h16_status_sites(int* out4_host);   /* the same per producer: split fixed / split dynamic / BN apply / BN dx */
int pxl_h16_reset_status(void);
/* hi = round-to-nearest tf32 of x (low 13 mantissa bits zero), lo = x - hi (exact); n % 4 == 0 */
int pxl_split_tf32(const float* x, float* hi, float* lo, int64_t n, void* stream);
/* watchdog of the mbarrier pipelines: 0 = healthy, else the role that timed out (synchronises) */
int pxl_conv_tc_status(void);
/* w [Cout][T][Cin] -> wt [Cin][T][Cout] */
int pxl_conv_transpose_weights(const float* w, float* wt, int Cout, int T, int Cin, void* stream);
/* the same for every conv weight of a parameter arena in one launch: table[n][6] (device, int64) = {src offset,
 * dst offset, Cout, T, Cin, first tile}; tiles = 32x32 (co,ci) blocks per tap, numbered tensor by tensor */
int pxl_conv_transpose_weights_batched(const float* src_base, float* dst_base, const int64_t* table, int n,
                                       int64_t total_tiles, void* stream);
/* dbias[co] (+)= sum over rows of dy[row, co] (row stride ldo) */
int pxl_bias_grad(const float* dy, int64_t rows, int Cout, int ldo, float* dbias, int accumulate,
                  void* stream);

/* stem: conv 7x7 stride 2 pad 3 on the planar [N,3,H,W] image -> NHWC [N,OH,OW,64]
 * (resnet.py:69,121); weights [64][7*7][3].  wgrad accumulates into dw. */
int pxl_stem_conv7x7s2(const float* img_planar, const float* w, float* out, int N, int H, int W,
                       int OH, int OW, void* stream);
int pxl_stem_conv7x7s2_wgrad(const float* img_planar, const float* dy, float* dw, int N, int H, int W,
                             int OH, int OW, void* stream);
/* im2col of the stem for the tensor-core path: cols [N*OH*OW][160], k = (r*7+s)*3+c (the weight's physical
 * order), lanes 147..159 zero; the stem then is a flat 1x1 convolution with 160 input lanes */
int pxl_stem_im2col(const float* img_planar, float* cols, int N, int H, int W, int OH, int OW, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optimiser + EMA on flat parameter arenas:
 *   torch.optim.SGD as configured by pixelssl/nn/optimizer.py:57-75 (momentum, wd, dampening 0)
 *   + SSLMT._update_ema_variables, ssl_mt.py:359-363 / ssl_cutmix.py:434-438
 * d = g + wd*p ; buf = d (first_step) else mom*buf + d ; p -= lr*buf ; if teacher != NULL:
 * teacher = teacher*ema_d + (1-ema_d)*p.   28 B/param fused (20 without the teacher).
 * ------------------------------------------------------------------------------------------- */
int pxl_sgd_ema(float* p, const float* g, float* buf, float* teacher, int64_t n, float lr,
                float momentum, float weight_decay, float ema_d, int first_step, void* stream);
int pxl_ema(float* teacher, const float* student, int64_t n, float ema_d, void* stream);

/* ---------------------------------------------------------------------------------------------
 * AdvSSL / GCT / CCT tails
 * ------------------------------------------------------------------------------------------- */
/* planar [n,C,HW] <-> NHWC [n,HW,ldc] lanes [coff, coff+C): inputs of FCDiscriminator.forward
 * (ssl_adv.py:472-488) and FlawDetector.forward (ssl_gct.py:566-570, cat(image, softmax)) */
int pxl_planar_to_nhwc(const float* in, float* out, int n, int C, int64_t HW, int ldc, int coff, void* stream);
int pxl_nhwc_to_planar(const float* in, float* out, int n, int C, int64_t HW, int ldc, int coff, void* stream);
/* one-hot of the float labels into NHWC lanes (ignore / out-of-range -> all zero):
 * ssladv_convert_task_gt_to_fcd_input, sslgct_prepare_task_gt_for_fdgt (task/sseg/func.py:157-192) */
int pxl_onehot_nhwc(const float* labels, float* out, int64_t pixels, int C, int ldc, int coff, void* stream);
/* LeakyReLU(slope) forward/backward (ssl_adv.py:478, ssl_gct.py:563); n % 4 == 0 */
int pxl_leaky_relu_fwd(const float* x, float* y, int64_t n, float slope, void* stream);
int pxl_leaky_relu_bwd(const float* y, const float* dy, float* dx, int64_t n, float slope, void* stream);
/* FCDiscriminatorCriterion (ssl_adv.py:496-503) fused with ssladv_preprocess_fcd_criterion
 * (task/sseg/func.py:137-155): BCE-with-logits against the constant `target`, pixels whose task label
 * (nullable) equals ignore_index contribute bce(0,0)=ln2 and no gradient; per_sample = mean over HW */
int pxl_bce_logits_masked(const float* pred, const float* labels, float target, int ignore_index, int n,
                          int64_t HW, float* per_sample, float* grad, const float* upstream,
                          float upstream_const, void* stream);
/* torch.optim.Adam step (no amsgrad) over a flat arena: ssl_adv.py:101-102, ssl_gct.py:153-154 */
int pxl_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
             float eps, float weight_decay, int step, void* stream);
/* GaussianBlurLayer (nn/module/gaussian_blur.py:18-64) on [n,H,W] maps as two 1-D reflect-padded
 * passes with the 1-D kernel weights_1d[k] (device); FlawmapHandler / FDGTGenerator, ssl_gct.py:624-728 */
int pxl_gauss_blur_sep(const float* in, float* tmp, float* out, int n, int H, int W, int k,
                       const float* weights_1d, float clamp_min, void* stream);
/* ReflectionPad2d(1) + MaxPool2d(3,1): FDGTGenerator.dilate, ssl_gct.py:708-712 */
int pxl_dilate3x3_reflect(const float* in, float* out, int n, int H, int W, void* stream);
/* per-sample (x-min)/(max-min+eps); zero_below >= 0: zero the map first when its max <= zero_below,
 * with min/max taken before zeroing (FlawmapHandler quirk, ssl_gct.py:648-654) */
int pxl_minmax_norm(const float* in, float* out, int n, int64_t HW, float eps, float zero_below,
                    float clamp_min, void* stream);

/* DCGTGenerator.forward (ssl_gct.py:668-689) on planar predictions and [n,HW] handled flaw maps */
int pxl_gct_dcgt(const float* l_pred, const float* r_pred, const float* l_fm, const float* r_fm, float thr,
                 int n, int C, int64_t HW, float* l_dc, float* r_dc, float* both_bad, void* stream);
/* mu * sum_c |onehot(label) - prob| (ignored / unlabeled pixels have an all-zero one-hot row):
 * FDGTGenerator.forward:714-716 + sslgct_prepare_task_gt_for_fdgt (task/sseg/func.py:179-192) */
int pxl_fdgt_absdiff(const float* prob, const float* labels, float mu, int n, int C, int64_t HW, float* out,
                     void* stream);

/* nn.PixelShuffle(2) on NHWC (C output channels, lanes up to ldo zero-filled); inverse != 0 = backward.
 * _pspnet.py:40-54, ssl_cct.py:501-516 */
int pxl_pixel_shuffle2_nhwc(const float* in, float* out, int N, int h, int w, int C, int ldi, int ldo,
                            int inverse, void* stream);
/* CCT feature perturbations on the NHWC latent (ssl_cct.py:542-745): out = x * pixel_mask[n,hw] *
 * chan_scale[n,c] * (1 + elem_noise[hw,c]), every factor nullable */
int pxl_perturb_nhwc(const float* x, const float* pixel_mask, const float* chan_scale, const float* elem_noise,
                     float* out, int N, int64_t HW, int C, void* stream);
int pxl_channel_mean_nhwc(const float* x, float* out, int64_t pixels, int C, void* stream);
int pxl_argmax_nonzero_mask(const float* logits, float* mask, int n, int C, int64_t HW, void* stream);

/* PSPNet pyramid pooling on NHWC (task/sseg/module/_pspnet.py:57-102): nn.AdaptiveAvgPool2d(bin)
 * forward (x [N,H,W,C] -> y [N,bin,bin,C]) / backward (x = dy, y = dx); bilinear NHWC -> lanes
 * [coff, coff+C) of a wider NHWC tensor (backward: in = grad of the wide tensor, out = grad of the small
 * one); channel-concat copy into / out of a lane range. */
int pxl_adaptive_avgpool_nhwc(const float* x, float* y, int N, int H, int W, int C, int bin, int backward, void* stream);
int pxl_bilinear_nhwc(const float* in, float* out, int N, int h, int w, int C, int H, int W, int ldo, int coff,
                      int align_corners, int backward, void* stream);
int pxl_copy_lanes_nhwc(const float* src, float* dst, int64_t rows, int C, int ld, int coff, int extract, void* stream);

/* Validation confusion matrix: cmat[gt*C + argmax_c pred] += 1 over pixels with 0 <= gt < C (planar pred
 * [n,C,HW], float labels [n,HW], int64 cmat[C*C] accumulated in place; C <= 64).
 * SemanticSegmentationFunc.metrics, task/sseg/func.py:36-48 (np.argmax / np.bincount) */
int pxl_confusion_matrix(const float* pred, const float* gt, int n, int C, int64_t HW, int64_t* cmat,
                         void* stream);
/* Mean-Teacher input noise, in place on inp [n,CHW]: per-sample min/max normalise, add noise, clip to
 * [0,1], de-normalise.  GaussianNoiseLayer.forward, pixelssl/nn/module/gaussian_noise.py:18-41
 * (the caller draws the N(0, uniform(0,std)) noise tensor). */
int64_t pxl_gaussian_noise_workspace_bytes(int n);
int pxl_gaussian_noise(float* inp, const float* noise, int n, int64_t CHW, float* workspace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Cross-GPU BatchNorm statistics over NVLink peer memory (one process per GPU).  Replaces the reference's
 * per-layer replica synchronisation (sync_batchnorm/batchnorm.py:55-78,90-125; comm.py) and, for the forward,
 * also _compute_mean_std: one single-CTA kernel pushes this rank's 2C fp64 sums into every rank's mailbox
 * (CUDA-IPC mapped), waits for all lanes, adds them in rank order and (count > 0) finalizes the layer.
 *   pxl_peer_alloc/export/open: mailbox of pxl_peer_mailbox_bytes() bytes, 64-byte IPC handle, peer mapping.
 *   pxl_peer_allreduce_bn: sums [n = 2C] in place; mailboxes = host array of `world` device pointers (own one at
 *   index rank); seq = 1, 2, 3, ... identical on all ranks; count <= 0: plain all-reduce (backward dsums), where
 *   dgamma_acc / dbeta_acc (both or neither) first receive += the LOCAL sums (the BN parameter gradients).
 * --------------------------------------------------------------------------------------------- */
int64_t pxl_peer_mailbox_bytes(void);
int pxl_peer_alloc(void** ptr);
int pxl_peer_free(void* ptr);
int pxl_peer_export(void* ptr, unsigned char* handle64);
int pxl_peer_open(const unsigned char* handle64, void** ptr);
int pxl_peer_close(void* ptr);
int pxl_peer_allreduce_bn(double* sums, int n, void* const* mailboxes, int rank, int world, int64_t seq,
                          double count, int C, const float* gamma, const float* beta, float* running_mean,
                          float* running_var, float momentum, float eps, int clamp_mode, float* mean,
                          float* invstd, float* scale, float* shift, float* dgamma_acc, float* dbeta_acc,
                          void* stream);
int pxl_peer_status(void);

/* stem im2col written directly as the fp16 pair [pixels][192] of the kind::f16 path (hi, lo nullable; value*scale) */
int pxl_stem_im2col_h16(const float* img_planar, void* hi, void* lo, float scale, int N, int H, int W, int OH, int OW,
                        void* stream);

/* ---- ASPP head as one GEMM + gather (csrc/aspp_gather.cu) ----------------------------------------------------
 * Classifier_Module.forward (task/sseg/module/deeplab_v2.py:81-85) = sum of four dilated 3x3 convolutions 2048 -> C.
 * On the fp16-pair path the channel contraction runs first as one 1x1 GEMM with N = ntaps*C outputs
 * (Z[p,t,co] = W_t x[p]); pxl_aspp_gather adds the taps: out[p,co] = bias[co] + sum_t Z[p + off_t, t, co] (zero
 * padding).  Backward: pxl_aspp_scatter_h16 builds the fp16 pair of dZ[q,t,co] = dy[q - off_t, co] (scale from the
 * absmax in slot[2], like pxl_h16_split) for the dgrad / wgrad GEMMs. */
int pxl_aspp_gather(const float* Z, const float* bias, float* out, int N, int H, int W, int C, int ldz, int ldo,
                    const int* taps_dydx_host, int ntaps, void* stream);
int pxl_aspp_scatter_h16(const float* dy, void* hi, void* lo, float* slot, int target_log2, int N, int H, int W, int C,
                         int ldy, int ldz, const int* taps_dydx_host, int ntaps, void* stream);

/* ---- S4L (pixelssl/ssl_algorithm/ssl_s4l.py) --------------------------------------------------------------
 * SSLS4L._batch_prehandle (:296-350): out [2*bs,C,H,W] = the batch followed by its rotated copies
 * (_rotate_tensor :352-360, angle in {1,2,3} quarter turns per sample; angles = DEVICE int32 [bs]). */
int pxl_s4l_rotate_batch(const float* in, float* out, const int* angles_dev, int bs, int C, int H, int W,
                         int any_quarter_turn, void* stream);

/* ---- input pipeline on the GPU (csrc/input_pipeline.cu) ------------------------------------------------------
 * Replaces the per-sample PIL / numpy work of PascalVocDataset._train_prehandle / _val_prehandle
 * (task/sseg/data.py:90-123): RandomScaleCrop (:223-256) = Pillow BILINEAR resize of the 8-bit image (22-bit
 * fixed-point separable antialiased resampling, 8-bit intermediate) + NEAREST resize of the label + zero padding +
 * crop, RandomHorizontalFlip (:184-192), Normalize (:142-161) and ToTensor (:164-181): HWC uint8 -> CHW float32,
 * bit for bit.  The host draws the random numbers and builds the per-axis tables (window start / tap count, 22-bit
 * weights, NEAREST indices) exactly as Pillow does; all table pointers are DEVICE int32.  lab_hw NULL = unlabeled
 * sample (label output = label_const).  no_resize != 0: plain normalise (+crop / flip) of the source. */
int pxl_input_prehandle(const uint8_t* img_hwc, const uint8_t* lab_hw, int H, int W, int ow, int oh, int no_resize,
                        const int* xb, const int* xk, int kmax_x, const int* yb, const int* yk, int kmax_y,
                        const int* lx, const int* ly, int x1, int y1, int crop_w, int crop_h, int flip,
                        float label_fill, float label_const, const double* mean3_host, const double* std3_host,
                        float* out_img_chw, float* out_lab_hw, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PIXELSSL_B200_H */
