/*
 * micronet_b200 — C-ABI of the B200 (sm_100a) fake-quant conv/linear engine.
 *
 * The reference (666DZY666/micronet) has no FFI: its hot path is Python
 * nn.Module code that composes ATen ops.  This header is the boundary a
 * maintainer binds instead (ctypes stub in INTEGRATION.md): plain device
 * pointers, sizes and a cudaStream_t — no torch types.  Every entry point
 * cites the reference lines it replaces; aliases:
 *   DF  = micronet/compression/quantization/wqaq/dorefa/quantize.py
 *   WB  = micronet/compression/quantization/wbwtab/quantize.py
 *   IAO = micronet/compression/quantization/wqaq/iao/quantize.py
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - tensors are contiguous fp32 NCHW (weights KCRS) as at the reference's
 *     module surface; "codes" are u8 integer levels (level - qmin);
 *   - every call is asynchronous on `stream`, allocates nothing and keeps no
 *     pointer after returning; scratch is passed in by the caller;
 *   - return value: 0 = ok, <0 = invalid argument (MNB_E_*), >0 = cudaError_t;
 *     mnb_last_error() gives a thread-local message.
 */
#ifndef MICRONET_B200_H
#define MICRONET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* mnb_stream_t; /* cudaStream_t */

#define MNB_E_ARG (-1)         /* bad shape / null pointer / unsupported bits */
#define MNB_E_UNSUPPORTED (-2) /* valid request this build has no kernel for  */

int mnb_version(void);
const char* mnb_last_error(void);
/* number of kernel launches issued through this library since load (bench.py's gpu_launches) */
int64_t mnb_launch_count(void);

/* ------------------------------------------------------------------------
 * Convolution geometry (F.conv2d arguments: WB:186-194, DF:113-121, IAO:498-506)
 * ---------------------------------------------------------------------- */
typedef struct {
  int32_t batch, in_c, in_h, in_w;
  int32_t out_c, ker_h, ker_w;
  int32_t stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, groups;
} mnb_conv_shape;

/* ------------------------------------------------------------------------
 * Activation fake-quantizers
 * ---------------------------------------------------------------------- */
#define MNB_ACT_DOREFA 1 /* DF:36-46   clamp(0.1x,0,1) -> round(./s), s = 1/(2^a-1)      */
#define MNB_ACT_IAO 2    /* IAO:214-240 clamp(round(x/s - zp), qmin, qmax)              */
#define MNB_ACT_SIGN 3   /* WB:11-36   sign(x) with 0 -> +1, saturate-STE               */

typedef struct {
  int32_t mode;        /* MNB_ACT_*                                                    */
  int32_t bits;        /* DoReFa a_bits (2..8)                                         */
  int32_t qmin, qmax;  /* IAO level range (IAO:243-288)                                */
  int32_t q_type;      /* IAO: 0 symmetric / 1 asymmetric STE range (IAO:148-157)      */
  const float* scale;  /* IAO: device scalar `scale`                                   */
  const float* zero_point; /* IAO: device scalar `zero_point`                          */
  const float* obs_min;    /* IAO: device scalar observer.min_val                      */
  const float* obs_max;    /* IAO: device scalar observer.max_val                      */
} mnb_act_qparams;

/* Forward.  Any of the three outputs may be NULL.
 *   codes    u8[n]      level - level_min   (DoReFa/IAO; SIGN: 0 or 2 so that e = code-1)
 *   pass_bits u32[ceil(n/32)]  bit i set  <=>  the STE passes the gradient at element i
 *   xq       f32[n]     the fake-quantized tensor the reference module returns           */
int mnb_act_quant_fwd(const float* x, int64_t n, const mnb_act_qparams* qp, uint8_t* codes,
                      uint32_t* pass_bits, float* xq, mnb_stream_t stream);
/* Backward of the same op (autograd of DF:43-45 / IAO:227-239 / WB:22-36):
 *   DoReFa dx = (((g*s)/s) * pass) * 0.1 ; IAO dx = ((g*s) * pass) / s ; SIGN dx = g * pass   */
int mnb_act_quant_bwd(const float* g, const uint32_t* pass_bits, int64_t n, const mnb_act_qparams* qp,
                      float* dx, mnb_stream_t stream);

/* IAO QuantBNFuseConv2d (IAO:858-945): fold BatchNorm statistics into (weight, bias) before quantization, one launch:
 *   ratio = gamma / sqrt(var + eps);  w_fused[k, :] = w[k, :] * ratio[k];  b_fused = beta + (bias - mean) * ratio  (bias may
 *   be NULL).  Backward: dw = dw_fused * ratio and out6[k] = {dgamma, dbeta, dbias, dmean, dvar, 0}.
 * mnb_bn_fold_running: running_mean / running_var <- batch statistics (first call) or (1 - momentum) r + momentum batch. */
int mnb_bn_fold_fwd(const float* w, int32_t out_c, int32_t per_channel, const float* gamma, const float* beta,
                    const float* bias, const float* mean, const float* var, double eps, float* w_fused, float* b_fused,
                    mnb_stream_t stream);
int mnb_bn_fold_bwd(const float* dw_fused, const float* db_fused, const float* w, int32_t out_c, int32_t per_channel,
                    const float* gamma, const float* bias, const float* mean, const float* var, double eps, float* dw,
                    float* out6, mnb_stream_t stream);
int mnb_bn_fold_running(float* running_mean, float* running_var, const float* batch_mean, const float* batch_var, int32_t n,
                        double momentum, int32_t first, mnb_stream_t stream);

/* IAO QuantAdd (IAO:1441-1498) in one pass: out = Q(a) + Q(b) with the shared union-range quantizer (read both addends
 * once, write the sum; pass masks for the backward pass, either may be NULL).  Backward: da = STE_a(g), db = STE_b(g). */
int mnb_quant_add_fwd(const float* a, const float* b, int64_t n, const mnb_act_qparams* qp, float* out,
                      uint32_t* pass_bits_a, uint32_t* pass_bits_b, int32_t relu /* out = max(., 0): inference graphs */,
                      mnb_stream_t stream);
int mnb_quant_add_bwd(const float* g, const uint32_t* pass_bits_a, const uint32_t* pass_bits_b, int64_t n,
                      const mnb_act_qparams* qp, float* da, float* db, mnb_stream_t stream);

/* ------------------------------------------------------------------------
 * IAO observers + update_qparams (IAO:15-139, 292-321), all on device, no host sync.
 *   observer kinds: 0 = MinMaxObserver (running extremum), 1 = MovingAverageMinMaxObserver,
 *                   2 = HistogramObserver (EMA of the k-th smallest |x|, k=int(p*n))
 *   `first` = 1 on the observer's first call (the reference's num_flag == 0 branch).
 *   `rows`  = 1 for q_level "L"; = out_channels for "C"/"FC" (x viewed as [rows, n/rows]).
 *   min_val/max_val/scale/zero_point: the module's registered buffers (rows floats each).
 *   symmetric: 1 -> SymmetricQuantizer, 0 -> AsymmetricQuantizer.  update_qparams=0 only observes.
 *   scratch: >= mnb_observe_scratch_bytes(n, rows) bytes, zero-initialised once by the caller
 *   (the kernels leave it zeroed again).                                                   */
int64_t mnb_observe_scratch_bytes(int64_t n, int32_t rows);
int mnb_iao_observe(const float* x, int64_t n, int32_t rows, int32_t observer_kind, int32_t first,
                    double momentum, double percentile, float* min_val, float* max_val,
                    int32_t update_qparams, int32_t symmetric, int32_t qmin, int32_t qmax,
                    float* scale, float* zero_point, void* scratch, mnb_stream_t stream);
/* update_qparams only (QuantAdd's union range, IAO:1487-1494). */
int mnb_iao_update_qparams(const float* min_val, const float* max_val, int32_t rows, int32_t symmetric,
                           int32_t qmin, int32_t qmax, float* scale, float* zero_point,
                           mnb_stream_t stream);

/* ------------------------------------------------------------------------
 * Weight quantizers.  Forward writes
 *   w_int   i16[numel]  effective integer e with  wq = e * w_scale[k]   (exact)
 *   w_scale f32[K]      per-output-channel dequantization scale
 *   wq      f32[numel]  the fake-quantized weight the reference feeds F.conv2d
 * and whatever the closed-form backward needs in `aux`.
 * ---------------------------------------------------------------------- */
/* DF:61-73.  aux: f32[numel + 4] (tanh values, then {max|t|, #ties, s, -}).  scratch as above. */
int mnb_dorefa_weight_fwd(const float* w, int64_t numel, int32_t out_c, int32_t w_bits, int16_t* w_int,
                          float* w_scale, float* wq, float* aux, void* scratch, mnb_stream_t stream);
int mnb_dorefa_weight_bwd(const float* g_wq, const float* aux, int64_t numel, int32_t w_bits, float* dw,
                          void* scratch, mnb_stream_t stream);
/* WB:98-149.  W = 2 (binary; MUTATES w in place: mean-centre over dim 1 + clamp, WB:98-102)
 *             W = 3 (ternary).  w is [out_c, in_c_per_group, kh*kw].
 * aux: f32[3*out_c] = {alpha_k, threshold_k, count_k}.                                          */
int mnb_wb_weight_fwd(float* w, int32_t out_c, int32_t in_c_per_group, int32_t ker_hw, int32_t W,
                      int16_t* w_int, float* w_scale, float* wq, float* aux, mnb_stream_t stream);
int mnb_wb_weight_bwd(const float* g_wq, const float* w, const float* aux, int32_t out_c,
                      int32_t in_c_per_group, int32_t ker_hw, int32_t W, float* dw, mnb_stream_t stream);
/* IAO:214-240 on a weight tensor with per-row (rows = out_c) or per-layer (rows = 1) qparams that
 * were just refreshed by mnb_iao_observe.  pass: u8[numel] STE mask.                           */
int mnb_iao_weight_fwd(const float* w, int64_t numel, int32_t out_c, int32_t rows, const float* scale,
                       const float* zero_point, const float* obs_min, const float* obs_max,
                       int32_t q_type, int32_t qmin, int32_t qmax, int16_t* w_int, float* w_scale,
                       float* wq, uint8_t* pass, mnb_stream_t stream);
int mnb_iao_weight_bwd(const float* g_wq, const uint8_t* pass, const float* scale, int64_t numel,
                       int32_t out_c, int32_t rows, float* dw, mnb_stream_t stream);

/* ------------------------------------------------------------------------
 * Fake-quantized convolution (WB:186, DF:113, IAO:498/947) and its autograd (ATen
 * convolution_backward).  F.linear (DF:198, IAO:1156) is the 1x1 case on a [B, C, 1, 1] view.
 *
 * Activation operand:  a_codes != NULL : u8 codes, effective integer e_a = code + a_offset,
 *                                        value = e_a * a_scale[0]; a_offset_zp (device scalar,
 *                                        may be NULL) is added to a_offset (IAO zero_point);
 *                      else            : a_f32 raw fp32 activations.
 * Weight operand:      w_int != NULL && a_codes != NULL : exact integer path, s32 accumulate,
 *                                        y = bias + acc * a_scale * w_scale[k];
 *                      else            : w_f32 fp32 weights, fp32 accumulate.
 * ---------------------------------------------------------------------- */
typedef struct {
  const uint8_t* a_codes;
  const float* a_f32;
  int32_t a_offset;
  const float* a_offset_zp;
  const float* a_scale; /* device scalar or NULL (= 1) */
  const int16_t* w_int;
  const float* w_scale; /* f32[out_c] */
  const float* w_f32;
  const float* bias; /* f32[out_c] or NULL */
} mnb_conv_operands;

int mnb_conv2d_fwd(const mnb_conv_shape* s, const mnb_conv_operands* op, float* y, mnb_stream_t stream);
/* dX = conv_transpose(dY, Wq) fused with the activation STE:  pass_bits/qp may be NULL (plain dgrad). */
int mnb_conv2d_dgrad(const mnb_conv_shape* s, const float* dy, const float* wq, const uint32_t* pass_bits,
                     const mnb_act_qparams* qp, float* dx, mnb_stream_t stream);
/* dWq = corr(Xq, dY); Xq given as codes (+offset, *a_scale) or fp32.  scratch >= mnb_wgrad_scratch_bytes. */
int64_t mnb_wgrad_scratch_bytes(const mnb_conv_shape* s);
int mnb_conv2d_wgrad(const mnb_conv_shape* s, const float* dy, const mnb_conv_operands* op, float* dwq,
                     void* scratch, mnb_stream_t stream);
/* per-channel sums over (B, H, W) of a [B, C, HW] tensor:
 *   stats[0..C) = sum, stats[C..2C) = sum of squares (both accumulated in fp64, stored fp32 as
 *   mean and UNBIASED variance when `as_mean_var` != 0 — torch.mean / torch.var of IAO:854-855). */
int mnb_channel_stats(const float* x, int32_t batch, int32_t channels, int32_t hw, int32_t as_mean_var,
                      float* stats, void* scratch, mnb_stream_t stream);
/* backward of (mean, var):  dx = dmean/N + dvar * 2 (x - mean)/(N-1) */
int mnb_channel_stats_bwd(const float* x, const float* mean, const float* dmean, const float* dvar,
                          int32_t batch, int32_t channels, int32_t hw, float* dx, mnb_stream_t stream);

/* Producer-side fusions of a wbwtab block (SURVEY.md 8 f2):
 *   conv -> nn.BatchNorm2d -> ActivationQuantizer(A=2) [-> nn.MaxPool2d] -> channel_shuffle -> next conv
 * (nin_gc.py:9-21 shuffle, :53-59 block, WB:79-94 binarizer).
 *
 * mnb_bn_sign_fwd / _bwd replace BatchNorm2d + binarizer:
 *   fwd : y = sign(gamma (x - mean) invstd + beta), 0 -> +1; pass bit = |bn| < 1 (saturate STE)
 *   bwd : training-mode batch-norm backward of the masked gradient (dgamma, dbeta, dx); `training` = 0
 *         uses fixed statistics (dx = gamma invstd g pass).  dx_channel_sum (may be NULL) receives
 *         sum_{b,h,w} dx per channel: the bias gradient of the convolution that produced x.
 * mean / invstd come from mnb_channel_stats(as_mean_var = 2: mean, biased var, unbiased var).
 *
 * out_shuffle_groups = sg > 1 folds the NEXT block's channel shuffle into the producer: the output is
 * written as out[:, a*sg + b] = result[:, b*(C/sg) + a] and the incoming gradient is read through the same
 * permutation; pass bits / argmax stay in the producer's own channel order.  sg = 1: no permutation.   */
/* nn.BatchNorm2d's training-mode statistics in one launch: mean_invstd[0..C) = batch mean,
 * mean_invstd[C..2C) = 1/sqrt(biased var + eps); running_mean / running_var are updated in place with `momentum`
 * (unbiased variance, torch semantics) and *num_batches_tracked (may be NULL) is incremented.              */
int mnb_bn_batch_stats(const float* x, int32_t batch, int32_t channels, int32_t hw, double eps, double momentum,
                       float* running_mean, float* running_var, int64_t* num_batches_tracked, float* mean_invstd,
                       void* scratch, mnb_stream_t stream);
int mnb_bn_sign_fwd(const float* x, int32_t batch, int32_t channels, int32_t hw, const float* mean, const float* invstd,
                    const float* gamma, const float* beta, int32_t out_shuffle_groups, float* y, uint32_t* pass_bits,
                    mnb_stream_t stream);
/* training: 1 batch statistics, 0 running statistics, 2 = reduce pass only (dgamma / dbeta; the caller applies them with
 * mnb_bn_sign_bwd_pack, which writes dx as a packed operand) */
int mnb_bn_sign_bwd(const float* g, const uint32_t* pass_bits, const float* x, int32_t batch, int32_t channels, int32_t hw,
                    const float* mean, const float* invstd, const float* gamma, int32_t training,
                    int32_t out_shuffle_groups, float* dx, float* dgamma, float* dbeta, float* dx_channel_sum,
                    void* scratch, mnb_stream_t stream);

/* BatchNorm2d + binarizer + nn.MaxPool2d(2, 2) in one pass (the block before a 2x2 pool: nin_gc.py:84-85, :88-89): the
 * full-resolution +-1 tensor and the un-pooled gradient are never materialised.  y / g: [B, C, H/2, W/2] (through the
 * output permutation), pass_bits: B*C*H*W bits, argmax: B*C*(H/2)*(W/2) bytes (window index, ATen's first-maximum
 * rule).  Needs even H and W % 8 == 0, else MNB_E_UNSUPPORTED (run mnb_bn_sign_* and mnb_maxpool2d_* instead).   */
int mnb_bn_sign_pool_fwd(const float* x, int32_t batch, int32_t channels, int32_t H, int32_t W, const float* mean,
                         const float* invstd, const float* gamma, const float* beta, int32_t out_shuffle_groups, float* y,
                         uint32_t* pass_bits, uint8_t* argmax, mnb_stream_t stream);
int mnb_bn_sign_pool_bwd(const float* g, const uint32_t* pass_bits, const uint8_t* argmax, const float* x, int32_t batch,
                         int32_t channels, int32_t H, int32_t W, const float* mean, const float* invstd, const float* gamma,
                         int32_t training, int32_t out_shuffle_groups, float* dx, float* dgamma, float* dbeta,
                         float* dx_channel_sum, void* scratch, mnb_stream_t stream);

/* nn.MaxPool2d (square kernel <= 15, dilation 1, floor mode; nin_gc.py:85,89 / nin.py pools) with a one-byte
 * window index per output instead of int64 indices.  Same first-maximum tie rule and gradient accumulation
 * order as ATen, so results are bit-identical.  argmax: batch*channels*OH*OW bytes.                   */
int mnb_maxpool2d_fwd(const float* x, int32_t batch, int32_t channels, int32_t H, int32_t W, int32_t kernel, int32_t stride,
                      int32_t pad, int32_t out_shuffle_groups, float* y, uint8_t* argmax, mnb_stream_t stream);
int mnb_maxpool2d_bwd(const float* g, const uint8_t* argmax, int32_t batch, int32_t channels, int32_t H, int32_t W,
                      int32_t kernel, int32_t stride, int32_t pad, int32_t out_shuffle_groups, float* dx,
                      mnb_stream_t stream);

/* mnb_bn_sign_fwd that additionally writes its +-1 output as the bf16 operand plane of the packed-operand tensor-core
 * family (below): x_packed = bf16 [B][C/8][H][W][8] in the OUTPUT channel order (B*C*H*W*2 bytes, 16-byte aligned); needs
 * C % 8 == 0 and H*W % 32 == 0, else MNB_E_UNSUPPORTED.  y may be NULL (the consumer reads only the plane).           */
int mnb_bn_sign_fwd_packed(const float* x, int32_t batch, int32_t channels, int32_t hw, const float* mean,
                           const float* invstd, const float* gamma, const float* beta, int32_t out_shuffle_groups, float* y,
                           uint32_t* pass_bits, void* x_packed, mnb_stream_t stream);

/* fp32 convolution with few input channels on the tensor-core path: the un-quantized first layer of the QAT
 * models (plain nn.Conv2d in the reference: nin_gc.py:82, nin.py:60, resnet.py first conv; WB:300-317 leaves it
 * unquantized).  im2col operand built in shared memory, exact 3-piece bf16 split of both fp32 operands, the six
 * leading piece products accumulated in fp32 (error <= 2^-23 relative, i.e. that of an fp32 convolution).
 * Cover: groups 1, stride 1, dilation 1, 'same' odd square filter, C*R*S <= 128, Cout <= 256, 128 % W == 0,
 * (H*W) % 128 == 0; anything else returns MNB_E_UNSUPPORTED (-2).
 *   fwd   : y = conv2d(x, w) + bias (bias may be NULL)
 *   wgrad : dw = corr(x, dy);  scratch >= mnb_fconv2d_wgrad_tc_scratch_bytes(s) (-1: unsupported)        */
int mnb_fconv2d_fwd_tc(const mnb_conv_shape* s, const float* x, const float* w, const float* bias, float* y,
                       int32_t* err_flag, mnb_stream_t stream);
int64_t mnb_fconv2d_wgrad_tc_scratch_bytes(const mnb_conv_shape* s);
int mnb_fconv2d_wgrad_tc(const mnb_conv_shape* s, const float* dy, const float* x, float* dw, void* scratch,
                         int32_t* err_flag, mnb_stream_t stream);

/* ------------------------------------------------------------------------
 * Packed-operand ("pk") tensor-core family (mnb_pk.cu): every conv geometry of the QAT models on tcgen05 - weights
 * streamed per K-chunk, N / W tiling, stride 1 and 2 (space-to-depth), any filter with <= 64 taps.  Same math as
 * F.conv2d of the fake-quantized tensors (WB:186, DF:113, IAO:498/843/947) and ATen convolution_backward.
 *
 * Operands are bf16 "term planes"  pk[t][b][ceil(C/8)][h][w][8] : t = 0..T-1 exact pieces of an fp32 value
 * (x = p0 + p1 + p2, 8 significand bits each) or ONE plane of exact integer levels.
 *   mnb_pk_pack_act   : fp32 NCHW -> term planes.  qp != NULL: fake-quantize (DF:36-46 / IAO:214-240 / WB:11-36), planes
 *                       hold the integer level e (value = e * scale), bits8[b][c/8][h][w] bit j = STE pass flag of channel
 *                       8*(c/8)+j.  qp == NULL: exact split of x (* ch_scale[c] when given).  phase_split: the four
 *                       (h%2, w%2) planes become channel octets (h%2*2 + w%2)*ceil(C/8) + c/8 of an [H/2, W/2] tensor
 *                       (the form a stride-2 consumer reads).  out_pk: mnb_pk_act_bytes() bytes, 16-byte aligned.
 *   mnb_pk_pack_weight: w_int (i16 levels) or w_f32 [K, C/g, R, S] -> the bf16 operand image of (shape, mode);
 *                       mode 0 forward, 1 data gradient.  kzero[k] == 0 zeroes channel k (dgrad of a zero-scale channel).
 *                       w_img: mnb_pk_wimage_bytes() bytes.  terms_a / terms_w must match the later mnb_pk_conv call.
 *   mnb_pk_conv       : mode 0: y = bias + (a_scale * n_scale[n]) * conv2d(A, W);  mode 1: dx = STE(conv_transpose(A = dy, W)),
 *                       bits8 / gain: STE mask of the quantizer that fed the forward conv and its gradient factor (0.1 DoReFa).
 *                       a_scale: device scalar or NULL (then a_scale_const); n_scale NULL = 1.
 *   mnb_pk_wgrad      : dw[k][c][r][s] = (a_scale / kdiv[k]) * corr(x, dy); kdiv = the ch_scale dy_pk was packed with.
 * All return MNB_E_UNSUPPORTED (nothing launched) outside the cover (dilation, > 64 taps, odd sizes with stride 2, ...).
 * ---------------------------------------------------------------------- */
int64_t mnb_pk_act_bytes(int32_t batch, int32_t channels, int32_t h, int32_t w, int32_t terms);
int mnb_pk_pack_act(const float* x, int32_t batch, int32_t channels, int32_t h, int32_t w, const mnb_act_qparams* qp,
                    int32_t terms, const float* ch_scale, int32_t phase_split, void* out_pk, uint8_t* bits8,
                    mnb_stream_t stream);
/* BatchNorm2d + ReLU + DoReFa activation quantizer (DF:36-46) of the NEXT conv + operand packing in one pass (the DoReFa
 * block conv -> nn.BatchNorm2d -> nn.ReLU -> [channel_shuffle] -> QuantConv2d, nin_gc.py:53-59): x_packed = that conv's packed
 * bf16 level plane [B][C/8][H][W][8] in the output channel order of the folded shuffle; pass_bits = relu'(bn) * [0.1 bn <= 1]
 * as flat NCHW bits in the producer's own channel order (what mnb_bn_sign_bwd consumes for the backward pass).
 * Needs C % 8 == 0 and H*W % 32 == 0, else MNB_E_UNSUPPORTED. */
int mnb_bn_relu_quant_pack_fwd(const float* x, int32_t batch, int32_t channels, int32_t hw, const float* mean,
                               const float* invstd, const float* gamma, const float* beta, const mnb_act_qparams* qp,
                               int32_t out_shuffle_groups, void* x_packed, uint32_t* pass_bits, mnb_stream_t stream);
/* Second pass of mnb_bn_sign_bwd for a producing conv that runs on the packed-operand family (nn.BatchNorm2d backward +
 * saturate STE of WB:11-36, after dgamma / dbeta were reduced): writes  dx * ch_scale[c]  (ch_scale NULL: dx) as `terms`
 * exact bf16 pieces in the plane layout of mnb_pk_pack_act - the dy operand of that conv's mnb_pk_conv (mode 1) and
 * mnb_pk_wgrad (kdiv = ch_scale) - and, when dx != NULL, plain fp32 dx.  Training-mode statistics only.  channels % 8 == 0. */
int mnb_bn_sign_bwd_pack(const float* g, const uint32_t* pass_bits, const float* x, int32_t batch, int32_t channels, int32_t hw,
                         const float* mean, const float* invstd, const float* gamma, const float* dgamma, const float* dbeta,
                         int32_t out_shuffle_groups, const float* ch_scale, int32_t terms, float* dx, void* dy_packed,
                         mnb_stream_t stream);
/* The same for a producer with the 2x2 max-pool folded in: second pass of mnb_bn_sign_pool_bwd (call that one with
 * training = 2 first: reduce pass only, dgamma / dbeta) writing the full-resolution gradient [batch, channels, H, W] as the
 * producing conv's packed operand.  argmax / pass_bits as written by mnb_bn_sign_pool_fwd; g is the pooled gradient
 * [batch, channels, H/2, W/2] in the shuffled order.  Needs even H, W % 8 == 0, channels % 8 == 0.                  */
int mnb_bn_sign_pool_bwd_pack(const float* g, const uint32_t* pass_bits, const uint8_t* argmax, const float* x, int32_t batch,
                              int32_t channels, int32_t H, int32_t W, const float* mean, const float* invstd,
                              const float* gamma, const float* dgamma, const float* dbeta, int32_t out_shuffle_groups,
                              const float* ch_scale, int32_t terms, void* dy_packed, mnb_stream_t stream);
/* mnb_pk_pack_act with a preceding nn.ReLU folded in (relu != 0: x is clamped at 0 before it is quantized / split) */
int mnb_pk_pack_act_relu(const float* x, int32_t batch, int32_t channels, int32_t h, int32_t w, const mnb_act_qparams* qp,
                         int32_t terms, const float* ch_scale, int32_t phase_split, int32_t relu, void* out_pk,
                         uint8_t* bits8, mnb_stream_t stream);
int mnb_pk_conv_plan(const mnb_conv_shape* s, int32_t mode, int32_t terms_a, int32_t terms_w, int32_t* out16); /* host only */
int64_t mnb_pk_wimage_bytes(const mnb_conv_shape* s, int32_t mode, int32_t terms_a, int32_t terms_w);
int mnb_pk_pack_weight(const mnb_conv_shape* s, int32_t mode, int32_t terms_a, int32_t terms_w, const int16_t* w_int,
                       const float* w_f32, const float* kzero, void* w_img, mnb_stream_t stream);
int mnb_pk_conv(const mnb_conv_shape* s, int32_t mode, const void* a_pk, int32_t terms_a, const void* w_img, int32_t terms_w,
                const float* n_scale, const float* a_scale, float a_scale_const, const float* bias, const uint8_t* bits8,
                float gain, float* out, int32_t* err_flag, mnb_stream_t stream);
/* Inference graphs with frozen quantizers (BASELINE.json configs[4], iao/main.py:511-519: eval forward of a calibrated model):
 * the producer writes the operand plane of its consumer, so the fp32 activation between two quantized convs is neither
 * written nor re-read nor packed in a separate pass.
 *   mnb_pk_conv_post        : forward conv (mode 0 of mnb_pk_conv) whose epilogue also computes
 *                             level = Q_consumer([ReLU](y)) (IAO:214-240 / DF:36-46 of the NEXT layer's activation quantizer)
 *                             and stores it as that layer's bf16 plane; out may be NULL (plane only).
 *   mnb_quant_add_pack_fwd  : IAO QuantAdd (IAO:1441-1498: out = Q(a) + Q(b) [-> ReLU]) that additionally quantizes its
 *                             result for the consuming conv and writes that conv's plane (a, b, out: fp32 [B, C, H, W]).
 * phase_split: the consumer is a stride-2 conv (space-to-depth plane order of mnb_pk_pack_act). */
typedef struct mnb_pk_post {
  const mnb_act_qparams* q; /* the consumer's activation quantizer, 2..8 bits, DoReFa or IAO */
  int32_t relu;             /* an nn.ReLU sits between producer and consumer */
  int32_t phase_split;
  void* out_pk;             /* mnb_pk_act_bytes(B, C_out, OH, OW, 1) bytes, 16-byte aligned */
} mnb_pk_post;
int mnb_pk_conv_post(const mnb_conv_shape* s, const void* a_pk, int32_t terms_a, const void* w_img, int32_t terms_w,
                     const float* n_scale, const float* a_scale, float a_scale_const, const float* bias, float* out,
                     const mnb_pk_post* post, int32_t* err_flag, mnb_stream_t stream);
int mnb_quant_add_pack_fwd(const float* a, const float* b, int32_t batch, int32_t channels, int32_t h, int32_t w,
                           const mnb_act_qparams* qp, int32_t relu, float* out, const mnb_pk_post* post, mnb_stream_t stream);
int64_t mnb_pk_wgrad_scratch_bytes(const mnb_conv_shape* s, int32_t terms_dy, int32_t terms_x);
int mnb_pk_wgrad(const mnb_conv_shape* s, const void* dy_pk, int32_t terms_dy, const void* x_pk, int32_t terms_x,
                 const float* a_scale, const float* kdiv, float* dw, void* scratch, int32_t* err_flag, mnb_stream_t stream);

/* ------------------------------------------------------------------------
 * Bit-packed XNOR-popcount forward for wbwtab layers (mnb_xnor.cu): binary activations (WB:11-36, sign with 0 -> +1)
 * times binary / ternary weights (WB:40-75, 98-146) as sum = popc(N) - 2 popc(N & (A ^ S)) on 1-bit planes; the integer
 * sum is exact, y = fmaf(sum, alpha[k], bias[k]) equals mnb_pk_conv's result bit for bit.  Forward only (the gradients
 * of a QAT step multiply real-valued dy).  functional.py picks it per layer from the measured table of
 * profiles/r2_xnor_vs_tc.md (north_star: "picked when ncu shows it beating the tensor-core path").
 *   a_bits : u32 [B][G][ceil(C/g / 32)][H][W], bit j of word n = [x[b][g*C/g + 32 n + j][h][w] is not < 0]
 *   w_img  : mnb_xnor_wimage_bytes() bytes, built from the i16 levels {-1, 0, +1} [K][C/g][R][S] of mnb_wb_weight_fwd
 * Cover: square filter 1/3/5, equal strides / pads, dilation 1, C/g <= 128 (3x3), <= 64 (5x5), <= 256 (1x1); else
 * MNB_E_UNSUPPORTED (mnb_xnor_supported: 1 / 0).                                                                      */
int mnb_xnor_supported(const mnb_conv_shape* s);
int64_t mnb_xnor_act_bytes(int32_t batch, int32_t channels, int32_t h, int32_t w, int32_t groups);
int mnb_xnor_pack_act(const float* x, int32_t batch, int32_t channels, int32_t h, int32_t w, int32_t groups, void* out_bits,
                      mnb_stream_t stream);
int64_t mnb_xnor_wimage_bytes(const mnb_conv_shape* s);
int mnb_xnor_pack_weight(const mnb_conv_shape* s, const int16_t* w_int, void* w_img, mnb_stream_t stream);
int mnb_xnor_conv_fwd(const mnb_conv_shape* s, const void* a_bits, const void* w_img, const float* alpha, const float* bias,
                      float* y, mnb_stream_t stream);

/* Optimizer step of the QAT loop (torch.optim.Adam semantics, L2 weight decay, no amsgrad;
 * wbwtab/main.py:84,331-339) over one flat fp32 parameter / gradient bucket: a single launch. */
int mnb_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int32_t step, mnb_stream_t stream);

/* ------------------------------------------------------------------------
 * Hardware self-tests of the sm_100a building blocks (run by tests/test_gpu_tc_selftest.py).
 * Bounded waits: a wrong descriptor sets *err_flag (device int) instead of hanging the GPU.
 * ---------------------------------------------------------------------- */
/* D[128 x N] = A[128 x K] * B[N x K]^T through tcgen05.mma (kind::f16 on bf16, or kind::i8) with
 * thread-written no-swizzle operands; A/B/D are fp32 row-major device arrays.
 * int8: 0 = bf16 K-major operands, 1 = int8 K-major, 2 = bf16 MN-major (the wgrad kernel's form).    */
int mnb_selftest_umma(const float* A, const float* B, float* D, int32_t N, int32_t K, int32_t int8,
                      int32_t* err_flag, mnb_stream_t stream);
/* one cp.async.bulk.tensor.3d box (dims/box/coord innermost-first, fp32) copied to `out`;
 * elements outside the tensor must read back as 0.                                              */
int mnb_selftest_tma3d(const float* src, const int64_t* dims3_host, const int32_t* box3_host,
                       const int32_t* coord3_host, float* out, int32_t* err_flag, mnb_stream_t stream);

/* micro-benchmark: `iters` back-to-back M128 x N x K16 bf16 MMAs from one thread over n_acc accumulators;
 * out2[0] = cycles until all have retired, out2[1] = cycles spent issuing.                         */
int mnb_selftest_mma_rate(int32_t N, int32_t n_acc, int32_t a_shift16, int32_t iters, int32_t mn_major,
                          int64_t* out2, int32_t* err_flag, mnb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MICRONET_B200_H */
