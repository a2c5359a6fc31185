/*
 * rehrseg_b200 -- C-ABI of the B200 (sm_100a) hot-path library `librehrseg_b200.so`.
 *
 * The reference (zhiyuns/REHRSeg) has no FFI of its own: every heavy op is a torch.nn / ATen / numpy
 * library call.  Each entry point below therefore names the reference *call site* it replaces
 * (file:line relative to the reference root).  The Python host layer (rehrseg_b200/*.py) binds these
 * with ctypes and re-exposes them as nn.Module / autograd.Function drop-ins.
 *
 * Conventions
 *  - All pointers are DEVICE pointers owned by the caller (PyTorch caching allocator); the library never
 *    allocates, frees or synchronises.  Every call is enqueued on `stream` and returns immediately.
 *  - Activations are channels-last ("NDHWC") tensors described by rehr_tensor: logical dims n,d,h,w,c and a
 *    voxel pitch `ld` (elements between consecutive voxels, >= c) so channel slices of a concat buffer can be
 *    passed without a copy.  bf16 unless the name says f32.
 *  - Return value: 0 = OK, negative = rehr_status.  rehr_strerror() translates.  No exceptions cross the ABI.
 *  - Thread-safe for concurrent calls on distinct streams (no hidden mutable state except a cached driver
 *    entry point and SM count).
 */
#ifndef REHRSEG_B200_H_
#define REHRSEG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* rehr_stream; /* cudaStream_t */

typedef enum {
  REHR_OK = 0,
  REHR_BAD_SHAPE = -1,      /* inconsistent dims between operands */
  REHR_UNSUPPORTED = -2,    /* configuration outside what the kernels implement */
  REHR_WORKSPACE = -3,      /* workspace too small */
  REHR_CUDA_ERROR = -4,     /* a CUDA runtime / driver call failed (see rehr_last_cuda_error) */
  REHR_BAD_ALIGNMENT = -5   /* pointer / pitch not aligned as required (16 B) */
} rehr_status;

/* 16-bit storage format of an activation tensor.  Gradients and FLAVR activations are bf16; the SegModel forward stores its
 * activations and pre-normalisation conv outputs in fp16 (InstanceNorm bounds them; 3 more mantissa bits bring the logits from
 * 9e-3 to 1e-3 of the fp32 reference at the same tensor-core rate), see DESIGN.md section 4.  A tcgen05.mma needs both operands
 * in ONE format: the packed weights of a forward conv must be packed in the format of its input tensor. */
typedef enum { REHR_BF16 = 0, REHR_F16 = 1 } rehr_dtype;

typedef struct {
  void* ptr;
  int n, d, h, w, c;
  long long ld; /* voxel pitch in elements */
  int dtype;    /* rehr_dtype of the 16-bit payload (ignored where an entry point says f32) */
} rehr_tensor;

/* A 3-D convolution "A <- B": weight Wc[A][B][kd][kh][kw], out[o] = sum_k Wc[k] . in[o*s + k - p].
 * ConvTranspose3d (weight [Cin][Cout][k]) is the same object read backwards: its forward is
 * rehr_conv3d_dgrad, its input-gradient is rehr_conv3d_fwd, its weight-gradient is rehr_conv3d_wgrad
 * with the operands swapped (see rehr_convtranspose3d_* below). */
typedef struct {
  int kd, kh, kw; /* kernel  */
  int sd, sh, sw; /* stride  (1 or 2 per dim) */
  int pd, ph, pw; /* padding */
} rehr_conv_desc;

typedef enum { REHR_ACT_NONE = 0, REHR_ACT_RELU = 1, REHR_ACT_LRELU = 2 } rehr_act;

const char* rehr_strerror(int status);
int rehr_last_cuda_error(void);     /* cudaError_t of the last failing CUDA call on this thread */
int rehr_version(void);             /* ABI version, currently 6 (4: rehr_tensor.dtype, dtype arguments of the weight packers; 5: batched
                                     * re-pack and fused InstanceNorm-backward sums added -- additive; 6: the normalise-on-load and fused
                                     * InstanceNorm-backward-sum entry points removed; the rehr_intensity_* and rehr_sr_loss_* entry
                                     * points were added later without a bump -- additive) */
int rehr_device_sm_count(void);

/* ------------------------------------------------------------------------------------------------
 * Dense convolution engine (tcgen05 / TMEM implicit GEMM, TMA-staged NDHWC bf16 tiles).
 * Replaces: torch.nn.Conv3d / ConvTranspose3d / Conv2d forward+backward as called by
 *   dynamic_network_architectures ConvDropoutNormReLU.conv (built at models/seg_model.py:174-191),
 *   UNetDecoder.transpconvs (models/seg_model.py:36), sr_head (models/seg_model.py:197-199),
 *   FLAVR Conv3DSimple / Conv_3d / upConv3D / Conv_2d (models/FLAVR/resnet_3D.py:19-33,
 *   models/FLAVR/FLAVR_arch.py:24-88).
 * ---------------------------------------------------------------------------------------------- */

/* Repack fp32 weights src[(r*sr + c*sc + t*st)] into 16-bit dst[r][t][c] (the K-major GEMM operand), dtype = rehr_dtype
 * of the packed copy: it must equal the dtype of the activation tensor the GEMM contracts it with.
 *   fwd   of Wc[A][B][T]: R=A, C=B, sr=B*T, sc=T, st=1
 *   dgrad of Wc[A][B][T]: R=B, C=A, sr=T,   sc=B*T, st=1 */
int rehr_pack_weight(const float* src, void* dst16, int R, int C, int T, long long sr, long long sc,
                     long long st, int dtype, rehr_stream stream);

/* y[A] = act(conv(x[B]) + bias).  w_packed = bf16 [A][T][B].  bias may be NULL.  y may be bf16 or f32.
 * stats (optional, f32 [rehr_conv3d_stats_tiles()][A][2]) receives per-output-tile (sum, sum of squares)
 * of the *pre-activation* outputs for the fused InstanceNorm statistics; only legal when
 * rehr_conv3d_stats_tiles() > 0 (every tile lies inside one sample). */
int rehr_conv3d_fwd(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                    const rehr_tensor* y, int y_is_f32, int act, float slope, float* stats,
                    rehr_stream stream);
/* Number of per-sample stat tiles rehr_conv3d_fwd will write for an output of this shape (0 = not fusable). */
int rehr_conv3d_stats_tiles(const rehr_tensor* y);

/* dx[B] = act(conv_transpose(dy[A]) + bias).  w_packed = bf16 [B][T][A].  (bias/act are used when this
 * runs as the *forward* of a ConvTranspose3d; pass NULL / REHR_ACT_NONE for a plain input-gradient.) */
int rehr_conv3d_dgrad(const rehr_conv_desc* desc, const rehr_tensor* dy, const void* w_packed,
                      const float* bias, const rehr_tensor* dx, int dx_is_f32, int act, float slope,
                      rehr_stream stream);

/* Split-K variants of the two calls above for layers with fewer output tiles than SMs (the <= 8^3 bottleneck stages would
 * otherwise stream megabytes of weights and taps through one or two SMs): the K loop is shared by several CTAs through an
 * fp32 scratch buffer and a second small kernel sums the partials and runs the epilogue.  rehr_conv3d_splitk_workspace(desc,
 * src, w_packed, dst, is_dgrad) returns the scratch bytes (0 = the layer does not split; then ws may be NULL). */
size_t rehr_conv3d_splitk_workspace(const rehr_conv_desc* desc, const rehr_tensor* src, const void* w_packed,
                                    const rehr_tensor* dst, int is_dgrad);
int rehr_conv3d_fwd_ws(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                       const rehr_tensor* y, int y_is_f32, int act, float slope, float* stats, void* ws, size_t ws_bytes,
                       rehr_stream stream);
int rehr_conv3d_dgrad_ws(const rehr_conv_desc* desc, const rehr_tensor* dy, const void* w_packed, const float* bias,
                         const rehr_tensor* dx, int dx_is_f32, int act, float slope, void* ws, size_t ws_bytes,
                         rehr_stream stream);

/* dW[A][B][T] (f32, PyTorch layout) = sum_o dy[o,A] (x) x[o*s+k-p, B].  Split-K partials go to `ws`. */
size_t rehr_conv3d_wgrad_workspace(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy);
int rehr_conv3d_wgrad(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy, float* dw,
                      int accumulate, void* ws, size_t ws_bytes, rehr_stream stream);

/* ConvTranspose3d views of the same engine (weight [Cin][Cout][T]). */
int rehr_convtranspose3d_fwd(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed /*[Cout][T][Cin]*/,
                             const float* bias, const rehr_tensor* y, int act, float slope, rehr_stream stream);
/* kernel == stride, padding 0 (the nnU-Net decoder up-sampling): ONE GEMM with N = classes x Cout and a scatter epilogue.
 * w_packed = bf16 [T][Cout][Cin] (rehr_pack_weight with R = T, C = Cin, T = Cout, sr = 1, sc = Cout*T, st = T).
 * y may be a channel slice of a wider concat buffer (ld > c). */
int rehr_convtranspose3d_fused_supported(const rehr_conv_desc* desc, int cin, int cout);
int rehr_convtranspose3d_fused_fwd(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                                   const rehr_tensor* y, int act, float slope, rehr_stream stream);
/* Same, and a second copy y2 of the result (same shape; its own buffer, pitch and 16-bit format) written by the same epilogue: the
 * bf16 twin of the fp16 up-sampled half of [up | skip] that the weight gradient of the decoder conv contracts with bf16 gradients. */
int rehr_convtranspose3d_fused_fwd2(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                                    const rehr_tensor* y, const rehr_tensor* y2, int act, float slope, rehr_stream stream);
int rehr_convtranspose3d_dgrad(const rehr_conv_desc* desc, const rehr_tensor* dy, const void* w_packed /*[Cin][T][Cout]*/,
                               const rehr_tensor* dx, rehr_stream stream);
size_t rehr_convtranspose3d_wgrad_workspace(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy);
int rehr_convtranspose3d_wgrad(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy, float* dw,
                               int accumulate, void* ws, size_t ws_bytes, rehr_stream stream);

/* "Marching" kernel for cubic kernels ks = 3 or 5, stride 1, pad (ks-1)/2, with few input channels (Cin in {16,32,64,128}
 * for ks = 3, Cin = 16 for ks = 5; any Cout): the halo'd input plane is TMA-loaded ONCE into a shared-memory ring and the
 * ks^3 taps become UMMA descriptor offsets / a kd-fused N = ks*Ct MMA (see csrc/conv_march.cu).  Same call sites as
 * rehr_conv3d_fwd (and sr_head.2, the 5x5x5 16->2 conv of models/seg_model.py:199); it needs its own packed weights.
 *   rehr_pack_weight_march: dst bf16 (rehr_conv3d_march_weight_bytes) from fp32 src[co*s_co + ci*s_ci + t], T = ks^3:
 *     forward of W[Cout][Cin][T]: cout, cin, s_co = Cin*T, s_ci = T, flip = 0
 *     input-gradient dx[B] <- dy[A] of W[A][B][T]: cout := B, cin := A, s_co = T, s_ci = B*T, flip = 1
 *   rehr_conv3d_march_fwd: y = act(conv(x) + bias); stats (optional) = f32 [n][rehr_conv3d_march_stats_tiles][cout][2].
 * Planar layers -- k = (1,3,3), stride 1, pad (0,1,1): the thick-slice stages of anisotropic nnU-Net plans (the kernel_sizes
 * argument of SegModel, models/seg_model.py:154-173) -- run through the same kernel restricted to the centre depth tap; they are
 * selected by passing the kernel's DEPTH extent ks = 1 to the functions below (T = 9, weights W[Cout][Cin][9]). */
int rehr_conv3d_march_supported(const rehr_conv_desc* desc, int cin, int cout);
size_t rehr_conv3d_march_weight_bytes(int cin, int cout, int ks);
int rehr_pack_weight_march(const float* src, void* dst16, int cout, int cin, int ks, long long s_co, long long s_ci, int flip,
                           int dtype, rehr_stream stream);
int rehr_conv3d_march_stats_tiles(const rehr_tensor* x, const rehr_tensor* y, int ks);
int rehr_conv3d_march_fwd(const rehr_tensor* x, const void* w_march, const float* bias, const rehr_tensor* y, int ks, int y_is_f32,
                          int act, float slope, float* stats, rehr_stream stream);
/* Batched weight re-pack (csrc/pack_batch.cu).  Between rehr_pack_batch_begin() and rehr_pack_batch_launch() every
 * rehr_pack_weight / rehr_pack_weight_march / rehr_pack_weight_march_s2dgrad call ON THIS THREAD is recorded instead of launched;
 * rehr_pack_batch_launch issues all of them as ONE kernel (one per 128 recorded calls) whose job table travels in the kernel
 * parameters -- no upload, capturable in a CUDA graph; results are bit-identical to the individual launches.  Replaces the ~57
 * per-parameter repacks a training step does after optimizer.step() (the reference has no counterpart: cuDNN reads
 * the fp32 NCDHW weights directly, train_all.py:553-555).  rehr_pack_batch_abort drops a recording without launching. */
int rehr_pack_batch_begin(void);
int rehr_pack_batch_launch(rehr_stream stream);
int rehr_pack_batch_abort(void);

/* fp16 saturation check (opt-in; csrc/ptx.cuh range_check).  rehr_range_sink(slots, slot) makes every later fp16 activation
 * store launched ON THIS THREAD by the conv forward (tapped, marching, small-Cin / tensor-core stem, the transposed-conv scatter
 * and the bias-only class fill), rehr_instnorm_lrelu_apply, rehr_upsample_linear_d and rehr_convert16 count into slots[slot]:
 * 16 bytes per slot, { uint64 count; uint32 max_abs_bits; uint32 pad }.  A value v saturates when !(|v| < 65520) (it rounds to
 * +-inf or is NaN; the store still writes +-65504 or NaN, bit-identical to an unchecked run); max_abs_bits is the largest
 * |v| of the saturated values as fp32 bits (atomicMax: NaN sorts above inf).  bf16 and fp32 stores are not checked.
 * slots == NULL turns the sink off: the kernels then take a null slot and check nothing.  The pointer is baked into the
 * launches, so a captured CUDA graph keeps writing to it on replay.  rehr_range_clear zeroes n slots with one memset. */
int rehr_range_sink(void* slots, int slot);
int rehr_range_clear(void* slots, int n, rehr_stream stream);

/* Input gradient of a k3 / pad 1 conv with strides in {1, 2} (the nnU-Net stage-entry convs) through the marching kernel:
 * every output parity class of dx is a stride-1 correlation over dy with 1 or 2 taps per strided dimension, written in place
 * at (2i + r).  w = conv weight f32 [Cout][Cin][27]; cin / cout are the CONV's channel counts. */
int rehr_conv3d_march_s2dgrad_supported(const rehr_conv_desc* desc, int cin, int cout);
size_t rehr_conv3d_march_s2dgrad_weight_bytes(const rehr_conv_desc* desc, int cin, int cout);
int rehr_pack_weight_march_s2dgrad(const rehr_conv_desc* desc, const float* w, void* dst_bf16, int cin, int cout,
                                   rehr_stream stream);
int rehr_conv3d_march_s2dgrad(const rehr_conv_desc* desc, const rehr_tensor* dy, const void* w_packed, const rehr_tensor* dx,
                              rehr_stream stream);

/* Marching weight-gradient kernel for cubic kernels ks = 3 or 5, stride 1, pad (ks-1)/2 (csrc/wgrad_march.cu): both
 * activations are TMA-loaded once per plane, the ks^3 taps are UMMA descriptor offsets / a kd-fused N = ks*PC MMA,
 * accumulators live in TMEM for the whole CTA.  Same call site as rehr_conv3d_wgrad.  dw = f32 [cout][x->c][ks^3] with
 * cout <= dy->c (dy may be zero-padded to a multiple of 16 channels).  ks = 3: channel counts multiples of 32 on one side
 * and of 16 on the other; ks = 5: 16 channels each (sr_head.2, models/seg_model.py:199).  ks = 1 selects the planar k = (1,3,3),
 * pad (0,1,1) layer (only the centre depth offset is accumulated; dw = f32 [cout][x->c][9]). */
int rehr_conv3d_wgrad_march_supported(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy);
size_t rehr_conv3d_wgrad_march_workspace(const rehr_tensor* x, const rehr_tensor* dy, int ks);
int rehr_conv3d_wgrad_march(const rehr_tensor* x, const rehr_tensor* dy, int ks, int cout, float* dw, int accumulate, void* ws,
                            size_t ws_bytes, rehr_stream stream);

/* Weight gradient of a k3 / pad 1 conv with strides in {1, 2}: one marching pass per parity class of X (a strided TMA view),
 * restricted to the 1-2 offsets per strided dimension that class contributes to; dw f32 [Cout][Cin][27]. */
int rehr_conv3d_wgrad_march_s2_supported(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy);
size_t rehr_conv3d_wgrad_march_s2_workspace(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy);
int rehr_conv3d_wgrad_march_s2(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy, float* dw, int accumulate,
                               void* ws, size_t ws_bytes, rehr_stream stream);

/* Direct convolution for tiny input-channel counts (Cin <= 4: the 1-channel nnU-Net stem, the 2-channel
 * FLAVR stem k(3,7,7)); x is NCDHW f32 exactly as the caller hands it (train_all.py:524), y NDHWC bf16.
 * w is the PyTorch f32 weight [Cout][Cin][kd][kh][kw]. */
int rehr_conv3d_smallcin_fwd(const rehr_conv_desc* desc, const float* x_ncdhw, int n, int cin, int d, int h, int w,
                             const float* weight, const float* bias, const rehr_tensor* y, int act, float slope,
                             float* stats, rehr_stream stream);
int rehr_conv3d_smallcin_wgrad(const rehr_conv_desc* desc, const float* x_ncdhw, int n, int cin, int d, int h, int w,
                               const rehr_tensor* dy, float* dw, int accumulate, void* ws, size_t ws_bytes,
                               rehr_stream stream);
size_t rehr_conv3d_smallcin_wgrad_workspace(const rehr_conv_desc* desc, int cin, const rehr_tensor* dy);
/* dx (NCDHW f32) for the small-Cin stem -- needed by FLAVR-as-student only; nnU-Net's first layer needs none. */
int rehr_conv3d_smallcin_dgrad(const rehr_conv_desc* desc, const rehr_tensor* dy, const float* weight,
                               float* dx_ncdhw, int n, int cin, int d, int h, int w, rehr_stream stream);

/* ------------------------------------------------------------------------------------------------
 * InstanceNorm3d(eps, affine) + LeakyReLU, HBM-bound vectorised kernels.
 * Replaces ConvDropoutNormReLU.norm / .nonlin (train_all.py:486-491).
 * ---------------------------------------------------------------------------------------------- */
/* Per-(n,c) sum / sum-of-squares of a bf16 tensor -> partial[(n*tiles + t)*C*2 ...]; use when the conv
 * epilogue could not fuse them.  tiles = rehr_instnorm_stats_tiles(x). */
int rehr_instnorm_stats_tiles(const rehr_tensor* x);
int rehr_instnorm_stats(const rehr_tensor* x, float* partial, rehr_stream stream);
/* partial [n][tiles][c][2] -> mean[n][c], rstd[n][c] (biased variance, double accumulation). */
int rehr_instnorm_finalize(const float* partial, int n, int tiles, int c, long long count, float eps,
                           float* mean, float* rstd, rehr_stream stream);
/* a = lrelu(gamma * (y - mean) * rstd + beta)   (slope = 1 -> no activation).  a2 (optional, may be NULL): a second copy of
 * the result in another 16-bit format / buffer, written in the same pass (the bf16 twin of an fp16 activation that the
 * weight-gradient GEMM of the consumer contracts with bf16 gradients). */
int rehr_instnorm_lrelu_apply(const rehr_tensor* y, const float* mean, const float* rstd, const float* gamma,
                              const float* beta, float slope, const rehr_tensor* a, const rehr_tensor* a2, rehr_stream stream);
/* Backward, two passes.  (1) reduce: partial[n][tiles][c][2] = (sum g, sum g*xhat), g = (da1 + da2) * lrelu'.
 * (2) apply: dy = gamma*rstd*(g - S1/V - xhat*S2/V).  da2 may be NULL (second gradient source of a skip). */
int rehr_instnorm_lrelu_bwd_reduce(const rehr_tensor* y, const rehr_tensor* da1, const rehr_tensor* da2,
                                   const float* mean, const float* rstd, const float* gamma, const float* beta,
                                   float slope, float* partial, rehr_stream stream);
int rehr_instnorm_lrelu_bwd_finalize(const float* partial, int n, int tiles, int c, const float* rstd,
                                     float* sums /*[n][c][2]*/, float* dgamma, float* dbeta, int accumulate,
                                     rehr_stream stream);
int rehr_instnorm_lrelu_bwd_apply(const rehr_tensor* y, const rehr_tensor* da1, const rehr_tensor* da2,
                                  const float* mean, const float* rstd, const float* gamma, const float* beta,
                                  float slope, const float* sums, const rehr_tensor* dy, rehr_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Small HBM-bound pieces of the two networks.
 * ---------------------------------------------------------------------------------------------- */
/* 1x1x1 conv to very few channels (seg_layers[-1], models/seg_model.py:44): y NCDHW f32 [n][cout][vox]. */
int rehr_pointwise_fwd(const rehr_tensor* x, const float* w /*[cout][cin]*/, const float* bias, float* y_ncdhw,
                       int cout, rehr_stream stream);
int rehr_pointwise_bwd(const rehr_tensor* x, const float* dy_ncdhw, const float* w, int cout,
                       const rehr_tensor* dx, float* dw, float* dbias, int accumulate, void* ws, size_t ws_bytes,
                       rehr_stream stream);
size_t rehr_pointwise_bwd_workspace(const rehr_tensor* x, int cout);
/* per-channel sum over all voxels of a bf16 tensor (bias gradients) */
int rehr_channel_sum(const rehr_tensor* x, float* out, int accumulate, void* ws, size_t ws_bytes, rehr_stream stream);
size_t rehr_channel_sum_workspace(const rehr_tensor* x);
/* F.interpolate(scale_factor=(s,1,1), mode='trilinear', align_corners=True) (models/seg_model.py:204) */
int rehr_upsample_linear_d(const rehr_tensor* x, const rehr_tensor* y, rehr_stream stream);
int rehr_upsample_linear_d_bwd(const rehr_tensor* dy, const rehr_tensor* dx, rehr_stream stream);
/* layout / dtype adapters at the model boundary (train_all.py:524 hands NCDHW f32) */
int rehr_ncdhw_f32_to_ndhwc_bf16(const float* src, const rehr_tensor* dst, rehr_stream stream);
int rehr_ndhwc_bf16_to_ncdhw_f32(const rehr_tensor* src, float* dst, rehr_stream stream);
/* dst = src converted between the two 16-bit storage formats (rehr_tensor.dtype of each side; pitched channel slices allowed) */
int rehr_convert16(const rehr_tensor* src, const rehr_tensor* dst, rehr_stream stream);
/* elementwise helpers for FLAVR blocks (models/FLAVR/resnet_3D.py:100-151, FLAVR_arch.py:169-248) */
int rehr_segate_scale_add_act(const rehr_tensor* x, const float* gate /*[n][c]*/, const rehr_tensor* residual,
                              int act, float slope, const rehr_tensor* y, rehr_stream stream);

/* Backward of the SE-gate tail y = act(x*gate[n,c] + residual) (resnet_3D.py:112-116,140-151).  With g = dy*act'(y):
 *   rehr_segate_bwd_reduce: partial[n][rehr_instnorm_stats_tiles(x)][c][2] = (sum_v g*x, 0)  (-> d gate, finalize with
 *                           rehr_instnorm_lrelu_bwd_finalize)
 *   rehr_segate_bwd_apply : dx = g*gate[n,c] + shift[n,c] (shift = gradient through the global average pool / V),
 *                           dres (optional) = g */
int rehr_segate_bwd_reduce(const rehr_tensor* x, const rehr_tensor* y, const rehr_tensor* dy, int act, float slope,
                           float* partial, rehr_stream stream);
int rehr_segate_bwd_apply(const rehr_tensor* y, const rehr_tensor* dy, int act, float slope, const float* gate,
                          const float* shift, const rehr_tensor* dx, const rehr_tensor* dres, rehr_stream stream);

/* dy = da * act'(.) evaluated from the activation OUTPUT a (ReLU, or LeakyReLU with slope > 0): the backward of the
 * bias+activation epilogues of rehr_conv3d_fwd / rehr_convtranspose3d_fwd (FLAVR_arch.py:86, resnet_3D.py:144-149). */
int rehr_act_bwd(const rehr_tensor* a, const rehr_tensor* da, int act, float slope, const rehr_tensor* dy,
                 rehr_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Sliding-window Gaussian blend (utils/seg_utils.py:240-287): fp16 accumulators exactly as the reference.
 *   logits[c, sl] += pred[c] * gauss ;  n_pred[sl] += gauss     (rehr_sw_accumulate)
 *   logits /= n_pred ; *inf_flag |= any(isinf(logits))          (rehr_sw_finalize)
 * logits [C][VD][VH][VW] f16, n_pred [VD][VH][VW] f16, pred [C][TD][TH][TW] f16 (or f32), gauss [TD][TH][TW] f16
 * (NULL = the reference's `gaussian = 1`).  npred_f16 may be NULL (blend the logits only).
 * ---------------------------------------------------------------------------------------------- */
int rehr_sw_accumulate(void* logits_f16, void* npred_f16, const void* pred, int pred_is_f32, const void* gauss_f16,
                       int C, int VD, int VH, int VW, int TD, int TH, int TW, int od, int oh, int ow,
                       rehr_stream stream);
int rehr_sw_finalize(void* logits_f16, const void* npred_f16, int C, long long voxels, int* inf_flag,
                     rehr_stream stream);

/* Blur degradation F.conv2d(x[Z,1,X,Y], k[1,1,L,1], padding="same") (utils/train_set.py:325,332;
 * utils/sr_utils.py:272,276,302): L-tap cross-correlation along X, zero padded, f32. */
int rehr_blur1d(const float* x, const float* taps, int L, float* y, long long Z, int X, int Y, rehr_stream stream);

/* UASR head of UNet_3D_3D (models/FLAVR/FLAVR_arch.py:203-227,244-246): softmax over `experts` (= 16) mixing weights per pixel and
 * output slice, img = sum p (tanh(o_img) + 1) / 2, seg = sum p o_seg, uncertainty = sigmoid(sum p w + b), forward and backward in
 * one pass each.  out_cl / ue_cl: the two fp32 channels-last conv outputs [batch * hw][n_out * 2 * experts] / [..][n_out * experts]
 * (feature_fuse1 / uncertainty_early); res f32 [batch][2][n_out][hw], unc f32 [batch][1][n_out][hw]; backward: d_res / d_unc (either
 * may be NULL) -> d_out_cl, d_ue_cl and per-block partial sums [rehr_uasr_mixture_blocks][experts + 1] of the uncertainty layer's
 * weight / bias gradients (the caller sums them). */
int rehr_uasr_mixture_blocks(long long pixels, int n_out);
int rehr_uasr_mixture_fwd(const float* out_cl, const float* ue_cl, const float* w, const float* b, float* res, float* unc, long long batch,
                          long long hw, int n_out, int experts, rehr_stream stream);
int rehr_uasr_mixture_bwd(const float* out_cl, const float* ue_cl, const float* w, const float* b, const float* d_res, const float* d_unc,
                          float* d_out_cl, float* d_ue_cl, float* partial, long long batch, long long hw, int n_out, int experts,
                          rehr_stream stream);

/* Low-resolution simulation of the SR stage: `resize(img, (slice_separation, 1), order=3 | 0)` (utils/train_set.py:395-396,
 * third-party resize.pytorch, source unavailable) as resampling along ONE axis of x[outer][n_in][inner] with step `step`, same
 * field of view (sample i at (i + 0.5) * step - 0.5), n_out = round(n_in / step) chosen by the caller; order 3 = cubic
 * convolution (A = -0.75) with clamped indices, order 0 = nearest.  f32.  The definition is the stand-in of oracle/degrade.py. */
int rehr_resample_axis(const float* x, float* y, long long outer, int n_in, int n_out, long long inner, float step, int order,
                       rehr_stream stream);

/* Stage-2 spatial augmentation (SURVEY section 8(f) row 2): `augment_spatial` (utils/seg_utils.py:378-458) in the dummy-2D
 * configuration of get_training_transforms (:652-676) resamples every slice of a patch under one affine map per sample through
 * batchgenerators' interpolate_img = scipy.ndimage.map_coordinates(order 3 for the image / uncertainty, order 1 per label for the
 * segmentations, mode "constant").
 *   rehr_bspline_prefilter_axis: scipy's cubic B-spline prefilter (mirror boundary) in place along the middle axis of
 *     c[outer][n][inner] -- call once per image axis before order-3 sampling.
 *   rehr_affine_sample2d: dst[s][i][j] = value of slice s at A_k (i - (px-1)/2, j - (py-1)/2) + c_k, k = s / slices_per_sample,
 *     affine = f32 device [samples][6] (a00 a01 a10 a11 cx cy).  order 3: src holds the prefiltered coefficients, positions outside
 *     [0, n-1] give cval.  order 1: interpolate_img(is_seg=True): for each of the n_labels (<= 8, ascending, HOST array) label
 *     values the bilinear interpolation of its indicator; the result is the last label reaching 0.5, 0 outside the image. */
int rehr_bspline_prefilter_axis(float* c, long long outer, int n, long long inner, rehr_stream stream);
int rehr_affine_sample2d(const float* src, float* dst, const float* affine, int slices, int x, int y, int px, int py, int slices_per_sample,
                         int order, float cval, const float* labels_host, int n_labels, rehr_stream stream);

/* Stage-2 intensity augmentation (rehrseg_b200/intensity.py): the noise / blur / brightness / contrast / low-resolution / gamma
 * transforms get_training_transforms appends after the spatial part (utils/seg_utils.py:677-689), batchgenerators 0.25 semantics
 * (restated, parity unpinned).  Every entry point works on ROWS: a row is one (sample, channel) volume [z][x][y] of the f32 data
 * tensor the transform fired on, described by one rehr_irow of a DEVICE table; rows not listed are never read.  One launch covers
 * all rows.  Moment tables are f64 [rows][rehr_intensity_moment_doubles()]: per-chunk partials of a row, reduced in a fixed order
 * (the chunking depends on the row's length only, so results do not depend on which other rows share the launch).
 *   rehr_intensity_moments     partials of (sum, sum of squares, min, max) of row.len elements at base + row.off (from_aux = 0)
 *                              or base + row.aux (from_aux = 1).
 *   rehr_intensity_pointwise   op 0: x += noise[aux + i] (the sum in f64, stored f32); op 1: x *= p[0]; op 2: contrast
 *                              (x - mean) * p[0] + mean from `moments` of the same rows, clipped to their [min, max] when n[0].
 *   rehr_intensity_noise_philox  x += (float)(p[0] * z_i) (the sum in f64, stored f32) with z generated in the kernel: row r's key is
 *                              keys[2r], keys[2r + 1] (a DEVICE array); element i takes word i % 4 of Philox4x64-10 block i / 4 at
 *                              counter (i / 4 + 1, 0, 0, 0) -- np.random.Philox(key=key).random_raw -- and z is Box-Muller in f64 over
 *                              the word pairs (2j, 2j + 1): u1 = ((w >> 11) + 1) 2^-53, u2 = (w' >> 11) 2^-53, r = sqrt(-2 ln u1),
 *                              z_2j = r cos(2 pi u2), z_2j+1 = r sin(2 pi u2).
 *   rehr_intensity_blur_axis   scipy.ndimage.gaussian_filter1d along `axis` (0 = z, 1 = x, 2 = y) of the [z][x][y] rows, sigma p[axis],
 *                              radius n[axis] (<= 63), mode 'reflect' for any length; src / dst at row.off or, when *_aux, row.aux.
 *   rehr_intensity_gamma       augment_gamma on s * x (s = p[1] = +-1, gamma p[0], retain_stats n[0]) with the `moments` of x:
 *                              apply = 0 writes the moments of the powered values to `powered`; apply = 1 writes the result.
 *   rehr_intensity_lowres_*    resize(x, (z, n[0], n[1]), order 0) then resize(., (z, x, y), order 3), scikit-image 'edge' semantics:
 *                              gather writes the order-0 image edge-padded by 12 samples, [z][n[0] + 24][n[1] + 24] at pad + row.aux
 *                              (row.len elements); prefilter runs the mirror B-spline prefilter along axis 1 or 2 of it; upsample
 *                              evaluates the cubic spline, clipped to the [min, max] of `moments` (of the padded rows). */
typedef struct {
  long long off;  /* first element of the row in the data tensor */
  long long aux;  /* first element of the row's scratch (noise field, blur temporary, padded low-resolution image) */
  long long len;  /* elements of the row, or of its scratch (low resolution) */
  int n[4];       /* integer parameters */
  double p[4];    /* real parameters */
} rehr_irow;
int rehr_intensity_moment_doubles(void);
int rehr_intensity_moments(const float* base, const rehr_irow* rows, int nrows, int from_aux, long long max_len, double* moments,
                           rehr_stream stream);
int rehr_intensity_pointwise(float* x, const rehr_irow* rows, int nrows, long long len, int op, const float* noise, const double* moments,
                             rehr_stream stream);
int rehr_intensity_noise_philox(float* x, const rehr_irow* rows, const unsigned long long* keys, int nrows, long long len,
                                rehr_stream stream);
int rehr_intensity_blur_axis(const float* src, int src_aux, float* dst, int dst_aux, const rehr_irow* rows, int nrows, int z, int x, int y,
                             int axis, rehr_stream stream);
int rehr_intensity_gamma(float* x, const rehr_irow* rows, int nrows, long long len, const double* moments, double* powered, int apply,
                         rehr_stream stream);
int rehr_intensity_lowres_gather(const float* x, float* pad, const rehr_irow* rows, int nrows, int z, int xs, int ys, long long max_len,
                                 rehr_stream stream);
int rehr_intensity_lowres_prefilter(float* pad, const rehr_irow* rows, int nrows, int z, int axis, long long max_lines, rehr_stream stream);
int rehr_intensity_lowres_upsample(float* x, const float* pad, const rehr_irow* rows, int nrows, int z, int xs, int ys,
                                   const double* moments, rehr_stream stream);

/* rotate_vol_2d (utils/rotate.py:5-31): rot90 by k quarter turns over dims (0,1) of vol[X][Y][inner]. */
int rehr_rot90(const void* src, void* dst, int X, int Y, long long inner_bytes, int k, rehr_stream stream);

/* FBA spectral combine (utils/fba.py:8-16) on K interleaved-complex64 spectra of `n` bins each.
 * p < 0 : the reference's np.max on complex = lexicographic (real, then imag) maximum.
 * p >= 0: sum_i w_i v_i with w_i = |v_i|^p / sum_j |v_j|^p. */
int rehr_fba_combine(const void* const* spectra_dev_ptrs, int K, float p, void* out, long long n,
                     rehr_stream stream);

/* mean over K volumes (utils/sr_utils.py:65,173,217) */
int rehr_mean_stack(const float* const* vols_dev_ptrs, int K, float* out, long long n, rehr_stream stream);

/* ----------------------------------------------------------------------------------------------
 * Fused loss reductions of the stage-2 step (csrc/loss_ops.cu): every forward entry point makes ONE pass over the fp32 NCDHW
 * tensor the caller holds and writes per-block partial sums (the caller adds the `rehr_loss_blocks(V)` partials of a sample and
 * forms the few loss scalars); every backward entry point turns the gradients of those sums into the dense gradient.
 *   rehr_seg_loss_sums      DC_and_weighted_CE_loss (utils/seg_utils.py:305-353): logits [B][C][V], target [B][V] (class index as
 *                           f32), weight [V] or NULL (multiplies the CE map of every sample -- the reference's uncertainty
 *                           broadcast); partial [B][blocks][1 + 3C] = {sum w*ce, then per class sum p*[y=c], sum p, sum [y=c]}
 *   rehr_seg_loss_bwd       g_ce [B], g_int [B][C], g_pred [B][C] -> dlogits [B][C][V]
 *   rehr_cosine_sums        cosine_distance_loss (models/seg_model.py:60-78): a, b [B][C][V]; partial [B][blocks][3][C] =
 *                           voxel sums of ahat*bhat, ahat^2, bhat^2 with xhat = x / max(||x[:, v]||, 1e-12)
 *   rehr_cosine_sums_bwd    g_ab, g_aa [B][C] -> da [B][C][V]  (b carries no gradient: the teacher is detached)
 *   rehr_plane_maxpool      CriterionPairWiseforWholeFeatAfterPool (models/seg_model.py:95-113): x [N][C][S][H][W], windows ph x pw,
 *                           stride = window, ceil mode -> out, idx [N][S][C][OH][OW] (idx = first arg-max inside the H*W plane)
 *   rehr_plane_maxpool_bwd  g, idx -> scatter into the caller-zeroed dx [N][C][S][H][W]
 * and of the SR-stage step (the loss statements of train_sr, train_all.py:124-133):
 *   rehr_sr_loss_sums       L1Loss(hat[:, 0:1], t[:, 0:1]), with the UASR head mean(|e| / u + log u) and L1Loss(u, |e|.detach())
 *                           (:125-130), and BCEDiceLoss(hat[:, 1:], t[:, 1:]) (:133, utils/seg_utils.py:821-886).  hat [B][C][S][HW]
 *                           contiguous (channel 0 the image, 1..C-1 segmentation logits, 2 <= C <= 4); target: contiguous H*W
 *                           planes at batch / channel / depth strides t_batch, t_channel, t_depth (elements), so the depth window
 *                           of patches_hr is read in place; u [B][1][S][HW] or NULL (plain head).  partial
 *                           [rehr_loss_blocks(B*S*HW)][3 + 4(C-1)] = {sum |e|, sum |e|/u + log u, sum |u - |e||, then per
 *                           segmentation channel sum bce(x, y), sum p*y, sum p^2, sum y^2}, e = hat_0 - t_0, p = sigmoid(x)
 *   rehr_sr_loss_bwd        g [3 + 4(C-1)] (device; gradients of the sums in the same order) -> d_hat [B][C][S][HW] and
 *                           d_u [B][1][S][HW] (non-NULL exactly when u is); sign(0) = 0 as torch's abs backward
 * ---------------------------------------------------------------------------------------------- */
int rehr_loss_blocks(long long voxels);
int rehr_seg_loss_sums(const float* logits, const float* target, const float* weight, int B, int C, long long V, float* partial,
                       rehr_stream stream);
int rehr_seg_loss_bwd(const float* logits, const float* target, const float* weight, int B, int C, long long V, const float* g_ce,
                      const float* g_int, const float* g_pred, float* dlogits, rehr_stream stream);
int rehr_cosine_sums(const float* a, const float* b, int B, int C, long long V, float* partial, rehr_stream stream);
int rehr_cosine_sums_bwd(const float* a, const float* b, int B, int C, long long V, const float* g_ab, const float* g_aa, float* da,
                         rehr_stream stream);
int rehr_plane_maxpool(const float* x, int N, int C, int S, int H, int W, int ph, int pw, float* out, int* idx, rehr_stream stream);
int rehr_plane_maxpool_bwd(const float* g, const int* idx, int N, int C, int S, int H, int W, int ph, int pw, float* dx_zeroed,
                           rehr_stream stream);
int rehr_sr_loss_sums(const float* hat, const float* target, const float* u, int B, int C, int S, int HW, long long t_batch,
                      long long t_channel, long long t_depth, float* partial, rehr_stream stream);
int rehr_sr_loss_bwd(const float* hat, const float* target, const float* u, int B, int C, int S, int HW, long long t_batch,
                     long long t_channel, long long t_depth, const float* g, float* d_hat, float* d_u, rehr_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* REHRSEG_B200_H_ */
