// extern "C" surface of the conv engine (see include/rehrseg_b200.h).  Pure shape checking + dispatch; the
// kernels live in conv_engine.cu / smallcin.cu / elementwise.cu.
#include "engine.h"

#include <algorithm>
#include <cstdint>

#include <cuda_bf16.h>

#include "ptx.cuh"

using namespace rehr;

namespace {

inline int conv_out(int in, int k, int s, int p) { return (in + 2 * p - k) / s + 1; }

bool conv_shapes_ok(const rehr_conv_desc* d, const rehr_tensor* x, const rehr_tensor* y) {
  if (!d || !x || !y || !x->ptr || !y->ptr) return false;
  if (d->kd <= 0 || d->kh <= 0 || d->kw <= 0 || d->sd <= 0 || d->sh <= 0 || d->sw <= 0) return false;
  if (x->n != y->n) return false;
  return y->d == conv_out(x->d, d->kd, d->sd, d->pd) && y->h == conv_out(x->h, d->kh, d->sh, d->ph) &&
         y->w == conv_out(x->w, d->kw, d->sw, d->pw);
}

// out(class) = act(bias): used for output parity classes no tap reaches.
__global__ void fill_class_kernel(void* out, int out_f32, int out_f16, long long ld, int cout, const float* bias, int act, float slope,
                                  int O0, int O1, int O2, int N, int s0, int s1, int s2, int o0, int o1, int o2, int A0, int A1,
                                  int A2, RangeSlot* range) {
  const long long total = (long long)N * O2 * O1 * O0 * cout;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % cout);
    long long r = i / cout;
    const int w = (int)(r % O0);
    r /= O0;
    const int h = (int)(r % O1);
    r /= O1;
    const int d = (int)(r % O2);
    const long long n = r / O2;
    float v = bias ? bias[c] : 0.f;
    if (act == REHR_ACT_RELU) v = v > 0.f ? v : 0.f;
    if (act == REHR_ACT_LRELU) v = v > 0.f ? v : v * slope;
    const long long vox = ((n * A2 + (d * s2 + o2)) * A1 + (h * s1 + o1)) * A0 + (w * s0 + o0);
    if (out_f32)
      reinterpret_cast<float*>(out)[vox * ld + c] = v;
    else
      reinterpret_cast<unsigned short*>(out)[vox * ld + c] = pack16(v, out_f16);
    if (range) range_check<1>(range, &v);
  }
}

thread_local RangeSlot* g_range_slots = nullptr;
thread_local int g_range_slot = 0;

}  // namespace

namespace rehr {
RangeSlot* range_target(int out_f16) { return out_f16 && g_range_slots ? g_range_slots + g_range_slot : nullptr; }
}  // namespace rehr

extern "C" {

const char* rehr_strerror(int status) {
  switch (status) {
    case REHR_OK: return "ok";
    case REHR_BAD_SHAPE: return "inconsistent or null operand shapes";
    case REHR_UNSUPPORTED: return "configuration not supported by the sm_100a kernels";
    case REHR_WORKSPACE: return "workspace missing or too small";
    case REHR_CUDA_ERROR: return "CUDA call failed (see rehr_last_cuda_error)";
    case REHR_BAD_ALIGNMENT: return "pointer or pitch not 16-byte aligned";
    default: return "unknown rehr_status";
  }
}
int rehr_last_cuda_error(void) { return g_last_cuda_error; }
int rehr_version(void) { return 6; }
int rehr_device_sm_count(void) { return sm_count(); }

int rehr_range_sink(void* slots, int slot) {
  if (slots && slot < 0) return REHR_BAD_SHAPE;
  g_range_slots = reinterpret_cast<RangeSlot*>(slots);
  g_range_slot = slots ? slot : 0;
  return REHR_OK;
}
int rehr_range_clear(void* slots, int n, rehr_stream stream) {
  if (!slots || n <= 0) return REHR_BAD_SHAPE;
  cudaError_t e = cudaMemsetAsync(slots, 0, sizeof(RangeSlot) * (size_t)n, (cudaStream_t)stream);
  if (e != cudaSuccess) {
    g_last_cuda_error = (int)e;
    return REHR_CUDA_ERROR;
  }
  return REHR_OK;
}

int rehr_pack_weight(const float* src, void* dst16, int R, int C, int T, long long sr, long long sc, long long st, int dtype,
                     rehr_stream stream) {
  if (!src || !dst16 || R <= 0 || C <= 0 || T <= 0) return REHR_BAD_SHAPE;
  return launch_pack_weight(src, dst16, R, C, T, sr, sc, st, (cudaStream_t)stream, dtype == REHR_F16);
}

int rehr_conv3d_stats_tiles(const rehr_tensor* y) {
  if (!y) return 0;
  int box[4];
  choose_box(y->w, y->h, y->d, y->n, 128, box);
  if (box[3] != 1) return 0;
  return ((y->w + box[0] - 1) / box[0]) * ((y->h + box[1] - 1) / box[1]) * ((y->d + box[2] - 1) / box[2]);
}

// ws / ws_bytes: optional split-K scratch (see rehr_conv3d_splitk_workspace); need != nullptr => planning query only.
static int conv_fwd_impl(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                         const rehr_tensor* y, int y_is_f32, int act, float slope, float* stats, rehr_stream stream, void* ws,
                         size_t ws_bytes, size_t* need) {
  if (!conv_shapes_ok(desc, x, y) || !w_packed) return REHR_BAD_SHAPE;
  TapPlan plan;
  int rc = build_fwd_taps(*desc, *x, &plan);
  if (rc != REHR_OK) return rc;
  const int O[4] = {y->w, y->h, y->d, y->n};
  const int os[3] = {1, 1, 1}, oo[3] = {0, 0, 0};
  return launch_tapped_gemm(plan, *x, w_packed, y->c, bias, *y, y_is_f32, O, os, oo, act, slope, stats, (cudaStream_t)stream, nullptr,
                            ws, ws_bytes, need);
}

// Fork / join helper for the parity classes of a small strided input gradient: each class is its own launch with a handful of
// CTAs (e.g. 2 of 148 for the 8^3 -> 4^3 stage entry), so the classes are issued on side streams and run side by side.  The
// fork / join is expressed with events only (no host synchronisation), which is also the pattern CUDA-graph capture accepts.
namespace {
struct ClassStreams {
  static constexpr int kSide = 7;
  cudaStream_t side[kSide];
  cudaEvent_t fork, join[kSide];
  bool ok = false;
};
ClassStreams* class_streams() {
  static thread_local ClassStreams per_dev[16];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
  ClassStreams& cs = per_dev[dev];
  if (!cs.ok) {
    if (cudaEventCreateWithFlags(&cs.fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    for (int i = 0; i < ClassStreams::kSide; ++i) {
      if (cudaStreamCreateWithFlags(&cs.side[i], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&cs.join[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    }
    cs.ok = true;
  }
  return &cs;
}
}  // namespace

static int conv_dgrad_impl(const rehr_conv_desc* desc, const rehr_tensor* dy, const void* w_packed, const float* bias,
                           const rehr_tensor* dx, int dx_is_f32, int act, float slope, rehr_stream stream, void* ws, size_t ws_bytes,
                           size_t* need) {
  // shapes: dy is the conv output grid, dx the conv input grid
  if (!conv_shapes_ok(desc, dx, dy) || !w_packed) return REHR_BAD_SHAPE;
  if (need) *need = 0;
  const int s[3] = {desc->sw, desc->sh, desc->sd};
  const int isz[3] = {dx->w, dx->h, dx->d};
  // classes side by side when each of them fills less than half the machine (a function of the shapes only, so that the
  // workspace query and the launch agree): every class then owns a slice of the split-K scratch
  const int ncls = s[0] * s[1] * s[2];
  bool parallel = false;
  if (ncls > 1) {
    long long vox = dx->n;
    for (int a = 0; a < 3; ++a) vox *= (isz[a] + s[a] - 1) / s[a];
    const long long tiles_cls = ((vox + 127) / 128) * ((dx->c + 255) / 256);
    parallel = tiles_cls * 2 <= sm_count();
  }
  ClassStreams* cs = (parallel && !need) ? class_streams() : nullptr;
  if (parallel && !need && cs == nullptr) parallel = false;
  const size_t slice = parallel && ws && ws_bytes ? (ws_bytes / ncls) & ~size_t(255) : 0;
  int launched = 0;
  if (cs) {
    cudaError_t e = cudaEventRecord(cs->fork, (cudaStream_t)stream);
    if (e != cudaSuccess) { g_last_cuda_error = (int)e; return REHR_CUDA_ERROR; }
  }
  int ci = -1;
  // the class launches live in a lambda so that EVERY exit path -- also an error half-way through -- reaches the join below (a
  // forked side stream that is never joined would poison an enclosing CUDA-graph capture)
  auto run_classes = [&]() -> int {
  for (int cd = 0; cd < s[2]; ++cd)
    for (int ch = 0; ch < s[1]; ++ch)
      for (int cw = 0; cw < s[0]; ++cw) {
        const int cls[3] = {cw, ch, cd};
        int O[4];
        bool empty = false;
        for (int a = 0; a < 3; ++a) {
          O[a] = (isz[a] - cls[a] + s[a] - 1) / s[a];
          if (O[a] <= 0) empty = true;
        }
        O[3] = dx->n;
        ++ci;
        if (empty) continue;
        TapPlan plan;
        int rc = build_dgrad_taps(*desc, cls, &plan);
        if (rc != REHR_OK) return rc;
        // class 0 stays on the caller's stream, the others go to side streams that wait for the fork event
        cudaStream_t cstream = (cudaStream_t)stream;
        if (cs && ci > 0) {
          cstream = cs->side[(ci - 1) % ClassStreams::kSide];
          if (!((launched >> ((ci - 1) % ClassStreams::kSide)) & 1)) {
            cudaError_t e = cudaStreamWaitEvent(cstream, cs->fork, 0);
            if (e != cudaSuccess) { g_last_cuda_error = (int)e; return REHR_CUDA_ERROR; }
            launched |= 1 << ((ci - 1) % ClassStreams::kSide);
          }
        }
        if (plan.num_taps == 0) {
          if (need) continue;
          const long long total = (long long)O[0] * O[1] * O[2] * O[3] * dx->c;
          const int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 8);
          fill_class_kernel<<<blocks, 256, 0, cstream>>>(dx->ptr, dx_is_f32, dx->dtype == REHR_F16, dx->ld, dx->c, bias, act, slope, O[0], O[1],
                                                                     O[2], O[3], s[0], s[1], s[2], cw, ch, cd, dx->w, dx->h, dx->d,
                                                                     range_target(!dx_is_f32 && dx->dtype == REHR_F16));
          REHR_CHECK_LAUNCH();
          continue;
        }
        size_t cls_need = 0;
        void* cws = parallel ? (slice ? reinterpret_cast<uint8_t*>(ws) + (size_t)ci * slice : nullptr) : ws;
        rc = launch_tapped_gemm(plan, *dy, w_packed, dx->c, bias, *dx, dx_is_f32, O, s, cls, act, slope, nullptr, cstream, nullptr, cws,
                                parallel ? slice : ws_bytes, need ? &cls_need : nullptr);
        if (rc != REHR_OK) return rc;
        // back to back on one stream the classes share the scratch; side by side each class gets its own slice
        if (need) {
          cls_need = (cls_need + 255) & ~size_t(255);
          if (parallel) *need = std::max(*need, cls_need * (size_t)ncls);
          else if (cls_need > *need) *need = cls_need;
        }
      }
  return REHR_OK;
  };
  int status = run_classes();
  if (cs) {  // join: the caller's stream continues after every side stream that was used
    for (int i = 0; i < ClassStreams::kSide; ++i)
      if ((launched >> i) & 1) {
        cudaError_t e = cudaEventRecord(cs->join[i], cs->side[i]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent((cudaStream_t)stream, cs->join[i], 0);
        if (e != cudaSuccess && status == REHR_OK) { g_last_cuda_error = (int)e; status = REHR_CUDA_ERROR; }
      }
  }
  return status;
}

int rehr_conv3d_fwd(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                    const rehr_tensor* y, int y_is_f32, int act, float slope, float* stats, rehr_stream stream) {
  return conv_fwd_impl(desc, x, w_packed, bias, y, y_is_f32, act, slope, stats, stream, nullptr, 0, nullptr);
}

int rehr_conv3d_dgrad(const rehr_conv_desc* desc, const rehr_tensor* dy, const void* w_packed, const float* bias,
                      const rehr_tensor* dx, int dx_is_f32, int act, float slope, rehr_stream stream) {
  return conv_dgrad_impl(desc, dy, w_packed, bias, dx, dx_is_f32, act, slope, stream, nullptr, 0, nullptr);
}

// Split-K variants: layers with fewer output tiles than SMs (the <= 8^3 bottleneck stages) share their K loop over several CTAs
// through an fp32 scratch buffer.  rehr_conv3d_splitk_workspace returns the bytes needed (0 = the layer does not split).
size_t rehr_conv3d_splitk_workspace(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const rehr_tensor* y,
                                    int is_dgrad) {
  size_t need = 0;
  int rc = is_dgrad ? conv_dgrad_impl(desc, x, w_packed, nullptr, y, 0, REHR_ACT_NONE, 0.f, nullptr, nullptr, 0, &need)
                    : conv_fwd_impl(desc, x, w_packed, nullptr, y, 0, REHR_ACT_NONE, 0.f, nullptr, nullptr, nullptr, 0, &need);
  return rc == REHR_OK ? need : 0;
}
int rehr_conv3d_fwd_ws(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                       const rehr_tensor* y, int y_is_f32, int act, float slope, float* stats, void* ws, size_t ws_bytes,
                       rehr_stream stream) {
  return conv_fwd_impl(desc, x, w_packed, bias, y, y_is_f32, act, slope, stats, stream, ws, ws_bytes, nullptr);
}
int rehr_conv3d_dgrad_ws(const rehr_conv_desc* desc, const rehr_tensor* dy, const void* w_packed, const float* bias,
                         const rehr_tensor* dx, int dx_is_f32, int act, float slope, void* ws, size_t ws_bytes, rehr_stream stream) {
  return conv_dgrad_impl(desc, dy, w_packed, bias, dx, dx_is_f32, act, slope, stream, ws, ws_bytes, nullptr);
}

size_t rehr_conv3d_wgrad_workspace(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy) {
  if (!conv_shapes_ok(desc, x, dy)) return 0;
  TapPlan plan;
  if (build_fwd_taps(*desc, *x, &plan) != REHR_OK) return 0;
  return tapped_wgrad_workspace(plan, *x, *dy);
}

int rehr_conv3d_wgrad(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy, float* dw, int accumulate,
                      void* ws, size_t ws_bytes, rehr_stream stream) {
  if (!conv_shapes_ok(desc, x, dy) || !dw) return REHR_BAD_SHAPE;
  TapPlan plan;
  int rc = build_fwd_taps(*desc, *x, &plan);
  if (rc != REHR_OK) return rc;
  const int T = desc->kd * desc->kh * desc->kw;
  if (plan.num_taps < T && !accumulate) {
    // taps that never touch the volume have an exactly-zero gradient
    cudaError_t e = cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)dy->c * x->c * T, (cudaStream_t)stream);
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
  }
  // dW[a][b][t]: a = dy channel (N side), b = x channel (M side)
  return launch_tapped_wgrad(plan, *x, *dy, dw, (long long)x->c * T, T, 1, accumulate, ws, ws_bytes, (cudaStream_t)stream);
}

// kernel == stride, padding 0 transposed conv as ONE GEMM: rows = input voxels, N = classes x Cout, scatter epilogue.
// w_packed = bf16 [T][Cout][Cin] (rehr_pack_weight with R = T, C = Cin, T = Cout, sr = 1, sc = Cout*T, st = T).
int rehr_convtranspose3d_fused_supported(const rehr_conv_desc* d, int cin, int cout) {
  if (!d) return 0;
  if (d->kd != d->sd || d->kh != d->sh || d->kw != d->sw || d->pd || d->ph || d->pw) return 0;
  if (cout % 16 != 0 || cin % 16 != 0) return 0;
  if (d->sd * d->sh * d->sw > 8) return 0;  // class offset table of the scatter epilogue
  return 1;
}
static int tconv_fused_impl(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias, const rehr_tensor* y,
                            const rehr_tensor* y2, int act, float slope, rehr_stream stream);
int rehr_convtranspose3d_fused_fwd(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                                   const rehr_tensor* y, int act, float slope, rehr_stream stream) {
  return tconv_fused_impl(desc, x, w_packed, bias, y, nullptr, act, slope, stream);
}
int rehr_convtranspose3d_fused_fwd2(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                                    const rehr_tensor* y, const rehr_tensor* y2, int act, float slope, rehr_stream stream) {
  if (!y2 || !y2->ptr || !y || y2->n != y->n || y2->d != y->d || y2->h != y->h || y2->w != y->w || y2->c != y->c) return REHR_BAD_SHAPE;
  return tconv_fused_impl(desc, x, w_packed, bias, y, y2, act, slope, stream);
}
static int tconv_fused_impl(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias, const rehr_tensor* y,
                            const rehr_tensor* y2, int act, float slope, rehr_stream stream) {
  if (!desc || !x || !y || !x->ptr || !y->ptr || !w_packed) return REHR_BAD_SHAPE;
  if (!rehr_convtranspose3d_fused_supported(desc, x->c, y->c)) return REHR_UNSUPPORTED;
  if (x->n != y->n || y->d != x->d * desc->sd || y->h != x->h * desc->sh || y->w != x->w * desc->sw) return REHR_BAD_SHAPE;
  TapPlan plan;
  plan.num_maps = 1;
  for (int a = 0; a < 3; ++a) {
    plan.map_r[0][a] = 0;
    plan.map_s[0][a] = 1;
    plan.map_ext[0][a] = 0;
  }
  plan.num_taps = 1;
  plan.weight_taps = 1;
  plan.taps[0].map_id = 0;
  plan.taps[0].dw = plan.taps[0].dh = plan.taps[0].dd = 0;
  plan.taps[0].widx = 0;
  const int O[4] = {x->w, x->h, x->d, x->n};
  const int os[3] = {1, 1, 1}, oo[3] = {0, 0, 0};
  const int sc[3] = {desc->sw, desc->sh, desc->sd};
  return launch_tapped_gemm(plan, *x, w_packed, 0, bias, *y, 0, O, os, oo, act, slope, nullptr, (cudaStream_t)stream, sc, nullptr, 0, nullptr,
                            y2);
}

// ---- ConvTranspose3d = the same conv read backwards (weight [Cin][Cout][T], underlying conv Cin <- Cout) ----
int rehr_convtranspose3d_fwd(const rehr_conv_desc* desc, const rehr_tensor* x, const void* w_packed, const float* bias,
                             const rehr_tensor* y, int act, float slope, rehr_stream stream) {
  return rehr_conv3d_dgrad(desc, x, w_packed, bias, y, 0, act, slope, stream);
}
int rehr_convtranspose3d_dgrad(const rehr_conv_desc* desc, const rehr_tensor* dy, const void* w_packed, const rehr_tensor* dx,
                               rehr_stream stream) {
  return rehr_conv3d_fwd(desc, dy, w_packed, nullptr, dx, 0, REHR_ACT_NONE, 0.f, nullptr, stream);
}
size_t rehr_convtranspose3d_wgrad_workspace(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy) {
  return rehr_conv3d_wgrad_workspace(desc, dy, x);
}
int rehr_convtranspose3d_wgrad(const rehr_conv_desc* desc, const rehr_tensor* x, const rehr_tensor* dy, float* dw, int accumulate,
                               void* ws, size_t ws_bytes, rehr_stream stream) {
  return rehr_conv3d_wgrad(desc, dy, x, dw, accumulate, ws, ws_bytes, stream);
}

}  // extern "C"
