// Internal C++ interface between the conv engine (conv_engine.cu), the elementwise kernels and the C-ABI
// shim (api.cu).  Nothing here is exported; the public surface is include/rehrseg_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "../../include/rehrseg_b200.h"

namespace rehr {

static constexpr int kMaxMaps = 8;    // input parity classes (stride 2 in 3 dims)
static constexpr int kMaxTaps = 128;  // 5x5x5 = 125

struct Tap {
  int map_id;
  int dw, dh, dd;  // coordinate shift inside the parity-class map
  int widx;        // tap index inside the packed weight (kd,kh,kw linearised)
};

struct TapPlan {
  int num_maps = 0;
  int map_r[kMaxMaps][3];    // parity offset (w h d)
  int map_s[kMaxMaps][3];    // decimation
  int map_ext[kMaxMaps][3];  // extent
  int num_taps = 0;
  int weight_taps = 0;       // kd*kh*kw of the packed weight
  Tap taps[kMaxTaps];
};

extern thread_local int g_last_cuda_error;
int sm_count();
static constexpr int kDefaultSmemReserveKB = 0;
size_t smem_budget();

int build_fwd_taps(const rehr_conv_desc& cd, const rehr_tensor& in, TapPlan* plan);
int build_dgrad_taps(const rehr_conv_desc& cd, const int cls[3], TapPlan* plan);
void choose_box(int W, int H, int D, int N, int vox, int box[4]);

int launch_tapped_gemm(const TapPlan& plan, const rehr_tensor& in, const void* w_packed, int w_rows,
                       const float* bias, const rehr_tensor& out, int out_f32, const int O[4], const int os[3],
                       const int oo[3], int act, float slope, float* stats, cudaStream_t stream,
                       const int* scatter_s = nullptr, void* ws = nullptr, size_t ws_bytes = 0, size_t* ws_need = nullptr,
                       const rehr_tensor* out2 = nullptr);
size_t tapped_wgrad_workspace(const TapPlan& plan, const rehr_tensor& X, const rehr_tensor& Y);
int launch_tapped_wgrad(const TapPlan& plan, const rehr_tensor& X, const rehr_tensor& Y, float* dw, long long s_n,
                        long long s_m, long long s_t, int accumulate, void* ws, size_t ws_bytes, cudaStream_t stream);
int launch_pack_weight(const float* src, void* dst, int R, int C, int T, long long sr, long long sc, long long st,
                       cudaStream_t stream, int f16 = 0);

// One recorded weight-pack call (pack_batch.cu).  kind 0: generic [R][T][C] gather; 1: marching layout; 2: marching layout of the
// parity classes of a stride-2 input gradient.  Plain data: the table travels in the kernel parameters.
static constexpr int kPackBatchMax = 128;
struct PackJob {
  const float* src;
  void* dst;
  long long total;          // destination elements
  long long sr, sc, st;     // kind 0 source strides
  long long s_co, s_ci;     // kind 1 source strides
  int kind, f16, runs, nblocks, block0;
  int R, C, T;                                        // kind 0
  int cout, cout_pad, cin, Ct, BK, ks, kdn, flip;     // kind 1 (kind 2: cin = A, cout = B, cout_pad = Bpad)
  int sd, sh, sw;                                     // kind 2
};
bool pack_recording();          // this thread is between rehr_pack_batch_begin and rehr_pack_batch_launch
int pack_record(PackJob job);   // append (fills total / runs / nblocks)

// fp16 saturation sink (rehr_range_sink, ptx.cuh range_check): the slot a launch wrapper hands its kernel, or null when this
// thread has no sink set or the store the wrapper launches is not fp16 -- a null slot means the kernel checks nothing.
struct RangeSlot;
RangeSlot* range_target(int out_f16);

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a PER-DEVICE setting: a process that drives several GPUs must apply it on
// each of them, so the "already done" flag lives per device (index = cudaGetDevice()).
static constexpr int kMaxDevices = 64;
int current_device();
#define REHR_SET_MAX_SMEM_ONCE(kernel, bytes)                                                                        \
  do {                                                                                                               \
    static bool done__[::rehr::kMaxDevices] = {};                                                                   \
    const int dev__ = ::rehr::current_device();                                                                      \
    if (!done__[dev__]) {                                                                                            \
      cudaError_t ea__ = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes));    \
      if (ea__ != cudaSuccess) {                                                                                     \
        ::rehr::g_last_cuda_error = (int)ea__;                                                                       \
        return REHR_CUDA_ERROR;                                                                                      \
      }                                                                                                              \
      done__[dev__] = true;                                                                                          \
    }                                                                                                                \
  } while (0)

#define REHR_CHECK_LAUNCH()                                   \
  do {                                                        \
    cudaError_t e__ = cudaGetLastError();                     \
    if (e__ != cudaSuccess) {                                 \
      ::rehr::g_last_cuda_error = (int)e__;                   \
      return REHR_CUDA_ERROR;                                 \
    }                                                         \
  } while (0)

}  // namespace rehr
