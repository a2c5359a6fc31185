// Stage-2 intensity augmentation (rehrseg_b200/intensity.py): Gaussian noise, Gaussian blur, multiplicative brightness, contrast,
// simulated low resolution and gamma of batchgenerators 0.25 (restated, parity unpinned) on ROWS of an f32 [b][c][z][x][y] tensor.
// A row is one (sample, channel) volume a transform fired on; its rehr_irow (device table) gives its offset and parameters.  Every
// kernel is HBM bound, runs a grid of (chunk, row) blocks and never touches a row that is not listed.  Reductions are per-chunk
// partials in f64 combined in a fixed order by their consumers (no atomics): the chunking depends on the row's length alone, so a row
// gives bit-identical results whatever rows share the launch.  Arithmetic that numpy does in f32 is done here in f32 with explicit
// round-to-nearest intrinsics (no FMA contraction); what scipy does in f64 is done in f64.
#include "bspline.cuh"
#include "engine.h"

#include <algorithm>

namespace rehr {

static constexpr int kIChunks = 256;            // most chunks a row is cut into (enough blocks to fill the GPU for one row)
static constexpr int kIMoment = 5;              // doubles per chunk partial: shift, sum(x - shift), sum((x - shift)^2), min, max
static constexpr int kIThreads = 256;
static constexpr int kMaxBlurRadius = 63;       // 2r + 1 <= 127 taps (numpy's pairwise sum of the weights is one 128-block)
static constexpr int kLowresPad = 12;           // scipy's pre-padding of a 'nearest' spline (_prepad_for_spline_filter)

__host__ __device__ __forceinline__ long long ichunk_len(long long len) {
  long long c = (len + kIChunks - 1) / kIChunks;
  c = (c + 1023) / 1024 * 1024;
  return c < 1024 ? 1024 : c;
}
__host__ __device__ __forceinline__ int ichunks(long long len) { return (int)((len + ichunk_len(len) - 1) / ichunk_len(len)); }

struct RowStats {
  double mean, var, mn, mx;
};

// Combine the chunk partials of one row: warp 0, lane l takes chunks l, l + 32, ..., then a butterfly -- a fixed order, so every
// block (and every launch) gets the same values.  All threads of the block return them.
__device__ __forceinline__ RowStats block_row_stats(const double* __restrict__ m, long long len) {
  __shared__ RowStats s;
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x, nch = ichunks(len);
    double s1 = 0.0, s2 = 0.0, mn = m[3], mx = m[4];
    for (int c = lane; c < nch; c += 32) {
      s1 += m[c * kIMoment + 1];
      s2 += m[c * kIMoment + 2];
      mn = fmin(mn, m[c * kIMoment + 3]);
      mx = fmax(mx, m[c * kIMoment + 4]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) {
      const double d = s1 / (double)len;
      s.mean = m[0] + d;
      s.var = fmax(0.0, s2 / (double)len - d * d);
      s.mn = mn;
      s.mx = mx;
    }
  }
  __syncthreads();
  return s;
}

// Block reduction of (s1, s2, min, max) in a fixed tree order; thread 0 writes the chunk partial.
__device__ __forceinline__ void block_moments_store(double s1, double s2, float mn, float mx, double shift, double* __restrict__ out) {
  __shared__ double r1[kIThreads], r2[kIThreads];
  __shared__ float rmn[kIThreads], rmx[kIThreads];
  const int t = threadIdx.x;
  r1[t] = s1; r2[t] = s2; rmn[t] = mn; rmx[t] = mx;
  __syncthreads();
  for (int h = kIThreads / 2; h > 0; h >>= 1) {
    if (t < h) {
      r1[t] += r1[t + h];
      r2[t] += r2[t + h];
      rmn[t] = fminf(rmn[t], rmn[t + h]);
      rmx[t] = fmaxf(rmx[t], rmx[t + h]);
    }
    __syncthreads();
  }
  if (t == 0) {
    out[0] = shift; out[1] = r1[0]; out[2] = r2[0]; out[3] = (double)rmn[0]; out[4] = (double)rmx[0];
  }
}

// The gamma transform of one value v = s * x: ((v - lo) / (r + eps)) ** g * (r + eps) + lo in f32, as numpy evaluates it.
struct GammaRow {
  float lo, re, g;
};
__device__ __forceinline__ float gamma_pow(float v, const GammaRow& q) {
  return __fadd_rn(__fmul_rn(powf(__fdiv_rn(__fsub_rn(v, q.lo), q.re), q.g), q.re), q.lo);
}
__device__ __forceinline__ GammaRow gamma_row(const RowStats& st, float s, double g) {
  // stats of s * x from those of x: min / max swap under negation
  const float lo = s > 0.f ? (float)st.mn : -(float)st.mx;
  const float hi = s > 0.f ? (float)st.mx : -(float)st.mn;
  GammaRow q;
  q.lo = lo;
  q.re = __fadd_rn(__fsub_rn(hi, lo), 1e-7f);
  q.g = (float)g;
  return q;
}

// ---- moments ---------------------------------------------------------------------------------------------------------------------
// GAMMA = false: plain moments of the row; true: moments of the powered values of augment_gamma (stats = moments of x).
template <bool GAMMA>
__global__ void __launch_bounds__(kIThreads) intensity_moments_kernel(const float* __restrict__ base, const rehr_irow* __restrict__ rows,
                                                                      int from_aux, const double* __restrict__ stats,
                                                                      double* __restrict__ out) {
  const int r = blockIdx.y;
  const rehr_irow row = rows[r];
  const long long len = row.len;
  const int ch = blockIdx.x;
  if (ch >= ichunks(len)) return;
  GammaRow q{};
  float s = 1.f;
  if (GAMMA) {
    s = (float)row.p[1];
    q = gamma_row(block_row_stats(stats + (long long)r * kIChunks * kIMoment, len), s, row.p[0]);
  }
  const float* x = base + (from_aux ? rows[r].aux : rows[r].off);   // (formed after the stats: fewer live registers across them)
  // shift = the row's first value (powered: the minimum lo), so the sum of squares does not cancel against the mean
  const double shift = GAMMA ? (double)q.lo : (double)x[0];
  const long long cl = ichunk_len(len), e0 = (long long)ch * cl;
  const int cn = (int)(min(len, e0 + cl) - e0);   // elements of this chunk (a chunk is far below 2^31)
  const float* xc = x + e0;
  double s1 = 0.0, s2 = 0.0;
  float mn = INFINITY, mx = -INFINITY;
  for (int k = threadIdx.x; k < cn; k += kIThreads) {
    float v = xc[k];
    if (GAMMA) v = gamma_pow(s * v, q);
    const double d = (double)v - shift;
    s1 += d;
    s2 += d * d;
    mn = fminf(mn, v);
    mx = fmaxf(mx, v);
  }
  block_moments_store(s1, s2, mn, mx, shift, out + (long long)r * kIChunks * kIMoment + ch * kIMoment);
}

// ---- noise / brightness / contrast -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kIThreads) intensity_pointwise_kernel(float* __restrict__ x, const rehr_irow* __restrict__ rows, long long len,
                                                                        int op, const float* __restrict__ noise,
                                                                        const double* __restrict__ moments) {
  const int r = blockIdx.y;
  const rehr_irow row = rows[r];
  const long long cl = ichunk_len(len), e0 = (long long)blockIdx.x * cl, e1 = min(len, e0 + cl);
  float* p = x + row.off;
  if (op == 0) {
    const float* nz = noise + row.aux;
    for (long long e = e0 + threadIdx.x; e < e1; e += kIThreads) p[e] = (float)((double)p[e] + (double)nz[e]);
  } else if (op == 1) {
    const float m = (float)row.p[0];
    for (long long e = e0 + threadIdx.x; e < e1; e += kIThreads) p[e] = __fmul_rn(p[e], m);
  } else {
    const RowStats st = block_row_stats(moments + (long long)r * kIChunks * kIMoment, len);
    const float mean = (float)st.mean, f = (float)row.p[0], lo = (float)st.mn, hi = (float)st.mx;
    const bool clip = row.n[0] != 0;
    for (long long e = e0 + threadIdx.x; e < e1; e += kIThreads) {
      float v = __fadd_rn(__fmul_rn(__fsub_rn(p[e], mean), f), mean);
      if (clip) {
        if (v < lo) v = lo;
        if (v > hi) v = hi;
      }
      p[e] = v;
    }
  }
}

// ---- Gaussian noise from a counter-based generator -----------------------------------------------------------------------------------
// Philox4x64-10 (Random123 constants).  Block g of a row with key (k0, k1) is philox(counter = (g + 1, 0, 0, 0), key): the word stream
// of np.random.Philox(key=key).random_raw, whose first block is counter 1.
__device__ __forceinline__ void philox4x64_10(unsigned long long c[4], unsigned long long k0, unsigned long long k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k0 += 0x9E3779B97F4A7C15ull;
      k1 += 0xBB67AE8584CAA73Bull;
    }
    const unsigned long long h0 = __umul64hi(0xD2E7470EE14C6C93ull, c[0]), l0 = 0xD2E7470EE14C6C93ull * c[0];
    const unsigned long long h1 = __umul64hi(0xCA5A826395121157ull, c[2]), l1 = 0xCA5A826395121157ull * c[2];
    c[0] = h1 ^ c[1] ^ k0;
    c[1] = l1;
    c[2] = h0 ^ c[3] ^ k1;
    c[3] = l0;
  }
}

// Box-Muller of the word pair (a, b) in f64: u1 = ((a >> 11) + 1) 2^-53 in (0, 1], u2 = (b >> 11) 2^-53, r = sqrt(-2 ln u1);
// the pair's normals are r cos(2 pi u2), r sin(2 pi u2).  sincospi(2 u2) takes the angle without rounding 2 pi u2 (numpy's
// cos(2.0 * np.pi * u2) differs by at most 5e-16 absolute) and has no large-argument reduction, whose scratch array would live in
// local memory.
__device__ __forceinline__ void box_muller(unsigned long long a, unsigned long long b, double& zc, double& zs) {
  const double u1 = __dmul_rn((double)((a >> 11) + 1), 0x1p-53), u2 = __dmul_rn((double)(b >> 11), 0x1p-53);
  const double r = sqrt(__dmul_rn(-2.0, log(u1)));
  double s, c;
  sincospi(2.0 * u2, &s, &c);
  zc = __dmul_rn(r, c);
  zs = __dmul_rn(r, s);
}

// x += (float)(p[0] * z) per element, the sum in f64 and stored f32 (the arithmetic of the host-field path).  Each thread makes whole
// Philox blocks, i.e. 4 elements; a chunk's length is a multiple of 1024, so no block straddles two chunks.
__global__ void __launch_bounds__(kIThreads) intensity_noise_philox_kernel(float* __restrict__ x, const rehr_irow* __restrict__ rows,
                                                                           const unsigned long long* __restrict__ keys, long long len) {
  const int r = blockIdx.y;
  const double vh = rows[r].p[0];
  const unsigned long long k0 = keys[2 * r], k1 = keys[2 * r + 1];
  float* p = x + rows[r].off;
  const long long cl = ichunk_len(len), e0 = (long long)blockIdx.x * cl, e1 = min(len, e0 + cl);
  for (long long g = e0 / 4 + threadIdx.x; 4 * g < e1; g += kIThreads) {
    unsigned long long w[4] = {(unsigned long long)g + 1, 0ull, 0ull, 0ull};
    philox4x64_10(w, k0, k1);
    double z[4];
    box_muller(w[0], w[1], z[0], z[1]);
    box_muller(w[2], w[3], z[2], z[3]);
    const long long e = 4 * g;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (e + i < e1) p[e + i] = (float)((double)p[e + i] + (double)(float)__dmul_rn(vh, z[i]));
  }
}

// ---- Gaussian blur, one axis -------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect_idx(int i, int n) {  // scipy 'reflect' (d c b a | a b c d | d c b a), any length
  const int period = 2 * n;
  i %= period;
  if (i < 0) i += period;
  return i < n ? i : period - 1 - i;
}

__global__ void __launch_bounds__(kIThreads) intensity_blur_kernel(const float* __restrict__ src, int src_aux, float* __restrict__ dst,
                                                                   int dst_aux, const rehr_irow* __restrict__ rows, int Z, int X, int Y,
                                                                   int axis) {
  __shared__ double phi[2 * kMaxBlurRadius + 1], w[kMaxBlurRadius + 1];
  const int r = blockIdx.y;
  const rehr_irow& row = rows[r];   // read in place: n[axis] / p[axis] index it at run time
  const long long len = (long long)Z * X * Y;
  const int rad = row.n[axis], L = 2 * rad + 1;
  // scipy _gaussian_kernel1d: phi = exp(-0.5 / sigma^2 * x^2) / sum(phi), x = -rad..rad; the sum in numpy's pairwise order
  const double sigma = row.p[axis];
  const int t = (int)threadIdx.x - rad;
  if (t <= rad) phi[threadIdx.x] = exp(-0.5 / (sigma * sigma) * (double)(t * t));
  __syncthreads();
  if (threadIdx.x == 0) {
    double sum = 0.0;
    if (L < 8) {
      for (int i = 0; i < L; ++i) sum += phi[i];
    } else {
      double a0 = phi[0], a1 = phi[1], a2 = phi[2], a3 = phi[3], a4 = phi[4], a5 = phi[5], a6 = phi[6], a7 = phi[7];
      int i = 8;
      for (; i < L - (L % 8); i += 8) {
        a0 += phi[i]; a1 += phi[i + 1]; a2 += phi[i + 2]; a3 += phi[i + 3];
        a4 += phi[i + 4]; a5 += phi[i + 5]; a6 += phi[i + 6]; a7 += phi[i + 7];
      }
      sum = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
      for (; i < L; ++i) sum += phi[i];
    }
    for (int j = 0; j <= rad; ++j) w[j] = phi[rad + j] / sum;
  }
  __syncthreads();
  const float* s = src + (src_aux ? row.aux : row.off);
  float* d = dst + (dst_aux ? row.aux : row.off);
  const long long stride = axis == 0 ? (long long)X * Y : axis == 1 ? Y : 1;
  const int n = axis == 0 ? Z : axis == 1 ? X : Y;
  const long long cl = ichunk_len(len), e0 = (long long)blockIdx.x * cl, e1 = min(len, e0 + cl);
  for (long long e = e0 + threadIdx.x; e < e1; e += kIThreads) {
    const int i = (int)((e / stride) % n);
    const float* line = s + (e - (long long)i * stride);
    // scipy correlate1d, symmetric weights: acc = x[i] w0 + sum_{j = rad..1} (x[i - j] + x[i + j]) w_j, in f64
    double acc = (double)line[(long long)i * stride] * w[0];
    for (int j = rad; j >= 1; --j)
      acc += ((double)line[(long long)reflect_idx(i - j, n) * stride] + (double)line[(long long)reflect_idx(i + j, n) * stride]) * w[j];
    d[e] = (float)acc;
  }
}

// ---- gamma apply ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kIThreads) intensity_gamma_apply_kernel(float* __restrict__ x, const rehr_irow* __restrict__ rows, long long len,
                                                                          const double* __restrict__ moments,
                                                                          const double* __restrict__ powered) {
  const int r = blockIdx.y;
  const rehr_irow row = rows[r];
  const float s = (float)row.p[1];
  const RowStats st = block_row_stats(moments + (long long)r * kIChunks * kIMoment, len);
  const GammaRow q = gamma_row(st, s, row.p[0]);
  const bool retain = row.n[0] != 0;
  float pm = 0.f, den = 1.f, sd = 0.f, mn = 0.f;
  if (retain) {
    __syncthreads();   // block_row_stats reuses its shared slot
    const RowStats ps = block_row_stats(powered + (long long)r * kIChunks * kIMoment, len);
    pm = (float)ps.mean;
    den = __fadd_rn((float)sqrt(ps.var), 1e-8f);
    sd = (float)sqrt(st.var);
    mn = s * (float)st.mean;
  }
  float* p = x + row.off;
  const long long cl = ichunk_len(len), e0 = (long long)blockIdx.x * cl, e1 = min(len, e0 + cl);
  for (long long e = e0 + threadIdx.x; e < e1; e += kIThreads) {
    float v = gamma_pow(s * p[e], q);
    if (retain) v = __fadd_rn(__fmul_rn(__fdiv_rn(__fsub_rn(v, pm), den), sd), mn);
    p[e] = s * v;
  }
}

// ---- simulated low resolution --------------------------------------------------------------------------------------------------------
// position of output sample i of a resize n_in -> n_out: (i + 0.5) * (n_in / n_out) - 0.5, each operation rounded as numpy does
__device__ __forceinline__ double resize_pos(int i, int n_in, int n_out) {
  return __dsub_rn(__dmul_rn((double)i + 0.5, __ddiv_rn((double)n_in, (double)n_out)), 0.5);
}

__global__ void __launch_bounds__(kIThreads) intensity_lowres_gather_kernel(const float* __restrict__ x, float* __restrict__ pad,
                                                                            const rehr_irow* __restrict__ rows, int Z, int X, int Y) {
  const int r = blockIdx.y;
  const rehr_irow row = rows[r];
  const long long len = row.len;
  if (blockIdx.x >= ichunks(len)) return;
  const int tx = row.n[0], ty = row.n[1], PX = tx + 2 * kLowresPad, PY = ty + 2 * kLowresPad;
  const float* s = x + row.off;
  float* d = pad + row.aux;
  const long long cl = ichunk_len(len), e0 = (long long)blockIdx.x * cl, e1 = min(len, e0 + cl);
  for (long long e = e0 + threadIdx.x; e < e1; e += kIThreads) {
    const int pj = (int)(e % PY);
    const long long t = e / PY;
    const int pi = (int)(t % PX), zz = (int)(t / PX);
    const int di = min(max(pi - kLowresPad, 0), tx - 1), dj = min(max(pj - kLowresPad, 0), ty - 1);   // np.pad(mode='edge')
    // order 0: floor(c + 0.5) (scipy's rounding of even orders), mode 'nearest'
    const int si = min(max((int)floor(resize_pos(di, X, tx) + 0.5), 0), X - 1);
    const int sj = min(max((int)floor(resize_pos(dj, Y, ty) + 0.5), 0), Y - 1);
    d[e] = s[((long long)zz * X + si) * Y + sj];
  }
}

__global__ void __launch_bounds__(128) intensity_lowres_prefilter_kernel(float* __restrict__ pad, const rehr_irow* __restrict__ rows, int Z,
                                                                         int axis) {
  const rehr_irow row = rows[blockIdx.y];
  const int PX = row.n[0] + 2 * kLowresPad, PY = row.n[1] + 2 * kLowresPad;
  const long long line = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  float* p = pad + row.aux;
  if (axis == 1) {   // lines along x: outer z, inner y
    if (line >= (long long)Z * PY) return;
    bspline_prefilter_line(p + (line / PY) * (long long)PX * PY + line % PY, PX, PY);
  } else {           // lines along y: contiguous
    if (line >= (long long)Z * PX) return;
    bspline_prefilter_line(p + line * PY, PY, 1);
  }
}

// scipy's order-3 spline weights at fractional offset t in [0, 1) (ni_splines.c: spline_interpolation_weights)
__device__ __forceinline__ void cubic_weights(double t, double (&w)[4]) {
  const double y = 1.0 - t;
  w[1] = (t * t * (t - 2.0) * 3.0 + 4.0) / 6.0;
  w[2] = (y * y * (y - 2.0) * 3.0 + 4.0) / 6.0;
  w[0] = y * y * y / 6.0;
  w[3] = 1.0 - w[0] - w[1] - w[2];
}

__global__ void __launch_bounds__(kIThreads) intensity_lowres_upsample_kernel(float* __restrict__ x, const float* __restrict__ pad,
                                                                              const rehr_irow* __restrict__ rows, int Z, int X, int Y,
                                                                              const double* __restrict__ moments) {
  const int r = blockIdx.y;
  const rehr_irow row = rows[r];
  const RowStats st = block_row_stats(moments + (long long)r * kIChunks * kIMoment, row.len);
  const int tx = row.n[0], ty = row.n[1], PX = tx + 2 * kLowresPad, PY = ty + 2 * kLowresPad;
  const float* c = pad + row.aux;
  float* d = x + row.off;
  const long long len = (long long)Z * X * Y;
  const long long cl = ichunk_len(len), e0 = (long long)blockIdx.x * cl, e1 = min(len, e0 + cl);
  for (long long e = e0 + threadIdx.x; e < e1; e += kIThreads) {
    const int j = (int)(e % Y);
    const long long t = e / Y;
    const int i = (int)(t % X), zz = (int)(t / X);
    // z is not resampled (ignore_axes): at integer positions the z spline returns the samples themselves
    const double cx = resize_pos(i, tx, X) + kLowresPad, cy = resize_pos(j, ty, Y) + kLowresPad;
    const int fx = (int)floor(cx), fy = (int)floor(cy);
    double wx[4], wy[4];
    cubic_weights(cx - fx, wx);
    cubic_weights(cy - fy, wy);
    const float* plane = c + (long long)zz * PX * PY;
    double v = 0.0;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const float* line = plane + (long long)min(max(fx - 1 + a, 0), PX - 1) * PY;
      double u = 0.0;
#pragma unroll
      for (int b = 0; b < 4; ++b) u += wy[b] * (double)line[min(max(fy - 1 + b, 0), PY - 1)];
      v += wx[a] * u;
    }
    d[e] = (float)fmin(fmax(v, st.mn), st.mx);
  }
}

static bool rows_ok(const rehr_irow* rows, int nrows) { return rows && nrows > 0 && nrows <= 65535; }

}  // namespace rehr

using namespace rehr;

int rehr_intensity_moment_doubles(void) { return kIChunks * kIMoment; }

int rehr_intensity_moments(const float* base, const rehr_irow* rows, int nrows, int from_aux, long long max_len, double* moments,
                           rehr_stream stream) {
  if (!base || !moments || !rows_ok(rows, nrows) || max_len <= 0) return REHR_BAD_SHAPE;
  intensity_moments_kernel<false><<<dim3(ichunks(max_len), nrows), kIThreads, 0, (cudaStream_t)stream>>>(base, rows, from_aux, nullptr,
                                                                                                          moments);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_intensity_pointwise(float* x, const rehr_irow* rows, int nrows, long long len, int op, const float* noise, const double* moments,
                             rehr_stream stream) {
  if (!x || !rows_ok(rows, nrows) || len <= 0) return REHR_BAD_SHAPE;
  if (op < 0 || op > 2 || (op == 0 && !noise) || (op == 2 && !moments)) return REHR_BAD_SHAPE;
  intensity_pointwise_kernel<<<dim3(ichunks(len), nrows), kIThreads, 0, (cudaStream_t)stream>>>(x, rows, len, op, noise, moments);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_intensity_noise_philox(float* x, const rehr_irow* rows, const unsigned long long* keys, int nrows, long long len,
                                rehr_stream stream) {
  if (!x || !keys || !rows_ok(rows, nrows) || len <= 0) return REHR_BAD_SHAPE;
  intensity_noise_philox_kernel<<<dim3(ichunks(len), nrows), kIThreads, 0, (cudaStream_t)stream>>>(x, rows, keys, len);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_intensity_blur_axis(const float* src, int src_aux, float* dst, int dst_aux, const rehr_irow* rows, int nrows, int z, int x, int y,
                             int axis, rehr_stream stream) {
  if (!src || !dst || !rows_ok(rows, nrows) || z <= 0 || x <= 0 || y <= 0) return REHR_BAD_SHAPE;
  if (axis < 0 || axis > 2) return REHR_BAD_SHAPE;
  const long long len = (long long)z * x * y;
  intensity_blur_kernel<<<dim3(ichunks(len), nrows), kIThreads, 0, (cudaStream_t)stream>>>(src, src_aux, dst, dst_aux, rows, z, x, y, axis);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_intensity_gamma(float* x, const rehr_irow* rows, int nrows, long long len, const double* moments, double* powered, int apply,
                         rehr_stream stream) {
  if (!x || !moments || !powered || !rows_ok(rows, nrows) || len <= 0) return REHR_BAD_SHAPE;
  const dim3 grid(ichunks(len), nrows);
  if (apply)
    intensity_gamma_apply_kernel<<<grid, kIThreads, 0, (cudaStream_t)stream>>>(x, rows, len, moments, powered);
  else
    intensity_moments_kernel<true><<<grid, kIThreads, 0, (cudaStream_t)stream>>>(x, rows, 0, moments, powered);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_intensity_lowres_gather(const float* x, float* pad, const rehr_irow* rows, int nrows, int z, int xs, int ys, long long max_len,
                                 rehr_stream stream) {
  if (!x || !pad || !rows_ok(rows, nrows) || z <= 0 || xs <= 0 || ys <= 0 || max_len <= 0) return REHR_BAD_SHAPE;
  intensity_lowres_gather_kernel<<<dim3(ichunks(max_len), nrows), kIThreads, 0, (cudaStream_t)stream>>>(x, pad, rows, z, xs, ys);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_intensity_lowres_prefilter(float* pad, const rehr_irow* rows, int nrows, int z, int axis, long long max_lines, rehr_stream stream) {
  if (!pad || !rows_ok(rows, nrows) || z <= 0 || max_lines <= 0) return REHR_BAD_SHAPE;
  if (axis != 1 && axis != 2) return REHR_BAD_SHAPE;
  intensity_lowres_prefilter_kernel<<<dim3((unsigned)((max_lines + 127) / 128), nrows), 128, 0, (cudaStream_t)stream>>>(pad, rows, z, axis);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_intensity_lowres_upsample(float* x, const float* pad, const rehr_irow* rows, int nrows, int z, int xs, int ys,
                                   const double* moments, rehr_stream stream) {
  if (!x || !pad || !moments || !rows_ok(rows, nrows) || z <= 0 || xs <= 0 || ys <= 0) return REHR_BAD_SHAPE;
  const long long len = (long long)z * xs * ys;
  intensity_lowres_upsample_kernel<<<dim3(ichunks(len), nrows), kIThreads, 0, (cudaStream_t)stream>>>(x, pad, rows, z, xs, ys, moments);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}
