// scipy's cubic B-spline prefilter of one line (elementwise.cu: spatial augmentation; intensity.cu: simulated low resolution).
#pragma once
#include <cuda_runtime.h>

namespace rehr {

// In place over p[0], p[inner], ..., p[(n - 1) * inner]: one causal + one anti-causal recursion with the pole z = sqrt(3) - 2 and
// MIRROR boundary initialisation, gain 6.  n >= 2.
__device__ __forceinline__ void bspline_prefilter_line(float* __restrict__ p, int n, long long inner) {
  const double z = -0.26794919243112270647;  // sqrt(3) - 2
  const double gain = 6.0;                   // (1 - z)(1 - 1/z)
  // causal initialisation, mirror boundary: c0 = sum_k z^k s[k] over the mirrored, periodised line (scipy _init_causal_mirror)
  const double zn1 = pow(z, (double)(n - 1));
  double c0 = gain * ((double)p[0] + zn1 * (double)p[(long long)(n - 1) * inner]);
  double zi = z;
  // the terms decay as z^i: beyond ~40 samples they are below fp64 resolution of the sum
  const int horizon = min(n - 1, 48);
  for (int i = 1; i < horizon; ++i) {
    c0 += gain * zi * ((double)p[(long long)i * inner] + zn1 * (double)p[(long long)(n - 1 - i) * inner]);
    zi *= z;
  }
  c0 /= 1.0 - zn1 * zn1;
  double prev = c0;
  p[0] = (float)c0;
  // the recursion runs in double and keeps the running value in a register; the stored coefficients are fp32
  double last2 = 0.0;
  for (int i = 1; i < n; ++i) {
    const double v = gain * (double)p[(long long)i * inner] + z * prev;
    if (i == n - 2) last2 = v;
    p[(long long)i * inner] = (float)v;
    prev = v;
  }
  if (n == 2) last2 = c0;
  double nxt = (z * last2 + prev) * z / (z * z - 1.0);   // anti-causal initialisation (mirror)
  p[(long long)(n - 1) * inner] = (float)nxt;
  for (int i = n - 2; i >= 0; --i) {
    const double v = z * (nxt - (double)p[(long long)i * inner]);
    p[(long long)i * inner] = (float)v;
    nxt = v;
  }
}

}  // namespace rehr
