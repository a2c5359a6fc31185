// Thin inline-PTX wrappers for the sm_100a features the conv kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / ld / commit).
// Everything here is device-only and header-only.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace rehr {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a pipeline bug must surface as a CUDA error (trap), never as a hung GPU.
// `err` (global int, may be null) receives a role/site code before the trap.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 1.9 GHz
      if (err) atomicExch(err, code);
      __threadfence_system();
      __trap();
    }
  }
}

// ---------------------------------------------------------------- TMA loads
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const void* desc, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(const void* desc, uint64_t* bar, void* dst, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
      "%7}], [%2];"
      :
      : "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(desc)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {  // whole warp
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate. One thread issues.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once every tcgen05 op previously issued by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 16 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
      "%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor (sm_100 "version 1"). Byte quantities, 16 B granular.
//   layout: 0 none, 2 = 128B swizzle, 4 = 64B swizzle, 6 = 32B swizzle
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint32_t layout) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;  // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(layout & 7) << 61;
  return d;
}
__device__ __forceinline__ uint32_t swizzle_layout_for_bytes(int row_bytes) {
  return row_bytes == 128 ? 2u : (row_bytes == 64 ? 4u : 6u);
}
// Instruction descriptor for kind::f16 with bf16 A/B, fp32 D.
__device__ __forceinline__ uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;   // D format  = F32
  d |= 1u << 7;   // A format  = BF16
  d |= 1u << 10;  // B format  = BF16
  d |= static_cast<uint32_t>(a_mn_major & 1) << 15;
  d |= static_cast<uint32_t>(b_mn_major & 1) << 16;
  d |= static_cast<uint32_t>(N >> 3) << 17;
  d |= static_cast<uint32_t>(M >> 4) << 24;
  return d;
}

// Instruction descriptor for kind::f16 with 16-bit A/B of ONE format (fp16: format code 0, bf16: 1; the two operands must share
// the format -- mixed fp16 x bf16 raises "illegal instruction" on B200, tools/umma_mixed_probe.cu), fp32 D.
__device__ __forceinline__ uint32_t make_idesc_16(int M, int N, int a_mn_major, int b_mn_major, int fp16) {
  uint32_t d = make_idesc_bf16(M, N, a_mn_major, b_mn_major);
  if (fp16) d &= ~((1u << 7) | (1u << 10));
  return d;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

// 16-bit activation storage formats (rehr_tensor.dtype): 0 = bf16, 1 = fp16.  fp16 stores saturate to +-65504 instead of
// overflowing to inf (cvt.rn.satfinite), loads are exact in fp32 for both.
__device__ __forceinline__ uint32_t pack_f16x2_sat(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack16x2(float lo, float hi, int fp16) {
  return fp16 ? pack_f16x2_sat(lo, hi) : pack_bf16x2(lo, hi);
}
__device__ __forceinline__ unsigned short pack16(float v, int fp16) {
  return (unsigned short)(pack16x2(v, 0.f, fp16) & 0xffffu);
}
__device__ __forceinline__ float2 unpack16x2(uint32_t u, int fp16) {
  if (fp16) {
    float2 r;
    asm("{\n\t.reg .f16 lo, hi;\n\tmov.b32 {lo, hi}, %2;\n\tcvt.f32.f16 %0, lo;\n\tcvt.f32.f16 %1, hi;\n\t}" : "=f"(r.x), "=f"(r.y) : "r"(u));
    return r;
  }
  return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
}
__device__ __forceinline__ float unpack16(unsigned short u, int fp16) { return unpack16x2((uint32_t)u, fp16).x; }

// One slot of the saturation record (layout shared with rehrseg_b200/rangecheck.py: 16 bytes, count then max bits).
struct RangeSlot {
  unsigned long long count;
  unsigned int max_bits;
  unsigned int pad;
};

// fp16 saturation record (rehr_range_sink): a value saturates when it is at least the smallest magnitude round-to-nearest
// would take to inf, or NaN -- on the bits of |v|: >= those of 65520.f (NaN sorts above inf).  The check only observes; the
// stores are unchanged.  Per warp, one ballot on the largest |v| of each lane decides; only when some lane saw a saturated value
// are the values counted and ONE atomic pair per warp issued (lane counts added, largest |v| bits as atomicMax).
static constexpr uint32_t kRangeSatBits = 0x477FF000u;  // __float_as_uint(65520.f)
__device__ __forceinline__ uint32_t range_abs_bits(float v) { return __float_as_uint(v) & 0x7FFFFFFFu; }
__device__ __forceinline__ void range_fold(float v, uint32_t& cnt, uint32_t& mbits) {
  const uint32_t b = range_abs_bits(v);
  if (b >= kRangeSatBits) {
    ++cnt;
    mbits = max(mbits, b);
  }
}
__device__ __forceinline__ void range_flush(RangeSlot* s, uint32_t cnt, uint32_t mbits) {
  const uint32_t mask = __activemask();
  if (__ballot_sync(mask, cnt != 0u) == 0u) return;
  const uint32_t total = __reduce_add_sync(mask, cnt);
  const uint32_t m = __reduce_max_sync(mask, mbits);
  uint32_t lane;
  asm("mov.u32 %0, %%laneid;" : "=r"(lane));
  if (lane == (uint32_t)(__ffs(mask) - 1)) {
    atomicAdd(&s->count, (unsigned long long)total);
    atomicMax(&s->max_bits, m);
  }
}
// the first `n` of K values about to be stored (fast path: one max per value and a ballot)
template <int K>
__device__ __forceinline__ void range_check(RangeSlot* s, const float* f, int n = K) {
  uint32_t m = 0;
#pragma unroll
  for (int i = 0; i < K; ++i)
    if (i < n) m = max(m, range_abs_bits(f[i]));
  const uint32_t mask = __activemask();
  if (__ballot_sync(mask, m >= kRangeSatBits) == 0u) return;
  uint32_t cnt = 0, mbits = 0;
#pragma unroll
  for (int i = 0; i < K; ++i)
    if (i < n) range_fold(f[i], cnt, mbits);
  range_flush(s, cnt, mbits);
}

}  // namespace rehr

namespace rehr {
// registers -> TMEM: this warp's 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// TMEM -> registers, 32 consecutive columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
}  // namespace rehr
