// Shared device helpers and inline-PTX wrappers for the sm_100a kernels of libpcad.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#ifndef __CUDA_ARCH_FEAT_SM100_ALL
// Host pass / other passes: nothing to check. Device code in this library is sm_100a only.
#endif

namespace pcad {

typedef __nv_bfloat16 bf16;

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device setting: remember which devices have it for one kernel.
// `done` is a function-local static of the (templated) launcher, one per kernel instantiation.
template <typename Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, int bytes, unsigned long long& done) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (done & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done |= bit;
  return e;
}

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// ---------------------------------------------------------------------------------------------
// dtype traits
// ---------------------------------------------------------------------------------------------
template <typename T> struct ActT;
template <> struct ActT<bf16> {
  static __device__ __forceinline__ float to_f(bf16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ bf16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <> struct ActT<float> {
  static __device__ __forceinline__ float to_f(float v) { return v; }
  static __device__ __forceinline__ float from_f(float v) { return v; }
};

// 16-byte vector of activations: 8 bf16 or 4 float.
template <typename T> struct Vec16 { static constexpr int N = 16 / sizeof(T); };

template <typename T>
__device__ __forceinline__ void load16(const T* p, float (&out)[16 / sizeof(T)]) {
  uint4 raw = *reinterpret_cast<const uint4*>(p);
  if constexpr (sizeof(T) == 2) {
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      out[2 * i] = __uint_as_float(w[i] << 16);
      out[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  } else {
    out[0] = __uint_as_float(raw.x); out[1] = __uint_as_float(raw.y);
    out[2] = __uint_as_float(raw.z); out[3] = __uint_as_float(raw.w);
  }
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

template <typename T>
__device__ __forceinline__ void store16(T* p, const float (&v)[16 / sizeof(T)]) {
  uint4 raw;
  if constexpr (sizeof(T) == 2) {
    raw.x = pack_bf16x2(v[0], v[1]); raw.y = pack_bf16x2(v[2], v[3]);
    raw.z = pack_bf16x2(v[4], v[5]); raw.w = pack_bf16x2(v[6], v[7]);
  } else {
    raw.x = __float_as_uint(v[0]); raw.y = __float_as_uint(v[1]);
    raw.z = __float_as_uint(v[2]); raw.w = __float_as_uint(v[3]);
  }
  *reinterpret_cast<uint4*>(p) = raw;
}

// ---------------------------------------------------------------------------------------------
// math
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <bool PRECISE>
__device__ __forceinline__ float silu(float x) {
  if constexpr (PRECISE) {
    return x / (1.0f + expf(-x));
  } else {
    return x * rcp_approx(1.0f + ex2_approx(-x * kLog2e));
  }
}

// softplus with the reference's threshold (identity above 20) [selective_scan_fwd_kernel / F.softplus]
template <bool PRECISE>
__device__ __forceinline__ float softplus(float x) {
  if constexpr (PRECISE) {
    return x > 20.0f ? x : log1pf(expf(x));
  } else {
    float sp = lg2_approx(1.0f + ex2_approx(x * kLog2e)) * kLn2;
    return x > 20.0f ? x : sp;
  }
}

// ---------------------------------------------------------------------------------------------
// packed fp32x2 arithmetic (sm_100: FFMA2 / FMUL2 / FADD2 -- two fp32 lanes per issue slot)
// ---------------------------------------------------------------------------------------------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// 2^x for a pair of x <= 0 on the FMA/ALU pipes (no MUFU): round-to-nearest range reduction by the
// 1.5*2^23 magic add, degree-4 polynomial for 2^f on [-0.5, 0.5] with p(0) = 1 exactly (so slowly
// decaying states do not drift: relative error ~ |f| * 2.3e-5 near 0, 2.9e-6 worst case), exponent
// inserted by an integer shift-add.  x is clamped at -126 (result ~ 1e-38, i.e. 0 for the recurrence).
__device__ __forceinline__ f32x2 exp2_poly2(f32x2 x2) {
  float x0, x1;
  unpack2(x2, x0, x1);
  x0 = fmaxf(x0, -126.0f);
  x1 = fmaxf(x1, -126.0f);
  x2 = pack2(x0, x1);
  const f32x2 magic = pack2(12582912.0f, 12582912.0f);
  const f32x2 r2 = add2(x2, magic);                                  // magic + rint(x)
  const f32x2 n2 = add2(r2, pack2(-12582912.0f, -12582912.0f));      // rint(x)
  const f32x2 f2 = fma2(n2, pack2(-1.0f, -1.0f), x2);                // x - rint(x) in [-0.5, 0.5]
  f32x2 p = fma2(pack2(0.009582849219441414f, 0.009582849219441414f), f2, pack2(0.05590642988681793f, 0.05590642988681793f));
  p = fma2(p, f2, pack2(0.24024099111557007f, 0.24024099111557007f));
  p = fma2(p, f2, pack2(0.6931241750717163f, 0.6931241750717163f));
  p = fma2(p, f2, pack2(1.0f, 1.0f));
  float p0, p1, r0, r1;
  unpack2(p, p0, p1);
  unpack2(r2, r0, r1);
  p0 = __int_as_float(__float_as_int(p0) + (__float_as_int(r0) << 23));
  p1 = __int_as_float(__float_as_int(p1) + (__float_as_int(r1) << 23));
  return pack2(p0, p1);
}

#ifndef PCAD_POLY_DEG
#define PCAD_POLY_DEG 4
#endif
// 2^(d*a) for a pair of products in [-126, 0], entirely on the FMA/ALU pipes, with the multiply folded into the
// range reduction: r = fma(d, a, 1.5*2^23) rounds the exact product to the nearest integer n, f = fma(d, a, -n) is
// the exactly-rounded remainder in [-0.5, 0.5]; minimax polynomial for 2^f with p(0) = 1 (degree 4: 2.9e-6 max
// relative error, degree 3: 1.0e-4); the exponent is inserted by an integer shift-add.  6 (degree 4) packed
// FMA-pipe instructions more than the MUFU path's one FMUL2, against two MUFU.EX2 saved.
__device__ __forceinline__ f32x2 exp2_prod_poly2(f32x2 d2, f32x2 a2) {
  const f32x2 magic = pack2(12582912.0f, 12582912.0f);
  const f32x2 r2 = fma2(d2, a2, magic);                               // magic + rint(d*a)
  const f32x2 nn2 = fma2(r2, pack2(-1.0f, -1.0f), magic);             // -rint(d*a)
  const f32x2 f2 = fma2(d2, a2, nn2);                                 // d*a - rint(d*a)
#if PCAD_POLY_DEG == 3
  f32x2 p = fma2(pack2(0.055009059607982635f, 0.055009059607982635f), f2, pack2(0.2422109693288803f, 0.2422109693288803f));
  p = fma2(p, f2, pack2(0.6932829022407532f, 0.6932829022407532f));
#else
  f32x2 p = fma2(pack2(0.009582576341927052f, 0.009582576341927052f), f2, pack2(0.05590682849287987f, 0.05590682849287987f));
  p = fma2(p, f2, pack2(0.24024106562137604f, 0.24024106562137604f));
  p = fma2(p, f2, pack2(0.6931241154670715f, 0.6931241154670715f));
#endif
  p = fma2(p, f2, pack2(1.0f, 1.0f));
  float p0, p1, r0, r1;
  unpack2(p, p0, p1);
  unpack2(r2, r0, r1);
  p0 = __int_as_float(__float_as_int(p0) + (__float_as_int(r0) << 23));
  p1 = __int_as_float(__float_as_int(p1) + (__float_as_int(r1) << 23));
  return pack2(p0, p1);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------
// shared-memory address, cp.async, mbarrier, TMA, tcgen05 wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// 16-byte async copy global->shared; src_bytes = 0 zero-fills (used for out-of-range rows).
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// mbarrier wait that traps instead of spinning forever if a phase never completes (a wrong descriptor or byte count would
// otherwise hang the GPU; ~2^28 polls is seconds, far beyond any legitimate wait)
__device__ __forceinline__ void mbar_wait_or_trap(uint64_t* bar, uint32_t parity) {
  for (uint32_t i = 0; i < (1u << 28); ++i)
    if (mbar_try_wait(bar, parity)) return;
  asm volatile("trap;");
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, px;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2D tiled load: coordinates are (c0 = innermost/K element index, c1 = row index).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 3D tiled load: coordinates (c0 = innermost element index, c1 = row, c2 = outermost); out-of-range elements
// (negative or past-the-end coordinates included) are zero-filled and still count towards the barrier's tx bytes.
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// Prefetch of a 3D tile into L2 (no shared-memory destination, no barrier): the later tma_load_3d of the same box hits L2.
__device__ __forceinline__ void tma_prefetch_l2_3d(const CUtensorMap* m, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];\n" ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0),
               "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;\n" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;\n" ::"n"(N) : "memory");
}

// ---- tcgen05 / TMEM ----
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(smem_result)), "n"(COLS)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 (bf16 inputs, fp32 accumulate).
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
               : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 16 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// ---- cta_group::2 (CTA pair on one TPC) variants ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// In the shared::cluster window of a CTA pair, clearing bit 24 of a local shared address names the same offset in the
// even-ranked (leader) CTA (cute::Sm100MmaPeerBitMask).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
// 2D tiled load issued by either CTA of a pair; the bytes are credited to the LEADER's mbarrier at the same offset.
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(smem_result)), "n"(COLS)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_cg2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(COLS) : "memory");
}
// D[tmem of both CTAs] (+)= A[256 rows: 128 from each CTA's smem] * B[N cols: N/2 from each CTA's smem]; issued by the leader.
__device__ __forceinline__ void umma_bf16_ss_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
  const uint32_t zero = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(zero)
      : "memory");
}
// Arrive (once all previously issued MMAs of this thread have completed) on the mbarrier at this offset in BOTH CTAs.
__device__ __forceinline__ void umma_commit_cg2(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}
// Arrive on the mbarrier at this offset in the leader CTA (from either CTA of the pair).
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];\n" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}

// Shared-memory matrix descriptor for a K-major operand tile stored with the 128-byte swizzle
// (rows of 64 bf16 = 128 B; 8-row groups 1024 B apart).  Field layout: cute::UMMA::SmemDescriptor.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
  uint64_t desc = 0;
  desc |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address, bits [0,14)
  desc |= static_cast<uint64_t>(1) << 16;                      // leading byte offset (unused for swizzled K-major)
  desc |= static_cast<uint64_t>(1024 >> 4) << 32;              // stride byte offset: 8 rows * 128 B
  desc |= static_cast<uint64_t>(1) << 46;                      // descriptor version 1 (sm_100)
  desc |= static_cast<uint64_t>(2) << 61;                      // layout: SWIZZLE_128B
  return desc;
}

// Instruction descriptor for kind::f16 with bf16 A/B (both K-major), fp32 D.  cute::UMMA::InstrDescriptor.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4)                              // c_format = F32
         | (1u << 7)                            // a_format = BF16
         | (1u << 10)                           // b_format = BF16
         | (0u << 15) | (0u << 16)              // a_major = K, b_major = K
         | (static_cast<uint32_t>(N >> 3) << 17)  // n_dim
         | (static_cast<uint32_t>(M >> 4) << 24); // m_dim
}

// ---------------------------------------------------------------------------------------------
// host side: cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda at link time)
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}


// 3D row-major [n2][n1][n0] tensor of bf16 or fp32 (n0 contiguous, row pitch ld elements, n2 slices of n1 rows back to
// back), box = [1][box1][box0], no swizzle (or the 128-byte swizzle: box0 * element size must be 128), out-of-range
// elements read as zero.
inline bool make_tmap_3d(CUtensorMap* map, bool f32, const void* base, long long n0, long long n1, long long n2,
                         long long ld, int box0, int box1, bool swizzle128 = false) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  const cuuint64_t es = f32 ? 4 : 2;
  cuuint64_t gdim[3] = {static_cast<cuuint64_t>(n0), static_cast<cuuint64_t>(n1), static_cast<cuuint64_t>(n2)};
  cuuint64_t gstride[2] = {static_cast<cuuint64_t>(ld) * es, static_cast<cuuint64_t>(ld) * es * static_cast<cuuint64_t>(n1)};
  cuuint32_t box[3] = {static_cast<cuuint32_t>(box0), static_cast<cuuint32_t>(box1), 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3,
                   const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

}  // namespace pcad
