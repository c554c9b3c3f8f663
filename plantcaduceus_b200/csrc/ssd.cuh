// Mamba-2 / SSD mixer kernels (PlantCAD2: 64-wide heads, 64 states, one B/C group) for the strand-major layout.
//
//   [EXT] mamba_ssm Mamba2.forward:  zxbcdt = in_proj(u);  xBC = silu(conv1d(xBC));
//         y = mamba_chunk_scan_combined(x, dt, A, B, C, D, dt_bias, dt_softplus=True);  y = RMSNormGated(y, z);  out_proj(y)
//   [EXT] Caduceus BiMambaWrapper (strategy "add", tied in/out projections): fwd(u) + flip_L(rev(flip_L(u)))
//
// Per head h (scalar decay): dt_t = softplus(dt_raw_t + dt_bias_h); S <- exp(dt_t A_h) S + dt_t x_t (x) B_t;
// y_t = S C_t + D_h x_t, with S a [P = 64] x [N = 64] fp32 state.  Both time directions are computed from the
// same conv outputs layout as the Mamba-1 path (direction by index math, nothing is flipped in memory).
//
// ssd_chunk_tc_kernel (bf16): the chunked "state-space dual" form on the tcgen05 tensor cores.  A CTA owns one sequence,
// one direction and a PAIR of heads (B and C are shared by all heads, so the pair shares their tiles and the C B^T
// product); it walks the sequence in chunks of Q = 128 positions in scan order and carries the two heads' states in
// registers (thread = one (head, p) state row, half of the 64 states).  Per chunk, with cum_t the cumulative log-decay
// in scan order and all tiles staged by TMA with the 128-byte swizzle:
//   GEMM1  G = C B^T                       128 x 128 x 64   (A, B K-major)                        -> TMEM
//   per head:  M[t,s] = G[t,s] exp(cum_t - cum_s) dt_s  for s not after t (else 0), bf16, written K-major into smem
//              (32 x 32 blocks off the diagonal: exp(cum_t - r) exp(r - cum_s) with r the block edge, both factors <= 1, so the
//              per-element exponential is two multiplies there; blocks on the masked side are zero-filled)
//   GEMM2  Y  = M X                         128 x 64 x 128   (B operand = the x tile as loaded: MN-major)
//   GEMM4  Y' = C S_prev^T                  128 x 64 x 64    (S_prev rounded to bf16 in smem, K-major)
//          y_t = Y + exp(cum_t) Y' + D x_t  -> global (bf16)
//   GEMM3  S_c = (X w)^T B                  (2 x 64) x 64 x 128  (both operands MN-major; w_s = exp(cum_end - cum_s) dt_s)
//          S <- exp(cum_end) S + S_c        (registers)
// The reverse direction reads the same natural-order tiles with suffix sums and the upper-triangular mask.
//
// ssd_scan_seq_kernel<T>: the plain sequential recurrence (fp32 state in registers), used by the fp32 parity mode and as the
// checker of the tensor-core kernel in tests.
//
// gated_norm_sum_kernel<T>: RMSNormGated (norm_before_gate = False, one group) of each direction's y with the shared gate z,
// and the BiMamba "add" of the two directions, in one pass: out = rms(y_f silu(z)) w_f + rms(y_r silu(z)) w_r.
#pragma once

#include <cuda_fp16.h>

#include "common.cuh"

namespace pcad {

constexpr int kSsdQ = 128;        // chunk length (positions)
constexpr int kSsdP = 64;         // head dim
constexpr int kSsdN = 64;         // state size
constexpr int kSsdThreads = 256;
constexpr int kSsdTile = kSsdQ * 64 * 2;   // one [128 rows x 64 bf16] swizzled tile: 16 KB

// ---------------------------------------------------------------------------------------------------------------------
// sequential recurrence (parity mode / checker)
// ---------------------------------------------------------------------------------------------------------------------
// grid (H, S, 2); block 64 threads: thread = p.  xbc_*: [S*L, ld_xbc] with x at [0, E), B at [E, E+64), C at [E+64, E+128);
// dt_raw: [S*L, ld_dt] (column = head); y_*: [S*L, E].
template <typename T>
__global__ void __launch_bounds__(64)
ssd_scan_seq_kernel(const T* __restrict__ xbc_f, const T* __restrict__ xbc_r, long long ld_xbc, const T* __restrict__ dt_raw,
                    long long ld_dt, const float* __restrict__ A_f, const float* __restrict__ D_f, const float* __restrict__ bias_f,
                    const float* __restrict__ A_r, const float* __restrict__ D_r, const float* __restrict__ bias_r,
                    T* __restrict__ y_f, T* __restrict__ y_r, int L, int E) {
  constexpr int TT = 16;
  __shared__ float sB[TT][kSsdN], sC[TT][kSsdN], sdt[TT];
  const int h = blockIdx.x, seq = blockIdx.y, dir = blockIdx.z, p = threadIdx.x;
  const T* xbc = dir ? xbc_r : xbc_f;
  T* y = dir ? y_r : y_f;
  const float A = (dir ? A_r : A_f)[h], D = (dir ? D_r : D_f)[h], bias = (dir ? bias_r : bias_f)[h];
  const long long row0 = static_cast<long long>(seq) * L;
  float S[kSsdN];
#pragma unroll
  for (int n = 0; n < kSsdN; ++n) S[n] = 0.f;
  for (int i0 = 0; i0 < L; i0 += TT) {
    const int nst = min(TT, L - i0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < nst * kSsdN; idx += 64) {
      const int j = idx / kSsdN, n = idx % kSsdN;
      const int pos = dir ? L - 1 - (i0 + j) : i0 + j;
      sB[j][n] = ActT<T>::to_f(xbc[(row0 + pos) * ld_xbc + E + n]);
      sC[j][n] = ActT<T>::to_f(xbc[(row0 + pos) * ld_xbc + E + kSsdN + n]);
    }
    if (threadIdx.x < nst) {
      const int pos = dir ? L - 1 - (i0 + threadIdx.x) : i0 + threadIdx.x;
      sdt[threadIdx.x] = softplus<true>(ActT<T>::to_f(dt_raw[(row0 + pos) * ld_dt + h]) + bias);
    }
    __syncthreads();
    for (int j = 0; j < nst; ++j) {
      const int pos = dir ? L - 1 - (i0 + j) : i0 + j;
      const float xv = ActT<T>::to_f(xbc[(row0 + pos) * ld_xbc + h * kSsdP + p]);
      const float dtv = sdt[j];
      const float dA = expf(dtv * A), dx = dtv * xv;
      float acc = D * xv;
#pragma unroll
      for (int n = 0; n < kSsdN; ++n) {
        S[n] = fmaf(dA, S[n], dx * sB[j][n]);
        acc = fmaf(S[n], sC[j][n], acc);
      }
      y[(row0 + pos) * E + h * kSsdP + p] = ActT<T>::from_f(acc);
    }
  }
}

__device__ __forceinline__ void unpack8(const uint4& raw, float (&v)[8]) {
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}

// one 32-bit word of two bf16 <-> a packed fp32 pair (FMUL2 / FFMA2 operate on the pair in one issue slot)
__device__ __forceinline__ f32x2 bf16x2_to_f32x2(uint32_t w) {
  return pack2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ uint32_t f32x2_to_bf16x2(f32x2 v) {
  float lo, hi;
  unpack2(v, lo, hi);
  return pack_bf16x2(lo, hi);
}
__device__ __forceinline__ f32x2 pack2u(uint32_t lo, uint32_t hi) { return pack2(__uint_as_float(lo), __uint_as_float(hi)); }

// ---------------------------------------------------------------------------------------------------------------------
// gated RMSNorm of both directions + add
// ---------------------------------------------------------------------------------------------------------------------
// One warp per row; two passes over the row (the second hits L1/L2).  z: [rows, *] with pitch ldz.
template <typename T, bool PRECISE>
__global__ void __launch_bounds__(256)
gated_norm_sum_kernel(const T* __restrict__ y_f, const T* __restrict__ y_r, const T* __restrict__ z, long long ldz,
                      const float* __restrict__ w_f, const float* __restrict__ w_r, T* __restrict__ out, long long rows, int E,
                      float eps) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  constexpr int V = 16 / sizeof(T);
  const T* yf = y_f + row * E;
  const T* yr = y_r + row * E;
  const T* zz = z + row * ldz;
  float ssf = 0.f, ssr = 0.f;
  for (int j = lane * V; j < E; j += 32 * V) {
    float a[V], b[V], g[V];
    load16<T>(yf + j, a);
    load16<T>(yr + j, b);
    load16<T>(zz + j, g);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      const float s = silu<PRECISE>(g[k]);
      const float af = a[k] * s, ar = b[k] * s;
      ssf = fmaf(af, af, ssf);
      ssr = fmaf(ar, ar, ssr);
    }
  }
  ssf = warp_sum(ssf);
  ssr = warp_sum(ssr);
  const float rf = rsqrtf(ssf / static_cast<float>(E) + eps), rr = rsqrtf(ssr / static_cast<float>(E) + eps);
  T* o = out + row * E;
  for (int j = lane * V; j < E; j += 32 * V) {
    float a[V], b[V], g[V], wf[V], wr[V], res[V];
    load16<T>(yf + j, a);
    load16<T>(yr + j, b);
    load16<T>(zz + j, g);
#pragma unroll
    for (int k = 0; k < V; k += 4) {
      const float4 q = *reinterpret_cast<const float4*>(w_f + j + k);
      const float4 r = *reinterpret_cast<const float4*>(w_r + j + k);
      wf[k] = q.x; wf[k + 1] = q.y; wf[k + 2] = q.z; wf[k + 3] = q.w;
      wr[k] = r.x; wr[k + 1] = r.y; wr[k + 2] = r.z; wr[k + 3] = r.w;
    }
#pragma unroll
    for (int k = 0; k < V; ++k) {
      const float s = silu<PRECISE>(g[k]);
      float nf = a[k] * s * rf * wf[k], nr = b[k] * s * rr * wr[k];
      if constexpr (sizeof(T) == 2) {   // each direction's norm output is a bf16 tensor in the reference
        nf = __bfloat162float(__float2bfloat16_rn(nf));
        nr = __bfloat162float(__float2bfloat16_rn(nr));
      }
      res[k] = nf + nr;
    }
    store16<T>(o + j, res);
  }
}

// bf16 variant with the gate cached.  The generic kernel above is MUFU-bound in bf16 (ncu: XU pipe 82 %: SiLU = ex2 + rcp per
// element, evaluated in both passes) while its second pass already hits L2 (DRAM reads = one pass).  Here SiLU(z) is evaluated
// once and parked as fp16 in registers (CH 16-byte vectors per lane, E <= 256 CH; 2^-11 relative, below the bf16 rounding of
// the output, down to |SiLU(z)| = 2^-14; below that fp16 is subnormal and the gate is exact only to 2^-25 absolute, which is
// 2^-25 of |y| rstd |w| on such an element; the statistics use the un-rounded fp32 value); y_f / y_r are re-read in the second pass (L2).  Keeping all
// three tensors in registers instead (one DRAM/L2 pass, 126-230 registers) measured slower: 1.0 vs 0.71 ms per layer at
// E = 1536 -- too few warps left to overlap the loads with the arithmetic.
template <int CH>
__global__ void __launch_bounds__(256)
gated_norm_sum_regs_kernel(const bf16* __restrict__ y_f, const bf16* __restrict__ y_r, const bf16* __restrict__ z, long long ldz,
                           const float* __restrict__ w_f, const float* __restrict__ w_r, bf16* __restrict__ out, long long rows,
                           int E, float eps) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const bf16* yf = y_f + row * E;
  const bf16* yr = y_r + row * E;
  const bf16* zz = z + row * ldz;
  uint4 rg[CH];
  float ssf = 0.f, ssr = 0.f;
#pragma unroll
  for (int c = 0; c < CH; ++c) {
    const int j = (c * 32 + lane) * 8;
    rg[c] = make_uint4(0u, 0u, 0u, 0u);
    if (j >= E) continue;
    float a[8], b[8], g[8];
    unpack8(*reinterpret_cast<const uint4*>(yf + j), a);
    unpack8(*reinterpret_cast<const uint4*>(yr + j), b);
    unpack8(*reinterpret_cast<const uint4*>(zz + j), g);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      g[k] = silu<false>(g[k]);
      const float af = a[k] * g[k], ar = b[k] * g[k];
      ssf = fmaf(af, af, ssf);
      ssr = fmaf(ar, ar, ssr);
    }
    __half2 h0 = __floats2half2_rn(g[0], g[1]), h1 = __floats2half2_rn(g[2], g[3]);
    __half2 h2 = __floats2half2_rn(g[4], g[5]), h3 = __floats2half2_rn(g[6], g[7]);
    rg[c] = make_uint4(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1), *reinterpret_cast<uint32_t*>(&h2),
                       *reinterpret_cast<uint32_t*>(&h3));
  }
  ssf = warp_sum(ssf);
  ssr = warp_sum(ssr);
  const float rf = rsqrtf(ssf / static_cast<float>(E) + eps), rr = rsqrtf(ssr / static_cast<float>(E) + eps);
  bf16* o = out + row * E;
#pragma unroll
  for (int c = 0; c < CH; ++c) {
    const int j = (c * 32 + lane) * 8;
    if (j >= E) continue;
    float a[8], b[8], g[8], res[8];
    unpack8(*reinterpret_cast<const uint4*>(yf + j), a);
    unpack8(*reinterpret_cast<const uint4*>(yr + j), b);
    {
      const uint32_t w[4] = {rg[c].x, rg[c].y, rg[c].z, rg[c].w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
        g[2 * i] = f.x;
        g[2 * i + 1] = f.y;
      }
    }
    const float4 f0 = *reinterpret_cast<const float4*>(w_f + j), f1 = *reinterpret_cast<const float4*>(w_f + j + 4);
    const float4 r0 = *reinterpret_cast<const float4*>(w_r + j), r1 = *reinterpret_cast<const float4*>(w_r + j + 4);
    const float wf[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
    const float wr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float nf = __bfloat162float(__float2bfloat16_rn(a[k] * g[k] * rf * wf[k]));   // each direction's norm output is bf16
      const float nr = __bfloat162float(__float2bfloat16_rn(b[k] * g[k] * rr * wr[k]));
      res[k] = nf + nr;
    }
    store16<bf16>(o + j, res);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// chunked SSD on tcgen05
// ---------------------------------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor for an MN-major operand stored with the 128-byte swizzle: K index = row (128 bytes each,
// 8-row groups 1024 B apart = SBO), MN index = the 64 bf16 of a row; further 64-element MN atoms are lbo_bytes apart
// (cute::UMMA canonical layout  Swizzle<3,4,3> o ((8,8,m),(8,k)) : ((1,8,LBO),(64,SBO))  in elements).
__device__ __forceinline__ uint64_t make_smem_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t desc = 0;
  desc |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  desc |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  desc |= static_cast<uint64_t>(1024 >> 4) << 32;
  desc |= static_cast<uint64_t>(1) << 46;
  desc |= static_cast<uint64_t>(2) << 61;
  return desc;
}
__host__ __device__ constexpr uint32_t make_idesc_bf16_major(int M, int N, int a_mn, int b_mn) {
  return make_idesc_bf16(M, N) | (static_cast<uint32_t>(a_mn) << 15) | (static_cast<uint32_t>(b_mn) << 16);
}

struct SsdSmem {
  static constexpr int kX0 = 0, kX1 = kSsdTile, kB = 2 * kSsdTile, kC = 3 * kSsdTile, kM = 4 * kSsdTile;   // M: 2 tiles
  static constexpr int kS = 6 * kSsdTile;                  // one head's state, bf16 [64 p][64 n] (8 KB)
  static constexpr int kSmall = kS + 8192;
  static constexpr int kDts = kSmall;                      // float [2][128]
  static constexpr int kCums = kDts + 1024;                // float [2][128]
  static constexpr int kColf = kCums + 1024;               // float [2][4][128]: column factors of the off-diagonal blocks
  static constexpr int kWsum = kColf + 4096;               // float [2][4] + tot [2]
  static constexpr int kBars = kWsum + 64;                 // 2 mbarriers + tmem ptr
  static constexpr int kBytes = kBars + 64;
};


// grid (H / 2, S, 2 directions); tm_f / tm_r: 3-D maps [S][L][ld_xbc] of the two directions' conv outputs, box [1][128][64],
// 128-byte swizzle.  dt_raw [S*L, ld_dt] (column = head).  y_* [S*L, E] un-gated outputs (D skip included).
__global__ void __launch_bounds__(kSsdThreads, 2)
ssd_chunk_tc_kernel(const __grid_constant__ CUtensorMap tm_f, const __grid_constant__ CUtensorMap tm_r,
                    const bf16* __restrict__ dt_raw, long long ld_dt, const float* __restrict__ A_f,
                    const float* __restrict__ D_f, const float* __restrict__ bias_f, const float* __restrict__ A_r,
                    const float* __restrict__ D_r, const float* __restrict__ bias_r, bf16* __restrict__ y_f,
                    bf16* __restrict__ y_r, int L, int E) {
  extern __shared__ uint8_t ssd_smem_raw[];
  // 1024-byte alignment for the swizzled tiles by pointer arithmetic on the array itself, so that the compiler keeps every
  // access in the shared address space (LDS / STS, not generic LD / ST)
  uint8_t* sm = ssd_smem_raw + ((1024u - (smem_u32(ssd_smem_raw) & 1023u)) & 1023u);
  float* dts = reinterpret_cast<float*>(sm + SsdSmem::kDts);      // [2][128]  dt (after softplus), 0 for rows past L
  float* cums = reinterpret_cast<float*>(sm + SsdSmem::kCums);    // [2][128]  cumulative dt*A*log2(e) in scan order
  float* colf = reinterpret_cast<float*>(sm + SsdSmem::kColf);    // [2][4][128] (head, row block I, column s): 2^(r_I - cum_s) dt_s
  float* wsum = reinterpret_cast<float*>(sm + SsdSmem::kWsum);    // [2][4] warp sums, then tot[2] at +8
  uint64_t* tma_bar = reinterpret_cast<uint64_t*>(sm + SsdSmem::kBars);
  uint64_t* mma_bar = tma_bar + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(mma_bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int hp = blockIdx.x, seq = blockIdx.y, dir = blockIdx.z;
  const CUtensorMap* tm = dir ? &tm_r : &tm_f;
  bf16* yout = dir ? y_r : y_f;
  const float* Ap = dir ? A_r : A_f;
  const float* Dp = dir ? D_r : D_f;
  const float* bp = dir ? bias_r : bias_f;
  const long long row0 = static_cast<long long>(seq) * L;
  const int nch = (L + kSsdQ - 1) / kSsdQ;

  if (tid == 0) {
    mbar_init(tma_bar, 1);
    mbar_init(mma_bar, 1);
    fence_mbar_init();
    tma_prefetch_desc(tm);
  }
  if (warp == 1) {
    tmem_alloc<256>(tmem_ptr);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;
  // TMEM columns: [0,128) G (later [0,64) S_c), [128,192) Y, [192,256) Y'
  const uint32_t sm_addr = smem_u32(sm);

  // this thread's accumulator row / column half, and (for the state) its (head, p) row
  const int trow = 32 * (warp & 3) + lane;
  const int half = warp >> 2;
  const uint32_t t_lane = tmem + (static_cast<uint32_t>(32 * (warp & 3)) << 16);
  float Srun[32];
#pragma unroll
  for (int n = 0; n < 32; ++n) Srun[n] = 0.f;

  // per-thread constants of the dt phase: thread = (head, position in chunk)
  const int dh = tid >> 7, dtp = tid & 127;
  const int head_d = 2 * hp + dh;
  const float A_l2 = Ap[head_d] * kLog2e, bias_d = bp[head_d];

  // raw dt of the chunk about to be processed, fetched one iteration ahead and kept as RAW BITS until it is used (converting
  // at the load would make the thread wait for the load there and then: its global-load latency must stay off the critical path)
  constexpr uint32_t kDtPastEnd = 0xff80u;   // bf16 -inf: row past the end (dt = 0)
  auto load_dt = [&](int it_) -> uint32_t {
    if (it_ >= nch) return kDtPastEnd;
    const int c_ = dir ? nch - 1 - it_ : it_;
    const int pos = c_ * kSsdQ + dtp;
    return pos < L ? static_cast<uint32_t>(reinterpret_cast<const unsigned short*>(dt_raw)[(row0 + pos) * ld_dt + head_d]) : kDtPastEnd;
  };
  uint32_t dt_next = load_dt(0);
  uint32_t tma_phase = 0, mma_phase = 0;
  constexpr uint32_t idesc_g1 = make_idesc_bf16_major(128, 128, 0, 0);
  constexpr uint32_t idesc_g2 = make_idesc_bf16_major(128, 64, 0, 1);
  constexpr uint32_t idesc_g3 = make_idesc_bf16_major(128, 64, 1, 1);
  constexpr uint32_t idesc_g4 = make_idesc_bf16_major(128, 64, 0, 0);

  for (int it = 0; it < nch; ++it) {
    const int c = dir ? nch - 1 - it : it;
    const int p0 = c * kSsdQ;
    if (warp == 0 && elect_one()) {   // whole warp, then elect.sync: issue instructions back to back
      mbar_arrive_expect_tx(tma_bar, 4 * kSsdTile);
      tma_load_3d(sm + SsdSmem::kX0, tm, tma_bar, (2 * hp) * kSsdP, p0, seq);
      tma_load_3d(sm + SsdSmem::kX1, tm, tma_bar, (2 * hp + 1) * kSsdP, p0, seq);
      tma_load_3d(sm + SsdSmem::kB, tm, tma_bar, E, p0, seq);
      tma_load_3d(sm + SsdSmem::kC, tm, tma_bar, E + kSsdN, p0, seq);
      // the tiles are single-buffered (shared memory is what caps the kernel at 2 CTAs/SM), so the next chunk's load cannot be
      // issued early; pulling it into L2 now at least takes the HBM latency off the next iteration's critical path
      if (it + 1 < nch) {
        const int pn = (dir ? nch - 2 - it : it + 1) * kSsdQ;
        tma_prefetch_l2_3d(tm, (2 * hp) * kSsdP, pn, seq);
        tma_prefetch_l2_3d(tm, (2 * hp + 1) * kSsdP, pn, seq);
        if (hp == 0) {   // B and C are shared by the head pairs of this (sequence, direction): one CTA prefetches them
          tma_prefetch_l2_3d(tm, E, pn, seq);
          tma_prefetch_l2_3d(tm, E + kSsdN, pn, seq);
        }
      }
    }
    // ---- dt, log-decay and its cumulative sum in scan order
    {
      const float raw = __uint_as_float(dt_next << 16);
      dt_next = load_dt(it + 1);
      const float dtv = raw > -1e29f ? softplus<true>(raw + bias_d) : 0.f;
      float v = dtv * A_l2;
      if (dir == 0) {
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const float u = __shfl_up_sync(0xffffffffu, v, o);
          if (lane >= o) v += u;
        }
        if (lane == 31) wsum[dh * 4 + (warp & 3)] = v;
      } else {
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const float u = __shfl_down_sync(0xffffffffu, v, o);
          if (lane + o < 32) v += u;
        }
        if (lane == 0) wsum[dh * 4 + (warp & 3)] = v;
      }
      dts[dh * 128 + dtp] = dtv;
      __syncthreads();
      float off = 0.f;
      const int wq = warp & 3;
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        const float s = wsum[dh * 4 + w];
        if (dir == 0 ? (w < wq) : (w > wq)) off += s;
      }
      const float cum_s = v + off;
      cums[dh * 128 + dtp] = cum_s;
      if (dtp == 0) wsum[8 + dh] = wsum[dh * 4] + wsum[dh * 4 + 1] + wsum[dh * 4 + 2] + wsum[dh * 4 + 3];
      // Column factors for the 32 x 32 blocks that lie wholly on the unmasked side of the diagonal.  With r_I the cumulative
      // log-decay at the edge of row block I that faces this column (= a sum of whole-warp totals), the decay from s to a row t
      // of block I splits as 2^(cum_t - r_I) 2^(r_I - cum_s) with BOTH exponents <= 0: no overflow however fast the state
      // forgets, and the per-element exponential of those blocks becomes two multiplies in build_M.
      {
        float r = 0.f;   // r_I, accumulated over the row blocks in scan order
#pragma unroll
        for (int k = 1; k < 4; ++k) {
          const int I = dir == 0 ? k : 3 - k;                 // row blocks that come after this column's block in scan order
          r += wsum[dh * 4 + (dir == 0 ? k - 1 : 4 - k)];     // fwd: r_I = sum of warps < I;  rev: sum of warps > I
          const bool needed = dir == 0 ? (wq < I) : (wq > I);
          if (needed) colf[(dh * 4 + I) * 128 + dtp] = ex2_approx(r - cum_s) * dtv;
        }
      }
    }
    __syncthreads();
    // ---- GEMM1: G = C B^T
    mbar_wait_or_trap(tma_bar, tma_phase);
    tma_phase ^= 1;
    if (warp == 0 && elect_one()) {   // whole warp, then elect.sync: issue instructions back to back
      tc_fence_after();
      const uint64_t da = make_smem_desc_sw128(sm_addr + SsdSmem::kC), db = make_smem_desc_sw128(sm_addr + SsdSmem::kB);
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_bf16_ss(tmem, da + 2 * k, db + 2 * k, idesc_g1, k ? 1u : 0u);
      umma_commit(mma_bar);
    }
    mbar_wait_or_trap(mma_bar, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();

    // ---- per-head pieces of the chunk.  Phases (one barrier each): [M_0, S_0] | MMA_0 | [y_0, M_1, S_1] | MMA_1 | [y_1, Xw] |
    //      MMA_3 | state -- the epilogue of one head shares a phase with the next head's operand build, so the light rows of the
    //      triangular M build have the (uniform) epilogue to do while the heavy rows finish.
    // M = G o decay o dt, bf16, K-major swizzled (tile = columns / 64).  A thread owns row `trow` and the four 16-column
    // pieces {half, half + 2, half + 4, half + 6}: interleaved, so the two warps that share a row block split its diagonal
    // block.  A piece lies in column block J = piece / 2; against the row block I (warp-uniform):
    //   masked side of the diagonal -> zero-filled, no TMEM load;
    //   J == I                      -> per element 2^(cum_t - cum_s) dt_s under the triangular mask;
    //   unmasked side               -> G[t,s] * rowf_t * colf_I[s]: two multiplies per element (see the dt phase).
    // Piece k + 1 is in flight from TMEM while piece k is being computed.
    auto build_M = [&](int h) {
      const float cum_t = cums[h * 128 + trow];
      const int I = warp & 3;
      uint8_t* mbase = sm + SsdSmem::kM + trow * 128;
      // r_I (edge of this row block facing the unmasked columns) from the whole-warp totals, and this row's factor
      float rI = 0.f;
#pragma unroll
      for (int w = 0; w < 4; ++w)
        if (dir == 0 ? (w < I) : (w > I)) rI += wsum[h * 4 + w];
      const float rowf = ex2_approx(cum_t - rI);
      const f32x2 rowf2 = pack2(rowf, rowf), cumt2 = pack2(cum_t, cum_t), neg1 = pack2(-1.0f, -1.0f);
      const float* cf = colf + (h * 4 + I) * 128;
      auto kind = [&](int kk) {   // 0 masked, 1 diagonal, 2 full
        const int J = (2 * kk + half) >> 1;
        if (J == I) return 1;
        return (dir == 0 ? (J < I) : (J > I)) ? 2 : 0;
      };
      uint32_t r[2][16];
      if (kind(0)) tmem_ld_32x32b_x16(t_lane + 16 * half, r[0]);
      tmem_ld_wait();
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const int piece = 2 * kk + half;
        const int s0 = 16 * piece;
        uint8_t* mrow = mbase + (piece >> 2) * kSsdTile;
        const int c0 = 2 * (piece & 3);                       // first 16-byte chunk of the piece inside its tile row
        if (kk + 1 < 4 && kind(kk + 1)) tmem_ld_32x32b_x16(t_lane + s0 + 32, r[(kk + 1) & 1]);
        const int kd = kind(kk);
        if (kd == 0) {
#pragma unroll
          for (int g = 0; g < 2; ++g)
            *reinterpret_cast<uint4*>(mrow + (((c0 + g) ^ (trow & 7)) << 4)) = make_uint4(0u, 0u, 0u, 0u);
        } else if (kd == 2) {
#pragma unroll
          for (int g = 0; g < 2; ++g) {   // (G rowf) colf on packed pairs: two multiplies per PAIR of elements
            const float4 f0 = *reinterpret_cast<const float4*>(&cf[s0 + 8 * g]);
            const float4 f1 = *reinterpret_cast<const float4*>(&cf[s0 + 8 * g + 4]);
            const f32x2 ff[4] = {pack2(f0.x, f0.y), pack2(f0.z, f0.w), pack2(f1.x, f1.y), pack2(f1.z, f1.w)};
            uint32_t ow[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
              ow[q] = f32x2_to_bf16x2(mul2(mul2(pack2u(r[kk & 1][8 * g + 2 * q], r[kk & 1][8 * g + 2 * q + 1]), rowf2), ff[q]));
            *reinterpret_cast<uint4*>(mrow + (((c0 + g) ^ (trow & 7)) << 4)) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
          }
        } else {
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            float v[8];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const float4 cs = *reinterpret_cast<const float4*>(&cums[h * 128 + s0 + 8 * g + 4 * q]);
              const float4 ds = *reinterpret_cast<const float4*>(&dts[h * 128 + s0 + 8 * g + 4 * q]);
              const f32x2 cc2[2] = {pack2(cs.x, cs.y), pack2(cs.z, cs.w)}, dd2[2] = {pack2(ds.x, ds.y), pack2(ds.z, ds.w)};
#pragma unroll
              for (int e2 = 0; e2 < 2; ++e2) {   // pairs: cum_t - cum_s, the two exponentials, G e dt
                float x0, x1, v0, v1;
                unpack2(fma2(cc2[e2], neg1, cumt2), x0, x1);
                const f32x2 ee = pack2(ex2_approx(x0), ex2_approx(x1));
                const int ri = 8 * g + 4 * q + 2 * e2;
                unpack2(mul2(mul2(pack2u(r[kk & 1][ri], r[kk & 1][ri + 1]), ee), dd2[e2]), v0, v1);
                const int s = s0 + ri;
                v[4 * q + 2 * e2] = (dir == 0 ? (s <= trow) : (s >= trow)) ? v0 : 0.f;
                v[4 * q + 2 * e2 + 1] = (dir == 0 ? (s + 1 <= trow) : (s + 1 >= trow)) ? v1 : 0.f;
              }
            }
            uint4 o;
            o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
            o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
            *reinterpret_cast<uint4*>(mrow + (((c0 + g) ^ (trow & 7)) << 4)) = o;
          }
        }
        tmem_ld_wait();
      }
    };
    // this head's carried state, bf16 K-major [p][n] (written by the threads that hold it)
    auto write_S = [&](int h) {
      if (it > 0 && (trow >> 6) == h) {
        uint8_t* srow = sm + SsdSmem::kS + (trow & 63) * 128;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 o;
          o.x = pack_bf16x2(Srun[8 * g], Srun[8 * g + 1]); o.y = pack_bf16x2(Srun[8 * g + 2], Srun[8 * g + 3]);
          o.z = pack_bf16x2(Srun[8 * g + 4], Srun[8 * g + 5]); o.w = pack_bf16x2(Srun[8 * g + 6], Srun[8 * g + 7]);
          *reinterpret_cast<uint4*>(srow + (((4 * half + g) ^ (trow & 7)) << 4)) = o;
        }
      }
    };
    // GEMM2: Y = M X_h;  GEMM4: Y' = C S^T;  then every thread waits for both
    auto mma_head = [&](int h) {
      if (warp == 0 && elect_one()) {   // whole warp, then elect.sync: issue instructions back to back
        tc_fence_after();
        const uint32_t xa = sm_addr + (h ? SsdSmem::kX1 : SsdSmem::kX0);
        const uint64_t db = make_smem_desc_mn_sw128(xa, 16);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          const uint64_t da = make_smem_desc_sw128(sm_addr + SsdSmem::kM + (ks >> 2) * kSsdTile) + 2 * (ks & 3);
          umma_bf16_ss(tmem + 128, da, db + 128 * ks, idesc_g2, ks ? 1u : 0u);
        }
        if (it > 0) {
          const uint64_t dc = make_smem_desc_sw128(sm_addr + SsdSmem::kC), ds = make_smem_desc_sw128(sm_addr + SsdSmem::kS);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16_ss(tmem + 192, dc + 2 * k, ds + 2 * k, idesc_g4, k ? 1u : 0u);
        }
        umma_commit(mma_bar);
      }
      mbar_wait_or_trap(mma_bar, mma_phase);
      mma_phase ^= 1;
      tc_fence_after();
    };
    // y = Y + exp(cum_t) Y' + D x  -> global
    auto epilogue = [&](int h) {
      const float cum_t = cums[h * 128 + trow];
      const float sc = it > 0 ? ex2_approx(cum_t) : 0.f;
      const float Dh = Dp[2 * hp + h];
      const f32x2 sc2 = pack2(sc, sc), Dh2 = pack2(Dh, Dh);
      const uint8_t* xrow = sm + (h ? SsdSmem::kX1 : SsdSmem::kX0) + trow * 128;
      const int pos = p0 + trow;
      bf16* yp = yout + (row0 + pos) * E + (2 * hp + h) * kSsdP + 32 * half;
#pragma unroll
      for (int k = 0; k < 2; ++k) {          // two 16-column pieces (register pressure: the state rows stay live)
        uint32_t yi[16], yo[16];
        tmem_ld_32x32b_x16(t_lane + 128 + 32 * half + 16 * k, yi);
        if (it > 0) tmem_ld_32x32b_x16(t_lane + 192 + 32 * half + 16 * k, yo);
        tmem_ld_wait();
#pragma unroll
        for (int g = 0; g < 2; ++g) {   // packed pairs: y = Y + sc Y' + D x
          const uint4 xr = *reinterpret_cast<const uint4*>(xrow + (((4 * half + 2 * k + g) ^ (trow & 7)) << 4));
          const uint32_t xw[4] = {xr.x, xr.y, xr.z, xr.w};
          uint32_t ow[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            f32x2 v = pack2u(yi[8 * g + 2 * q], yi[8 * g + 2 * q + 1]);
            if (it > 0) v = fma2(sc2, pack2u(yo[8 * g + 2 * q], yo[8 * g + 2 * q + 1]), v);
            ow[q] = f32x2_to_bf16x2(fma2(Dh2, bf16x2_to_f32x2(xw[q]), v));
          }
          if (pos < L) *reinterpret_cast<uint4*>(yp + 16 * k + 8 * g) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
        }
      }
    };
    const bool more = it + 1 < nch;

    // X w for both heads (into the M tiles), w_s = exp(cum_end - cum_s) dt_s
    auto build_Xw = [&]() {
      // thread = (head, position): its row of the x tile scaled by w into the same (swizzled) place of the M tile.  The eight
      // 16-byte chunks are walked in the order chunk ^ (row & 7), so that eight consecutive rows touch eight different chunks:
      // conflict-free quarter-warps on the 128-byte-pitch tiles.
      const int hh = tid >> 7, r = tid & 127;
      const float w = ex2_approx(wsum[8 + hh] - cums[hh * 128 + r]) * dts[hh * 128 + r];
      const f32x2 w2 = pack2(w, w);
      const uint8_t* src = sm + (hh ? SsdSmem::kX1 : SsdSmem::kX0) + r * 128;
      uint8_t* dst = sm + SsdSmem::kM + hh * kSsdTile + r * 128;
#pragma unroll
      for (int cp = 0; cp < 8; ++cp) {
        const int pc = (cp ^ (r & 7)) << 4;
        const uint4 raw = *reinterpret_cast<const uint4*>(src + pc);
        uint4 o;
        o.x = f32x2_to_bf16x2(mul2(bf16x2_to_f32x2(raw.x), w2));
        o.y = f32x2_to_bf16x2(mul2(bf16x2_to_f32x2(raw.y), w2));
        o.z = f32x2_to_bf16x2(mul2(bf16x2_to_f32x2(raw.z), w2));
        o.w = f32x2_to_bf16x2(mul2(bf16x2_to_f32x2(raw.w), w2));
        *reinterpret_cast<uint4*>(dst + pc) = o;
      }
    };
    // one copy of every piece (runtime phase index): phase 0 [M_0 S_0] MMA_0, phase 1 [y_0 M_1 S_1] MMA_1, phase 2 [y_1 Xw]
#pragma unroll 1
    for (int ph = 0; ph < 3; ++ph) {
      if (ph > 0) epilogue(ph - 1);   // the previous head's MMAs have completed: its M tiles and the S tile are free as well
      if (ph < 2) {
        build_M(ph);
        write_S(ph);
      } else if (more) {
        build_Xw();
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncthreads();                // every thread has read the previous head's Y / Y' before the next MMAs overwrite them
      if (ph < 2) mma_head(ph);
    }
    if (more) {
      // ---- GEMM3: S_c[(h, p), n] = sum_s Xw[s, (h, p)] B[s, n]
      if (warp == 0 && elect_one()) {   // whole warp, then elect.sync: issue instructions back to back
        tc_fence_after();
        const uint64_t da = make_smem_desc_mn_sw128(sm_addr + SsdSmem::kM, kSsdTile);
        const uint64_t db = make_smem_desc_mn_sw128(sm_addr + SsdSmem::kB, 16);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) umma_bf16_ss(tmem, da + 128 * ks, db + 128 * ks, idesc_g3, ks ? 1u : 0u);
        umma_commit(mma_bar);
      }
      mbar_wait_or_trap(mma_bar, mma_phase);
      mma_phase ^= 1;
      tc_fence_after();
      {
        uint32_t sc[32];
        tmem_ld_32x32b_x32(t_lane + 32 * half, sc);
        tmem_ld_wait();
        const float decay = ex2_approx(wsum[8 + (trow >> 6)]);
#pragma unroll
        for (int n = 0; n < 32; ++n) Srun[n] = fmaf(decay, Srun[n], __uint_as_float(sc[n]));
      }
      tc_fence_before();
    }
    __syncthreads();   // every read of this chunk's tiles is done before the next chunk's TMA overwrites them
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<256>(tmem);
  }
}

inline cudaError_t launch_ssd_tc(const bf16* xbc_f, const bf16* xbc_r, long long ld_xbc, const bf16* dt_raw, long long ld_dt,
                                 const float* A_f, const float* D_f, const float* bias_f, const float* A_r, const float* D_r,
                                 const float* bias_r, bf16* y_f, bf16* y_r, int S, int L, int H, cudaStream_t stream) {
  const int E = H * kSsdP;
  const int smem = SsdSmem::kBytes + 1024;
  static unsigned long long attr_done = 0;
  cudaError_t e = ensure_dynamic_smem(ssd_chunk_tc_kernel, smem, attr_done);
  if (e != cudaSuccess) return e;
  CUtensorMap tf, tr;
  if (!make_tmap_3d(&tf, false, xbc_f, E + 2 * kSsdN, L, S, ld_xbc, 64, kSsdQ, true) ||
      !make_tmap_3d(&tr, false, xbc_r, E + 2 * kSsdN, L, S, ld_xbc, 64, kSsdQ, true))
    return cudaErrorInvalidValue;
  dim3 grid(H / 2, S, 2);
  ssd_chunk_tc_kernel<<<grid, kSsdThreads, smem, stream>>>(tf, tr, dt_raw, ld_dt, A_f, D_f, bias_f, A_r, D_r, bias_r, y_f, y_r, L, E);
  return cudaGetLastError();
}

template <typename T>
inline cudaError_t launch_ssd_seq(const T* xbc_f, const T* xbc_r, long long ld_xbc, const T* dt_raw, long long ld_dt,
                                  const float* A_f, const float* D_f, const float* bias_f, const float* A_r, const float* D_r,
                                  const float* bias_r, T* y_f, T* y_r, int S, int L, int H, cudaStream_t stream) {
  dim3 grid(H, S, 2);
  ssd_scan_seq_kernel<T><<<grid, 64, 0, stream>>>(xbc_f, xbc_r, ld_xbc, dt_raw, ld_dt, A_f, D_f, bias_f, A_r, D_r, bias_r, y_f, y_r,
                                                   L, H * kSsdP);
  return cudaGetLastError();
}

}  // namespace pcad
