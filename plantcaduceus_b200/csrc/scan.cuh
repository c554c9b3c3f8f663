// Bidirectional selective scan (Mamba-1, d_state = 16) with softplus(delta + bias), D skip and SiLU(z)
// gate; the forward-in-time and backward-in-time scans of BiMambaWrapper (strategy "add") run side by side in
// one CTA and meet in the middle, so their sum is formed without a flipped copy and y is written once.
//
//   [EXT] mamba_ssm selective_scan_fn(u, delta, A, B, C, D, z, delta_bias, delta_softplus=True)
//   [EXT] Caduceus BiMambaWrapper.forward: mamba_fwd(u) + flip_L(mamba_rev(flip_L(u)))
//
// Work decomposition: one CTA = one sequence x 64 channels; 128 threads: warps 0-1 run the forward scan, warps 2-3
// the reverse scan, one thread = one (direction, channel) holding its 16 fp32 states and 16 A coefficients in
// registers.  Measured on B200 (l32, B = 256, ms per launch): 128 channels x 3 CTAs/SM (80 registers, 24 warps/SM)
// 5.16; 128 x 2 CTAs (128 registers) 5.08; 64 channels x 5 CTAs (96 registers) 4.94; 64 x 4 CTAs (124 registers)
// 4.89, and 4.79 with 8-step blocks.  Smaller blocks mean more independently phased blocks per SM (the chunk phases of
// one block overlap the main loops of the others, and a barrier waits for 4 warps, not 8); 124 registers let the
// compiler keep a whole 8-step block in flight.  16 warps/SM are enough: the step is MUFU-bound, not latency-bound.
// Step i advances the forward scan at t_f = i and the reverse scan at t_r = L-1-i.  Inputs are streamed in chunks
// of 16 steps by TMA (3-D tensor maps, one elected lane, 2-stage mbarrier ring: see biscan_kernel); the 32 B/C
// values per step arrive as fp32 rows (kScanBcF32: converted once per layer by bc_to_f32_kernel) or are converted to fp32
// once per chunk (kScanPlain) and are broadcast-read.  Each thread leaves its un-gated y for
// the chunk in shared memory; a vectorised chunk epilogue then either parks the partial in y (the other direction
// has not reached that position yet) or adds the other direction's parked partial, applies SiLU(z) and stores the
// final value -- 16-byte global accesses only.
//
// The bf16 kernel is bound by the MUFU pipe (16 ex2 / clk / SM) and by instruction issue together, not by HBM (ncu:
// profiles/; tools/ub/scan_step.cu isolates the step).  What the kernel does about it:
// (a) (n, n+1) state pairs live in 64-bit registers and use the packed fp32x2 instructions of sm_100 (FFMA2 /
//     FMUL2: two lanes per issue slot);
// (b) everything is in the log2 domain: d' = log2(1 + 2^((delta + bias) log2 e)), exp(d A) = 2^(d' A), and the ln 2
//     that d = d' ln 2 owes to the input term is folded into B when B is converted;
// (c) softplus costs one MUFU op, not two: log2(1 + e), e = 2^-|x| in (0, 1], is a 7-coefficient FMA-pipe polynomial
//     (PCAD_SCAN_SPPOLY), and it runs one step ahead of the recurrence;
// (d) the main loop advances in blocks of 8 steps whose shared-memory stores are deferred to the end of the block, so
//     the scheduler overlaps one step's tail with the next step's loads (and the state-register copies of a 1-step
//     loop disappear);
// (e) every instruction outside the main loop counts (the kernel issues at ~0.65 IPC): loads are TMA issued behind
//     elect.sync (the six UTMALDG back to back), the forward's mode has no B|C conversion pass and ONE block barrier per
//     chunk, the epilogue and the prefetch of parked partials have branch-free block-uniform fast paths.
// Built, measured and removed (profiles/r01_scan_step_ub.txt): FMA-pipe polynomial exponentials for part of the 8 pairs
// (packed FFMA2 with three distinct operands runs at ~2.7 cycles, so a polynomial pair costs more issue/FMA time than the
// MUFU time it frees: 5.11 / 5.33 ms with 1 / 2 of 8 pairs against 5.08), whole-warp polynomial flavours, a
// software-pipelined step, an in-loop park/finalise, softplus in dt_proj's epilogue and SiLU(z) in in_proj's (both zero-sum
// under the power cap).
#pragma once

#include <stdlib.h>

#include "common.cuh"

namespace pcad {

#ifndef PCAD_SCAN_TC
#define PCAD_SCAN_TC 16
#endif
constexpr int kScanTC = PCAD_SCAN_TC;      // timesteps per chunk
#ifndef PCAD_SCAN_CH
#define PCAD_SCAN_CH 64
#endif
constexpr int kScanCH = PCAD_SCAN_CH;     // channels per CTA (128, or 64: smaller blocks, more of them per SM)
constexpr int kScanSeg8 = kScanCH / 8;    // 8-channel (16-byte bf16) segments per row
constexpr int kScanThreads = 2 * kScanCH;
constexpr int kScanN = 16;       // d_state
#ifndef PCAD_SCAN_SPPOLY
#define PCAD_SCAN_SPPOLY 7   // 0: softplus through MUFU.EX2 + MUFU.LG2; 6 / 7: log2(1 + e) from a polynomial with that many coefficients
#endif
#ifndef PCAD_SCAN_UNROLL
#define PCAD_SCAN_UNROLL 8
#endif
constexpr int kScanUnroll = PCAD_SCAN_UNROLL;   // steps per main-loop block (stores deferred to the end of the block)
#ifndef PCAD_SCAN_MINBLOCKS64
#define PCAD_SCAN_MINBLOCKS64 4   // 64-channel blocks (128 threads, 41 KB): 4 per SM leave 128 registers per thread (124 used)
#endif
#ifndef PCAD_SCAN_MINBLOCKS
#define PCAD_SCAN_MINBLOCKS 3
#endif

template <int V> struct IntTag { static constexpr int value = V; };

// Kernel modes (the values are part of the kernel names that profiles/ and tools/summarize_profiles.py quote).
//   kScanPlain: delta arrives ready-made (dt_proj ran as a GEMM), B|C arrive as activations and are converted to fp32 in the
//     kernel, once per chunk, behind a block barrier (the fp32 parity path and the operator API).
//   kScanBcF32 (bf16, what the forward runs): B|C arrive as fp32 rows (B already scaled by ln 2: bc_to_f32_kernel), delivered by
//     TMA like everything else -- no conversion pass, and with the chunk outputs double-buffered ONE block barrier per chunk.
constexpr int kScanPlain = 0, kScanBcF32 = 2;
template <typename T, int MODE> struct ScanStage;
template <typename T>
struct ScanStage<T, kScanPlain> {
  T u[2][kScanTC][kScanCH];          // [direction][step][channel]
  T d[2][kScanTC][kScanCH];
  T bc_raw[2][kScanTC][2 * kScanN];
};
template <typename T>
struct ScanStage<T, kScanBcF32> {
  T u[2][kScanTC][kScanCH];
  T d[2][kScanTC][kScanCH];
  float bc[2][kScanTC][2 * kScanN];   // fp32 [B ln 2 | C] rows as the TMA delivered them (reverse direction: box row 15 - j = step j)
};

template <typename T, int MODE> struct ScanShared;
template <typename T>
struct ScanShared<T, kScanPlain> {
  ScanStage<T, kScanPlain> st[2];
  float bc[2][kScanTC][2 * kScanN];   // fp32 B|C of the chunk being computed
  T pz[2][2][kScanTC][kScanCH];       // [partial | z][direction][step][channel]: prefetched for the chunk epilogue
};
template <typename T>
struct ScanShared<T, kScanBcF32> {
  ScanStage<T, kScanBcF32> st[2];
  T pz[2][2][kScanTC][kScanCH];
};

// One direction's 16 states of one channel.  step() advances h <- exp(d*A) h + du*B and returns
// y0 + <C, h>;  bc points at this timestep's fp32 [B(16) | C(16)] row in shared memory (broadcast reads).
template <bool PRECISE> struct ScanDir;

template <> struct ScanDir<true> {
  float h[kScanN], a[kScanN];
  float bias;
  __device__ __forceinline__ void init(const float* A, float bias_) {
    bias = bias_;
#pragma unroll
    for (int n = 0; n < kScanN; ++n) { h[n] = 0.f; a[n] = A ? A[n] : 0.f; }
  }
  static __device__ __forceinline__ float b_scale() { return 1.0f; }
  __device__ __forceinline__ void load_state(const float* p) {
#pragma unroll
    for (int n = 0; n < kScanN; ++n) h[n] = p[n];
  }
  __device__ __forceinline__ void store_state(float* p) const {
#pragma unroll
    for (int n = 0; n < kScanN; ++n) p[n] = h[n];
  }
  // decay of a state over a run of steps whose delta values (in this class's units) sum to sd
  __device__ __forceinline__ float run_decay(float sd, int n) const { return expf(sd * a[n]); }
  // returns d (natural units)
  __device__ __forceinline__ float delta(float raw) const { return softplus<true>(raw + bias); }
  __device__ __forceinline__ float step(float d, float du, float y0, const float* bc) {
    float y = y0;
#pragma unroll
    for (int n = 0; n < kScanN; ++n) {
      h[n] = fmaf(expf(d * a[n]), h[n], du * bc[n]);
      y = fmaf(h[n], bc[kScanN + n], y);
    }
    return y;
  }
};

template <> struct ScanDir<false> {
  f32x2 h[kScanN / 2], a[kScanN / 2];   // a = A (log2 domain: multiplied by d' = d / ln 2)
  float bias_l2;   // bias * log2(e)
  __device__ __forceinline__ void init(const float* A, float bias_) {
    bias_l2 = bias_ * kLog2e;
#pragma unroll
    for (int p = 0; p < kScanN / 2; ++p) {
      h[p] = pack2(0.f, 0.f);
      a[p] = A ? pack2(A[2 * p], A[2 * p + 1]) : pack2(0.f, 0.f);
    }
  }
  static __device__ __forceinline__ float b_scale() { return kLn2; }   // B is pre-multiplied by ln 2
  __device__ __forceinline__ void load_state(const float* p) {
#pragma unroll
    for (int q = 0; q < kScanN / 2; ++q) h[q] = pack2(p[2 * q], p[2 * q + 1]);
  }
  __device__ __forceinline__ void store_state(float* p) const {
#pragma unroll
    for (int q = 0; q < kScanN / 2; ++q) unpack2(h[q], p[2 * q], p[2 * q + 1]);
  }
  __device__ __forceinline__ float run_decay(float sd, int n) const {
    float a0, a1;
    unpack2(a[n >> 1], a0, a1);
    return ex2_approx(sd * ((n & 1) ? a1 : a0));
  }
  // returns d' = softplus(raw + bias) / ln 2  (identity above 20, as the reference)
  __device__ __forceinline__ float delta(float raw) const {
    const float xl = fmaf(raw, kLog2e, bias_l2);
#if PCAD_SCAN_SPPOLY
    // log2(1 + 2^x) = max(x, 0) + log2(1 + e), e = 2^-|x| in (0, 1]: one MUFU.EX2, and log2(1 + e) = e q(e) from a
    // minimax polynomial on the FMA pipe (relative error 1.5e-6 / 8.6e-6 for 7 / 6 coefficients) instead of
    // MUFU.LG2 -- the scan is bound by the MUFU pipe and the FMA pipe has room.  Above the reference's threshold
    // (x > 20) the correction is < 2^-28 x, i.e. the identity branch is reproduced to fp32 rounding.
    const float e = ex2_approx(-fabsf(xl));
#if PCAD_SCAN_SPPOLY >= 7
    float q = fmaf(2.035518363e-02f, e, -9.567064047e-02f);
    q = fmaf(q, e, 2.151583284e-01f);
    q = fmaf(q, e, -3.390359282e-01f);
    q = fmaf(q, e, 4.776608944e-01f);
    q = fmaf(q, e, -7.211598754e-01f);
    q = fmaf(q, e, 1.442693233e+00f);
#else
    float q = fmaf(-3.443166614e-02f, e, 1.460243315e-01f);
    q = fmaf(q, e, -3.030317128e-01f);
    q = fmaf(q, e, 4.691744745e-01f);
    q = fmaf(q, e, -7.204267383e-01f);
    q = fmaf(q, e, 1.442682981e+00f);
#endif
    return fmaf(q, e, fmaxf(xl, 0.0f));
#else
    const float sp = lg2_approx(1.0f + ex2_approx(xl));
    return xl > 20.0f * kLog2e ? xl : sp;
#endif
  }
  __device__ __forceinline__ float step(float d, float du, float y0, const float* bc) {
    const f32x2 dd = pack2(d, d), duu = pack2(du, du);
    const ulonglong2* bc2 = reinterpret_cast<const ulonglong2*>(bc);   // 16 bytes = two (n, n+1) pairs
    f32x2 acc[2] = {pack2(y0, 0.f), pack2(0.f, 0.f)};   // two chains: the FFMA2 -> FFMA2 latency is exposed otherwise
#pragma unroll
    for (int g = 0; g < kScanN / 4; ++g) {
      const ulonglong2 Bq = bc2[g], Cq = bc2[kScanN / 4 + g];
      const f32x2 Bp[2] = {Bq.x, Bq.y}, Cp[2] = {Cq.x, Cq.y};
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int p = 2 * g + k;
        float x0, x1;
        unpack2(mul2(dd, a[p]), x0, x1);
        const f32x2 dA = pack2(ex2_approx(x0), ex2_approx(x1));
        h[p] = fma2(dA, h[p], mul2(duu, Bp[k]));
        acc[k] = fma2(h[p], Cp[k], acc[k]);
      }
    }
    float s0, s1;
    unpack2(add2(acc[0], acc[1]), s0, s1);
    return s0 + s1;
  }
};

// Staging.  u, delta and B|C of both directions arrive by TMA: six 3-D tensor maps [sequence][row][channel] with a
// [1][16][64] (B|C: [1][16][32]) box, issued by one thread per chunk into a 2-stage ring and completed on an
// mbarrier, so the other threads spend no instructions on loads and rows outside [0, L) (ragged last chunk,
// either direction) are zero-filled by the hardware.  The reverse direction's box holds ascending rows
// L-16(c+1) .. L-16c-1, i.e. step j of the chunk sits in box row 15-j.  The parked partials and z rows that the
// chunk epilogue needs are fetched with cp.async (generic proxy: they were written by this CTA's own st.global).
template <typename T, bool PRECISE, int MODE>
__global__ void __launch_bounds__(kScanThreads, PRECISE ? 1 : (kScanCH == 64 ? PCAD_SCAN_MINBLOCKS64 : PCAD_SCAN_MINBLOCKS))
biscan_kernel(const __grid_constant__ CUtensorMap tm_uf, const __grid_constant__ CUtensorMap tm_df,
              const __grid_constant__ CUtensorMap tm_bcf, const __grid_constant__ CUtensorMap tm_ur,
              const __grid_constant__ CUtensorMap tm_dr, const __grid_constant__ CUtensorMap tm_bcr,
              const T* __restrict__ z, long long ldz, const float* __restrict__ A_f, const float* __restrict__ D_f,
              const float* __restrict__ bias_f, const float* __restrict__ A_r, const float* __restrict__ D_r,
              const float* __restrict__ bias_r, T* y, int L, int E, const float* __restrict__ h0, int Lrun) {
  constexpr bool BCF32 = MODE == kScanBcF32;
  static_assert(MODE == kScanPlain || (sizeof(T) == 2 && !PRECISE && kScanCH == 64 && kScanTC == 16),
                "the fp32 B|C rows are a bf16-path feature of the 64-channel, 16-step kernel");
  // TMA destinations need 128-byte alignment; the declared 1024 also rounds the static shared memory up to whole KB (the
  // 41 KB per 64-channel block counted above)
  extern __shared__ __align__(1024) uint8_t scan_smem_raw[];
  typedef ScanShared<T, MODE> Shared;
  typedef ScanStage<T, MODE> Stage;
  Shared& sm = *reinterpret_cast<Shared*>(scan_smem_raw);
  // Un-gated outputs of the chunk, per direction.  A separate (static) symbol on purpose: the compiler can then
  // prove that the main loop's stores to it do not alias the loads of later steps and overlaps consecutive steps.
  // kScanBcF32: two buffers (chunk parity), so that a chunk's main loop never writes what the previous chunk's epilogue reads.
  __shared__ __align__(16) float ys_all[BCF32 ? 2 : 1][2][kScanTC][kScanCH];
  __shared__ __align__(8) uint64_t full_bar[2];

  const int tid = threadIdx.x;
  const int dir = tid / kScanCH;          // warp-uniform: the first half of the warps runs forward, the second half reverse
  const int ch = tid & (kScanCH - 1);
  const int e0 = blockIdx.x * kScanCH;
  const int e = e0 + ch;
  const bool active = e < E;
  const int seq = blockIdx.y;
  const long long row0 = static_cast<long long>(seq) * L;
  // Lrun <= L: number of steps each direction takes.  Lrun < L is the score-only LAST layer, where y is wanted at one position p
  // only: after max(p, L-1-p) + 1 steps both directions have been there (rows further on hold parked partials nobody reads).
  const int nch = (Lrun + kScanTC - 1) / kScanTC;
  constexpr int VEC = 16 / sizeof(T);              // elements per 16-byte vector
  constexpr int SEGS = kScanCH / VEC;              // 16-byte segments per 128-channel row

  if (tid == 0) {
    mbar_init(&full_bar[0], 1);
    mbar_init(&full_bar[1], 1);
    fence_mbar_init();
    tma_prefetch_desc(&tm_uf); tma_prefetch_desc(&tm_df); tma_prefetch_desc(&tm_bcf);
    tma_prefetch_desc(&tm_ur); tma_prefetch_desc(&tm_dr); tma_prefetch_desc(&tm_bcr);
  }
  __syncthreads();

  // chunk c: forward rows 16c .. 16c+15, reverse rows L-16(c+1) .. L-16c-1 (box row 15-j = step j).  One thread.
  auto issue = [&](int c, int stage) {
    Stage& s = sm.st[stage];
    uint64_t* bar = &full_bar[stage];
    mbar_arrive_expect_tx(bar, sizeof(Stage));
    const int rf = c * kScanTC, rr = L - (c + 1) * kScanTC;
    tma_load_3d(&s.u[0][0][0], &tm_uf, bar, e0, rf, seq);
    tma_load_3d(&s.u[1][0][0], &tm_ur, bar, e0, rr, seq);
    if constexpr (BCF32) {
      tma_load_3d(&s.bc[0][0][0], &tm_bcf, bar, 0, rf, seq);
      tma_load_3d(&s.bc[1][0][0], &tm_bcr, bar, 0, rr, seq);
    } else {
      tma_load_3d(&s.bc_raw[0][0][0], &tm_bcf, bar, 0, rf, seq);
      tma_load_3d(&s.bc_raw[1][0][0], &tm_bcr, bar, 0, rr, seq);
    }
    tma_load_3d(&s.d[0][0][0], &tm_df, bar, e0, rf, seq);
    tma_load_3d(&s.d[1][0][0], &tm_dr, bar, e0, rr, seq);
  };

  ScanDir<PRECISE> S;
  {
    const float* A = dir ? A_r : A_f;
    const float* bias = dir ? bias_r : bias_f;
    S.init(active ? A + e * kScanN : nullptr, active ? bias[e] : 0.f);
    // time-parallel mode: this "sequence" is one segment of a longer one and starts from the carried state
    if (h0 != nullptr && active) S.load_state(h0 + ((static_cast<long long>(blockIdx.y) * 2 + dir) * E + e) * kScanN);
  }
  const float Dskip = active ? (dir ? D_r : D_f)[e] : 0.f;
  const float bscale = ScanDir<PRECISE>::b_scale();

  if (tid < 32 && elect_one()) issue(0, 0);
  bool prev_late = false;
  for (int c = 0; c < nch; ++c) {
    const int stage = c & 1;
    // TMA issue by warp 0.  Whole warp into the branch, then elect.sync: the compiler then knows a single lane issues and
    // emits the TMA instructions back to back instead of one election loop per instruction.
    // every thread is past the barrier that followed chunk c-1's main loop: stage^1 is free to be overwritten
    if (tid < 32 && c + 1 < nch) {
      if (elect_one()) issue(c + 1, stage ^ 1);
    }
    const Stage& s = sm.st[stage];
    const int i0 = c * kScanTC;
    const int nsteps = min(kScanTC, Lrun - i0);
    const bool has_final = (L - 1 - (i0 + nsteps - 1)) < i0 + nsteps;
    // (kScanBcF32: the stage's byte count includes the fp32 B|C rows of a second buffer, through tensor maps of their own:
    // a mismatch there must trap, not hang the GPU)
    if constexpr (BCF32) mbar_wait_or_trap(&full_bar[stage], (c >> 1) & 1);
    else mbar_wait(&full_bar[stage], (c >> 1) & 1);
    float (*ys)[kScanTC][kScanCH] = ys_all[BCF32 ? (c & 1) : 0];
    const bool late_chunk = (L - 1 - i0) < i0;   // every position of the chunk was parked in an earlier chunk
    if constexpr (!BCF32) {
      // B|C to fp32, once per chunk, 4 values per thread (B carries the ln 2 of the log2-domain delta on the fast
      // path); the reverse direction's rows are un-flipped here so that the main loop indexes both alike
#pragma unroll
      for (int gi = tid; gi < 2 * kScanTC * 2 * kScanN / 4; gi += kScanThreads) {   // 256 groups of 4 values
        const int dd = gi >> 7, r = gi & 127;
        const int j = r >> 3, k0 = (r & 7) * 4;
        const T* src = &s.bc_raw[dd][dd ? kScanTC - 1 - j : j][k0];
        float4 v;
        if constexpr (sizeof(T) == 2) {
          const uint2 raw = *reinterpret_cast<const uint2*>(src);
          v.x = __uint_as_float(raw.x << 16); v.y = __uint_as_float(raw.x & 0xffff0000u);
          v.z = __uint_as_float(raw.y << 16); v.w = __uint_as_float(raw.y & 0xffff0000u);
        } else {
          v = *reinterpret_cast<const float4*>(src);
        }
        if (k0 < kScanN) { v.x *= bscale; v.y *= bscale; v.z *= bscale; v.w *= bscale; }
        *reinterpret_cast<float4*>(&sm.bc[dd][j][k0]) = v;
      }
      __syncthreads();   // sm.bc is complete; chunk c-1's epilogue (its parked partials, its reads of ys / pz) is done
    } else {
      // No conversion pass, and normally no barrier here: the stage holds fp32 rows, ys is double-buffered, and in the
      // block-uniform ("late") path every thread prefetches into the very pz items it reads back in the epilogue.  The one
      // thing the old barrier still has to do happens in the middle of the sequence: a chunk that finalises positions must
      // not fetch partials that the PREVIOUS chunk's epilogue (other threads, possibly still running) parked.  Once the
      // previous chunk is itself "late", everything this chunk needs was parked at least two chunks -- two block barriers --
      // ago (chunk c-1 late means L-1 < 32 (c-1), and the youngest partial chunk c reads comes from chunk (L-1-16c)/16 <= c-2);
      // so only the first finalising chunk(s) pay: the middle chunk and the first late one.  The same barrier orders the
      // middle chunk's cross-thread use of pz against its neighbours.
      if (has_final && !prev_late) __syncthreads();
      prev_late = late_chunk;
    }
    // Positions of this chunk that the other direction visited in an EARLIER chunk will be finalised in the
    // epilogue: fetch their parked partials and z rows now (every earlier epilogue is complete and visible after the
    // barrier above), so that the epilogue does not wait on global memory.
    if (sizeof(T) == 2 && late_chunk) {
      // block-uniform fast path (bf16): one (step, segment) item per thread and direction, no per-item classification
      const int j = tid / kScanSeg8, seg = tid % kScanSeg8;
      const int chn = e0 + seg * 8;
      if (j < nsteps && chn < E) {
        const long long rf = row0 + i0 + j, rr = row0 + (L - 1 - i0 - j);
        cp_async16(&sm.pz[0][0][j][seg * 8], y + rf * E + chn, 16);
        cp_async16(&sm.pz[1][0][j][seg * 8], z + rf * ldz + chn, 16);
        cp_async16(&sm.pz[0][1][j][seg * 8], y + rr * E + chn, 16);
        cp_async16(&sm.pz[1][1][j][seg * 8], z + rr * ldz + chn, 16);
      }
    } else if (has_final) {
      for (int idx = tid; idx < 2 * kScanTC * SEGS; idx += kScanThreads) {
        const int dd = idx / (kScanTC * SEGS);
        const int rem = idx - dd * (kScanTC * SEGS);
        const int j = rem / SEGS, seg = rem % SEGS;
        const int i = i0 + j, io = L - 1 - i;
        const int chn = e0 + seg * VEC;
        const bool ok = (j < nsteps) && (chn < E) && (io < i0 + nsteps);
        const long long r = row0 + (ok ? (dd ? io : i) : 0);
        const int chs = ok ? chn : 0;
        if (ok && io < i0) cp_async16(&sm.pz[0][dd][j][seg * VEC], y + r * E + chs, 16);
        if (ok) cp_async16(&sm.pz[1][dd][j][seg * VEC], z + r * ldz + chs, 16);
      }
    }
    cp_async_commit();

    if (active) {
      const float* bcp;
      if constexpr (BCF32) bcp = &s.bc[dir][0][0];
      else bcp = &sm.bc[dir][0][0];
      float* ysp = &ys[dir][0][ch];
      auto run_chunk = [&](auto rev_tag) {
        constexpr bool REV = decltype(rev_tag)::value != 0;   // compile-time row order: immediate offsets in the unrolled loop
        const T* up = &s.u[REV ? 1 : 0][0][ch];
        auto row = [](int j) { return (REV ? kScanTC - 1 - j : j) * kScanCH; };
        // softplus runs one step ahead of the recurrence, so its load -> EX2 -> polynomial latency chain is off the
        // critical path of the step that consumes it
        float uu = ActT<T>::to_f(up[row(0)]);
        float dl;
        // one step: consumes (uu, dl) prepared by the previous call, prepares the next from row jn and the raw delta draw_n
        auto advance = [&](int j, int jn, float draw_n) -> float {
          const float uu_n = ActT<T>::to_f(up[row(jn)]);
          const float dl_n = S.delta(draw_n);
          // (fp32 rows straight from the TMA box are in box order: the reverse direction's step j is row 15 - j)
          const float yv = S.step(dl, dl * uu, Dskip * uu, bcp + (BCF32 && REV ? kScanTC - 1 - j : j) * 2 * kScanN);
          uu = uu_n;
          dl = dl_n;
          return yv;
        };
        const T* dp = &s.d[REV ? 1 : 0][0][ch];
        dl = S.delta(ActT<T>::to_f(dp[row(0)]));
        // blocks of kScanUnroll steps with the stores deferred to the end of the block: no shared-memory store sits
        // between the loads of consecutive steps, so the scheduler overlaps one step's tail with the next step's head
        int j = 0;
#pragma unroll 1
        for (; j + kScanUnroll <= nsteps; j += kScanUnroll) {
          float yv[kScanUnroll];
#pragma unroll
          for (int k = 0; k < kScanUnroll; ++k) {
            const int jn = min(j + k + 1, kScanTC - 1);
            yv[k] = advance(j + k, jn, ActT<T>::to_f(dp[row(jn)]));
          }
#pragma unroll
          for (int k = 0; k < kScanUnroll; ++k) ysp[(j + k) * kScanCH] = yv[k];
        }
#pragma unroll 1
        for (; j < nsteps; ++j) {
          const int jn = min(j + 1, kScanTC - 1);
          ysp[j * kScanCH] = advance(j, jn, ActT<T>::to_f(dp[row(jn)]));
        }
      };
      if (dir) run_chunk(IntTag<1>());
      else run_chunk(IntTag<0>());
    }
    cp_async_wait<0>();
    __syncthreads();   // both directions' un-gated outputs of the chunk are in ys, partials / z in sm.pz

    // ---- chunk epilogue: 16-byte vectors; item = (direction, step, segment of VEC channels)
    bool fast_done = false;
    if constexpr (!PRECISE && sizeof(T) == 2) {
      // bf16 fast paths for the two block-uniform cases (every chunk of an even-length sequence): all items of
      // the chunk park ("early": the other direction comes in a later chunk) or all finalise from a partial parked
      // in an earlier chunk ("late").  No per-item branching, packed fp32x2 arithmetic for the add and the gate.
      const bool early = !has_final, late = late_chunk;
      if (early || late) {
        fast_done = true;
        static_assert(kScanTC * kScanSeg8 == kScanThreads, "one item per thread and direction");
        const int j = tid / kScanSeg8, seg = tid % kScanSeg8;
        const int chn = e0 + seg * 8;
        if (j < nsteps && chn < E) {
#pragma unroll
          for (int dd = 0; dd < 2; ++dd) {
            const int i = i0 + j;
            const int t = dd ? L - 1 - i : i;
            const float4 a = *reinterpret_cast<const float4*>(&ys[dd][j][seg * 8]);
            const float4 b = *reinterpret_cast<const float4*>(&ys[dd][j][seg * 8 + 4]);
            f32x2 v2[4] = {pack2(a.x, a.y), pack2(a.z, a.w), pack2(b.x, b.y), pack2(b.z, b.w)};
            if (late) {
              const uint4 pr = *reinterpret_cast<const uint4*>(&sm.pz[0][dd][j][seg * 8]);
              const uint4 zr = *reinterpret_cast<const uint4*>(&sm.pz[1][dd][j][seg * 8]);
              const uint32_t pw[4] = {pr.x, pr.y, pr.z, pr.w}, zw[4] = {zr.x, zr.y, zr.z, zr.w};
              const f32x2 nl2 = pack2(-kLog2e, -kLog2e), one2 = pack2(1.0f, 1.0f);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const f32x2 p2 = pack2(__uint_as_float(pw[q] << 16), __uint_as_float(pw[q] & 0xffff0000u));
                const f32x2 z2 = pack2(__uint_as_float(zw[q] << 16), __uint_as_float(zw[q] & 0xffff0000u));
                float x0, x1, d0, d1;
                unpack2(mul2(z2, nl2), x0, x1);
                unpack2(add2(pack2(ex2_approx(x0), ex2_approx(x1)), one2), d0, d1);
                const f32x2 g2 = mul2(z2, pack2(rcp_approx(d0), rcp_approx(d1)));   // SiLU(z)
                v2[q] = mul2(add2(v2[q], p2), g2);
              }
            }
            uint4 out;
            float lo, hi;
            unpack2(v2[0], lo, hi); out.x = pack_bf16x2(lo, hi);
            unpack2(v2[1], lo, hi); out.y = pack_bf16x2(lo, hi);
            unpack2(v2[2], lo, hi); out.z = pack_bf16x2(lo, hi);
            unpack2(v2[3], lo, hi); out.w = pack_bf16x2(lo, hi);
            *reinterpret_cast<uint4*>(y + (row0 + t) * E + chn) = out;
          }
        }
      }
    }
    if (fast_done) continue;
    for (int idx = tid; idx < 2 * kScanTC * SEGS; idx += kScanThreads) {
      const int dd = idx / (kScanTC * SEGS);
      const int rem = idx - dd * (kScanTC * SEGS);
      const int j = rem / SEGS, seg = rem % SEGS;
      const int chn = e0 + seg * VEC;
      if (j >= nsteps || chn >= E) continue;
      const int i = i0 + j;                 // this direction's step index
      const int io = L - 1 - i;             // step at which the OTHER direction visits the same position
      const int t = dd ? io : i;            // the position itself
      float v[VEC];
#pragma unroll
      for (int k = 0; k < VEC; ++k) v[k] = ys[dd][j][seg * VEC + k];
      T* yp = y + (row0 + t) * E + chn;
      if (io >= i0 + nsteps) {              // the other direction comes later: park the partial
        store16<T>(yp, v);
        continue;
      }
      if (io >= i0) {                       // both visits fall in this chunk: combine from shared memory, once
        if (io > i || (io == i && dd == 1)) continue;   // the later visitor (forward on a tie) writes
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[k] += ys[dd ^ 1][io - i0][seg * VEC + k];
      } else {                              // parked in an earlier chunk (by another thread of this CTA)
        float p[VEC];
        load16<T>(&sm.pz[0][dd][j][seg * VEC], p);
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[k] += p[k];
      }
      float zz[VEC];
      load16<T>(&sm.pz[1][dd][j][seg * VEC], zz);
#pragma unroll
      for (int k = 0; k < VEC; ++k) v[k] *= silu<PRECISE>(zz[k]);
      store16<T>(yp, v);
    }
    // no barrier here: the next iteration's first __syncthreads orders these reads of sm.ys and of the stage
    // against their next writers
  }
}

// B|C columns of the two x_proj outputs ([rows, ldbc] bf16, B at bc_off, C at bc_off + 16) -> float [2][rows][32] rows
// [B ln 2 | C]: what the kScanBcF32 kernel's TMA delivers (the ln 2 is owed by the log2-domain delta, see ScanDir<false>).
// One thread per 8 values.  128 bytes per token and direction written once and read once: < 2 % of the scan's traffic.
__global__ void bc_to_f32_kernel(const bf16* __restrict__ dbc_f, const bf16* __restrict__ dbc_r, long long ldbc, int bc_off,
                                 float* __restrict__ out, long long rows) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= rows * 8) return;
  const int q = static_cast<int>(idx & 3), dd = static_cast<int>((idx >> 2) & 1);
  const long long r = idx >> 3;
  const uint4 raw = *reinterpret_cast<const uint4*>((dd ? dbc_r : dbc_f) + r * ldbc + bc_off + 8 * q);
  const float sc = q < 2 ? kLn2 : 1.0f;
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
  float4 o0, o1;
  o0.x = __uint_as_float(w[0] << 16) * sc; o0.y = __uint_as_float(w[0] & 0xffff0000u) * sc;
  o0.z = __uint_as_float(w[1] << 16) * sc; o0.w = __uint_as_float(w[1] & 0xffff0000u) * sc;
  o1.x = __uint_as_float(w[2] << 16) * sc; o1.y = __uint_as_float(w[2] & 0xffff0000u) * sc;
  o1.z = __uint_as_float(w[3] << 16) * sc; o1.w = __uint_as_float(w[3] & 0xffff0000u) * sc;
  float4* op = reinterpret_cast<float4*>(out + (static_cast<long long>(dd) * rows + r) * 2 * kScanN + 8 * q);
  op[0] = o0;
  op[1] = o1;
}

// u_* and delta_* are [S*L, E]; bc_* hold B|C at column bc_off of [S*L, ldbc] rows (read by kScanPlain, while kScanBcF32
// reads bcf_*).  h0: the states each sequence starts from (time-parallel segments), or null for zeros.
template <typename T, bool PRECISE, int MODE = kScanPlain>
inline cudaError_t launch_biscan(const T* u_f, const T* delta_f, const T* bc_f, const T* u_r, const T* delta_r,
                                 const T* bc_r, long long ldbc, int bc_off, const T* z, long long ldz,
                                 const float* A_f, const float* D_f, const float* bias_f, const float* A_r,
                                 const float* D_r, const float* bias_r, T* y, int S, int L, int E,
                                 cudaStream_t stream, const float* h0 = nullptr, int Lrun = 0, const float* bcf_f = nullptr,
                                 const float* bcf_r = nullptr) {
  constexpr bool BCF32 = MODE == kScanBcF32;
  size_t smem = sizeof(ScanShared<T, MODE>);
  if (const char* ex = getenv("PCAD_SCAN_EXTRA_SMEM")) smem += static_cast<size_t>(atoi(ex));   // occupancy experiments
  static unsigned long long attr_done = 0;
  cudaError_t e1 = ensure_dynamic_smem(biscan_kernel<T, PRECISE, MODE>, static_cast<int>(smem), attr_done);
  if (e1 != cudaSuccess) return e1;
  constexpr bool f32 = sizeof(T) == 4;
  CUtensorMap tm[6];
  bool ok = make_tmap_3d(&tm[0], f32, u_f, E, L, S, E, kScanCH, kScanTC) && make_tmap_3d(&tm[2], f32, u_r, E, L, S, E, kScanCH, kScanTC);
  ok = ok && make_tmap_3d(&tm[1], f32, delta_f, E, L, S, E, kScanCH, kScanTC) &&
       make_tmap_3d(&tm[3], f32, delta_r, E, L, S, E, kScanCH, kScanTC);
  if (BCF32) {   // bcf_*: float [S*L, 32] rows [B ln 2 | C] (bc_to_f32_kernel)
    if (!bcf_f || !bcf_r) return cudaErrorInvalidValue;
    ok = ok && make_tmap_3d(&tm[4], true, bcf_f, 2 * kScanN, L, S, 2 * kScanN, 2 * kScanN, kScanTC);
    ok = ok && make_tmap_3d(&tm[5], true, bcf_r, 2 * kScanN, L, S, 2 * kScanN, 2 * kScanN, kScanTC);
  } else {
    ok = ok && make_tmap_3d(&tm[4], f32, bc_f + bc_off, 2 * kScanN, L, S, ldbc, 2 * kScanN, kScanTC);
    ok = ok && make_tmap_3d(&tm[5], f32, bc_r + bc_off, 2 * kScanN, L, S, ldbc, 2 * kScanN, kScanTC);
  }
  if (!ok) return cudaErrorInvalidValue;
  dim3 grid((E + kScanCH - 1) / kScanCH, S);
  biscan_kernel<T, PRECISE, MODE><<<grid, kScanThreads, smem, stream>>>(
      tm[0], tm[1], tm[4], tm[2], tm[3], tm[5], z, ldz, A_f, D_f, bias_f, A_r, D_r, bias_r, y, L, E, h0,
      (Lrun > 0 && Lrun < L) ? Lrun : L);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
// Time-parallel scan for low batch / long context (BASELINE.json north_star: chunk-local scan -> carry combine -> fix-up).
// biscan_kernel is sequential in time with one CTA per (sequence, 64 channels): at B = 1 that is E / 64 x 2 CTAs for 592
// resident slots.  Here a sequence of length L is cut into P segments that are scanned concurrently:
//   1. scan_segment_state_kernel: every segment from a ZERO state, keeping only its end state h_end0 and the sum of its
//      deltas (the segment's total decay per state is exp(A sum(delta)): the recurrence is linear in h);
//   2. scan_segment_carry_kernel: the P end states of a (sequence, direction, channel) combined in scan order,
//      h_in(k+1) = decay_k h_in(k) + h_end0(k) -- a serial chain of P steps on 16 values;
//   3. biscan_kernel on the segments as [S P] "sequences" of length L / P, each starting from its h_in.
// The exponentials are evaluated twice (passes 1 and 3), so this pays only while the grid of the sequential kernel leaves
// the machine empty; pcad.cu picks P so that E / 64 x S x P just fills the resident slots.
// ---------------------------------------------------------------------------------------------------------------------
template <typename T, bool PRECISE>
__global__ void __launch_bounds__(kScanThreads)
scan_segment_state_kernel(const T* __restrict__ u_f, const T* __restrict__ delta_f, const T* __restrict__ bc_f,
                          const T* __restrict__ u_r, const T* __restrict__ delta_r, const T* __restrict__ bc_r, long long ldbc,
                          int bc_off, const float* __restrict__ A_f, const float* __restrict__ bias_f,
                          const float* __restrict__ A_r, const float* __restrict__ bias_r, float* __restrict__ hend,
                          float* __restrict__ sumd, int Lseg, int E) {
  __shared__ __align__(16) float sbc[2][kScanTC][2 * kScanN];
  const int tid = threadIdx.x;
  const int dir = tid / kScanCH, ch = tid & (kScanCH - 1);
  const int e = blockIdx.x * kScanCH + ch;
  const bool active = e < E;
  const long long row0 = static_cast<long long>(blockIdx.y) * Lseg;     // blockIdx.y = sequence * P + segment
  const T* u = dir ? u_r : u_f;
  const T* dl = dir ? delta_r : delta_f;
  ScanDir<PRECISE> S;
  S.init(active ? (dir ? A_r : A_f) + e * kScanN : nullptr, active ? (dir ? bias_r : bias_f)[e] : 0.f);
  const float bscale = ScanDir<PRECISE>::b_scale();
  float sd = 0.f;
  for (int i0 = 0; i0 < Lseg; i0 += kScanTC) {
    const int nst = min(kScanTC, Lseg - i0);
    __syncthreads();
    for (int idx = tid; idx < 2 * kScanTC * 2 * kScanN; idx += kScanThreads) {
      const int dd = idx / (kScanTC * 2 * kScanN), rem = idx % (kScanTC * 2 * kScanN);
      const int j = rem / (2 * kScanN), k = rem % (2 * kScanN);
      float v = 0.f;
      if (j < nst) {
        const long long r = row0 + (dd ? Lseg - 1 - (i0 + j) : i0 + j);
        v = ActT<T>::to_f((dd ? bc_r : bc_f)[r * ldbc + bc_off + k]);
      }
      sbc[dd][j][k] = k < kScanN ? v * bscale : v;
    }
    float uu[kScanTC], dr[kScanTC];
#pragma unroll
    for (int j = 0; j < kScanTC; ++j) {
      const long long r = row0 + (dir ? Lseg - 1 - (i0 + j) : i0 + j);
      const bool ok = active && j < nst;
      uu[j] = ok ? ActT<T>::to_f(u[r * E + e]) : 0.f;
      dr[j] = ok ? ActT<T>::to_f(dl[r * E + e]) : 0.f;
    }
    __syncthreads();
    if (active) {
#pragma unroll
      for (int j = 0; j < kScanTC; ++j) {
        if (j < nst) {
          const float d = S.delta(dr[j]);
          sd += d;
          S.step(d, d * uu[j], 0.f, &sbc[dir][j][0]);
        }
      }
    }
  }
  if (active) {
    const long long o = (static_cast<long long>(blockIdx.y) * 2 + dir) * E + e;
    S.store_state(hend + o * kScanN);
    sumd[o] = sd;
  }
}

// hend [S*P][2][E][16] -> in place: the state each segment STARTS from.  One thread per (sequence, direction, channel).
template <bool PRECISE>
__global__ void scan_segment_carry_kernel(const float* __restrict__ A_f, const float* __restrict__ A_r, float* __restrict__ hend,
                                          const float* __restrict__ sumd, int S, int P, int E) {
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= static_cast<long long>(S) * 2 * E) return;
  const int e = static_cast<int>(gid % E);
  const int dir = static_cast<int>((gid / E) % 2);
  const int seq = static_cast<int>(gid / (2LL * E));
  ScanDir<PRECISE> D;
  D.init((dir ? A_r : A_f) + e * kScanN, 0.f);
  float carry[kScanN];
#pragma unroll
  for (int n = 0; n < kScanN; ++n) carry[n] = 0.f;
  for (int k = 0; k < P; ++k) {
    const int seg = dir ? P - 1 - k : k;                       // scan order of the segments
    const long long o = ((static_cast<long long>(seq) * P + seg) * 2 + dir) * E + e;
    float* hp = hend + o * kScanN;
    const float sd = sumd[o];
#pragma unroll
    for (int n = 0; n < kScanN; ++n) {
      const float end0 = hp[n];
      hp[n] = carry[n];
      carry[n] = fmaf(D.run_decay(sd, n), carry[n], end0);
    }
  }
}

// launch_biscan over P concurrent segments per sequence (L % P == 0).  state: float [S*P*2*E*16], sumd: float [S*P*2*E].
template <typename T, bool PRECISE>
inline cudaError_t launch_biscan_time_parallel(const T* u_f, const T* delta_f, const T* bc_f, const T* u_r, const T* delta_r,
                                               const T* bc_r, long long ldbc, int bc_off, const T* z, long long ldz,
                                               const float* A_f, const float* D_f, const float* bias_f, const float* A_r,
                                               const float* D_r, const float* bias_r, T* y, int S, int L, int E, int P,
                                               float* state, float* sumd, cudaStream_t stream, const float* bcf_f = nullptr,
                                               const float* bcf_r = nullptr) {
  if (P < 2 || L % P) return cudaErrorInvalidValue;
  const int Lseg = L / P;
  dim3 grid((E + kScanCH - 1) / kScanCH, S * P);
  scan_segment_state_kernel<T, PRECISE><<<grid, kScanThreads, 0, stream>>>(u_f, delta_f, bc_f, u_r, delta_r, bc_r, ldbc, bc_off, A_f,
                                                                           bias_f, A_r, bias_r, state, sumd, Lseg, E);
  const long long n = static_cast<long long>(S) * 2 * E;
  scan_segment_carry_kernel<PRECISE><<<static_cast<unsigned>((n + 127) / 128), 128, 0, stream>>>(A_f, A_r, state, sumd, S, P, E);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if constexpr (sizeof(T) == 2 && !PRECISE) {
    if (bcf_f && bcf_r)
      return launch_biscan<T, PRECISE, kScanBcF32>(u_f, delta_f, bc_f, u_r, delta_r, bc_r, ldbc, bc_off, z, ldz, A_f, D_f, bias_f, A_r,
                                                   D_r, bias_r, y, S * P, Lseg, E, stream, state, 0, bcf_f, bcf_r);
  }
  return launch_biscan<T, PRECISE, kScanPlain>(u_f, delta_f, bc_f, u_r, delta_r, bc_r, ldbc, bc_off, z, ldz, A_f, D_f, bias_f, A_r, D_r,
                                               bias_r, y, S * P, Lseg, E, stream, state);
}

}  // namespace pcad
