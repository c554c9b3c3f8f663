// HBM-bound kernels of the Caduceus forward: tokenise, RC-aware embedding, fused residual-add RMSNorm,
// depthwise causal conv + SiLU (both scan directions from one read), RC LM head, hidden-state tap.
//
// Internal layout ("strand-major"): the B input windows become S = 2B independent sequences,
//   s <  B : forward strand of window s,                 ids_s[t] = ids[s][t]
//   s >= B : reverse-complement strand of window s - B,  ids_s[t] = comp[ids[s-B][L-1-t]]
// stored token-major as [S*L, channels].  In this orientation the RC half of the reference's
// [B, L, 2d] tensors (which it keeps flipped in sequence AND channel, SURVEY.md Appendix A 1-3) is an
// ordinary sequence, so every layer treats both strands identically with the same weights and no flip
// is ever materialised; the flips reappear only as index arithmetic in embed / lm_head / hidden tap.
#pragma once

#include "common.cuh"

namespace pcad {

// ---- 8-element vector helpers (one "vec" = 8 consecutive channels, any dtype) -----------------
template <typename T>
__device__ __forceinline__ void load8(const T* p, float (&v)[8]) {
  if constexpr (sizeof(T) == 2) {
    load16<T>(p, v);
  } else {
    float a[4], b[4];
    load16<T>(p, a);
    load16<T>(p + 4, b);
#pragma unroll
    for (int i = 0; i < 4; ++i) { v[i] = a[i]; v[4 + i] = b[i]; }
  }
}
template <typename T>
__device__ __forceinline__ void store8(T* p, const float (&v)[8]) {
  if constexpr (sizeof(T) == 2) {
    store16<T>(p, v);
  } else {
    float a[4] = {v[0], v[1], v[2], v[3]}, b[4] = {v[4], v[5], v[6], v[7]};
    store16<T>(p, a);
    store16<T>(p + 4, b);
  }
}

// ---- tokenise -----------------------------------------------------------------------------------
// ids[i] = lut[ascii[i]]; if mask_pos >= 0, position mask_pos of every window of length L gets mask_id.
// Replaces tokenizer.encode_plus + ids[0, tokenIdx] = mask_token_id (reference zero_shot_score.py:51-57).
__global__ void tokenize_kernel(const uint8_t* __restrict__ ascii, uint8_t* __restrict__ ids, long long n,
                                const uint8_t* __restrict__ lut, int L, int mask_pos, int mask_id) {
  __shared__ uint8_t s_lut[256];
  s_lut[threadIdx.x & 255] = lut[threadIdx.x & 255];
  __syncthreads();
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t id = s_lut[ascii[i]];
  if (mask_pos >= 0 && (i % L) == mask_pos) id = static_cast<uint8_t>(mask_id);
  ids[i] = id;
}

// ---- window extraction on the device (reference seq_from_vcf, src/zero_shot_score.py:185-198) --------------------
// out[b, k] = the L-base context of the variant at 0-based chromosome position pos0[b], variant at index token_idx:
// chrom[pos0 - token_idx : pos0 + L - token_idx] upper-cased; windows that would start before the chromosome are
// right-justified with 'N' (the slice chrom[0 : pos0 + L - token_idx] is kept whole), all others left-justified.
__global__ void extract_windows_kernel(const uint8_t* __restrict__ chrom, long long chrom_len,
                                       const long long* __restrict__ pos0, uint8_t* __restrict__ out, int B, int L,
                                       int token_idx) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * L) return;
  const int b = static_cast<int>(i / L), k = static_cast<int>(i % L);
  const long long p = pos0[b];
  const long long add = L - token_idx;
  long long src;
  if (p - token_idx < 0) {
    long long n_s = p + add;                       // length of chrom[0 : p + add]
    n_s = n_s < 0 ? 0 : (n_s > chrom_len ? chrom_len : n_s);
    const long long pad = L - n_s;
    src = (k < pad) ? -1 : (k - pad);
  } else {
    src = p - token_idx + k;
    if (src >= chrom_len) src = -1;
  }
  uint8_t c = 'N';
  if (src >= 0) {
    c = chrom[src];
    if (c >= 'a' && c <= 'z') c -= 32;             // str.upper() on ASCII
  }
  out[i] = c;
}

__global__ void ids64_to_u8_kernel(const long long* __restrict__ in, uint8_t* __restrict__ out, long long n, int V,
                                   int* __restrict__ bad) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long v = in[i];
  if (v < 0 || v >= V) { atomicExch(bad, 1); out[i] = 0; return; }
  out[i] = static_cast<uint8_t>(v);
}

// uint8 ids from the caller (pcad_score_masked): same validation, no widening
__global__ void ids_u8_check_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, long long n, int V,
                                    int* __restrict__ bad) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t v = in[i];
  if (v >= V) { atomicExch(bad, 1); out[i] = 0; return; }
  out[i] = v;
}

// ---- RC-aware embedding [EXT RCPSEmbedding.forward] --------------------------------------------
// out[s*L + t, :] = emb[id_s[t], :]  (see layout note above).  One thread per 8 channels.
template <typename T>
__global__ void embed_kernel(const uint8_t* __restrict__ ids, const T* __restrict__ emb, T* __restrict__ out, int B,
                             int L, int d, const uint8_t* __restrict__ comp) {
  const int vec_per_row = d / 8;
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = 2LL * B * L * vec_per_row;
  if (gid >= total) return;
  const int v = static_cast<int>(gid % vec_per_row);
  const long long row = gid / vec_per_row;
  const int t = static_cast<int>(row % L);
  const int s = static_cast<int>(row / L);
  int id;
  if (s < B) id = ids[static_cast<long long>(s) * L + t];
  else id = comp[ids[static_cast<long long>(s - B) * L + (L - 1 - t)]];
  float x[8];
  load8<T>(emb + static_cast<long long>(id) * d + v * 8, x);
  store8<T>(out + row * d + v * 8, x);
}

// ---- fused residual add + RMSNorm [EXT rms_norm_fn(prenorm=True, residual_in_fp32)] ------------
// One warp per row.  res_out = x + res_in (fp32 sum, stored as RT); y = sum * rstd * w (stored as T);
// statistics from the un-rounded fp32 sum, as the reference's Triton kernel does.
template <typename T, typename RT, int CH>
__global__ void __launch_bounds__(256)
add_rmsnorm_kernel(const T* __restrict__ x, const RT* __restrict__ res_in, const float* __restrict__ w,
                   T* __restrict__ y, RT* __restrict__ res_out, long long rows, int d, float eps) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int nvec = d >> 3;
  float v[CH][8];
  float ss = 0.f;
#pragma unroll
  for (int c = 0; c < CH; ++c) {
    const int vi = lane + 32 * c;
    if (vi < nvec) {
      load8<T>(x + row * d + vi * 8, v[c]);
      if (res_in != nullptr) {
        float r[8];
        load8<RT>(res_in + row * d + vi * 8, r);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[c][i] += r[i];
      }
      if (res_out != nullptr) store8<RT>(res_out + row * d + vi * 8, v[c]);
#pragma unroll
      for (int i = 0; i < 8; ++i) ss = fmaf(v[c][i], v[c][i], ss);
    }
  }
  ss = warp_sum(ss);
  const float rstd = rsqrtf(ss / static_cast<float>(d) + eps);
#pragma unroll
  for (int c = 0; c < CH; ++c) {
    const int vi = lane + 32 * c;
    if (vi < nvec) {
      float o[8];
      const float4 w0 = *reinterpret_cast<const float4*>(w + vi * 8);
      const float4 w1 = *reinterpret_cast<const float4*>(w + vi * 8 + 4);
      o[0] = v[c][0] * rstd * w0.x; o[1] = v[c][1] * rstd * w0.y; o[2] = v[c][2] * rstd * w0.z; o[3] = v[c][3] * rstd * w0.w;
      o[4] = v[c][4] * rstd * w1.x; o[5] = v[c][5] * rstd * w1.y; o[6] = v[c][6] * rstd * w1.z; o[7] = v[c][7] * rstd * w1.w;
      store8<T>(y + row * d + vi * 8, o);
    }
  }
}

// ---- depthwise causal conv k=4 + SiLU, both directions [EXT causal_conv1d_fn(activation="silu")] --
// x: [S*L, *] with row pitch ldx (the x half of xz).  4 channels per thread, TT timesteps per thread,
// sliding 7-row register window.  out_f[t] = SiLU(b_f + sum_k w_f[k] x[t-3+k]);
// out_r[t] = SiLU(b_r + sum_k w_r[k] x[t+3-k])  (the causal conv of the time-reversed sequence).
constexpr int kConvTT = 64;   // timesteps per thread (halo re-read: 6 / 64)
constexpr int kConvBlk = 8;   // rows fetched per batch of back-to-back loads
template <int V> struct ConvTag { static constexpr int value = V; };

// CPT channels per thread as loaded from memory
template <typename T, int CPT> struct RawC;
template <> struct RawC<bf16, 4> { typedef uint2 type; };
template <> struct RawC<bf16, 2> { typedef uint32_t type; };
template <> struct RawC<float, 4> { typedef float4 type; };
template <> struct RawC<float, 2> { typedef float2 type; };

__device__ __forceinline__ void cvtc(const uint2& raw, float (&v)[4]) {
  v[0] = __uint_as_float(raw.x << 16); v[1] = __uint_as_float(raw.x & 0xffff0000u);
  v[2] = __uint_as_float(raw.y << 16); v[3] = __uint_as_float(raw.y & 0xffff0000u);
}
__device__ __forceinline__ void cvtc(const uint32_t& raw, float (&v)[2]) {
  v[0] = __uint_as_float(raw << 16); v[1] = __uint_as_float(raw & 0xffff0000u);
}
__device__ __forceinline__ void cvtc(const float4& raw, float (&v)[4]) { v[0] = raw.x; v[1] = raw.y; v[2] = raw.z; v[3] = raw.w; }
__device__ __forceinline__ void cvtc(const float2& raw, float (&v)[2]) { v[0] = raw.x; v[1] = raw.y; }

template <typename T, int CPT>
__device__ __forceinline__ void storec(T* p, const float (&v)[CPT]) {
  typename RawC<T, CPT>::type raw;
  if constexpr (sizeof(T) == 2) {
    if constexpr (CPT == 4) { raw.x = pack_bf16x2(v[0], v[1]); raw.y = pack_bf16x2(v[2], v[3]); }
    else raw = pack_bf16x2(v[0], v[1]);
  } else {
    if constexpr (CPT == 4) raw = make_float4(v[0], v[1], v[2], v[3]);
    else raw = make_float2(v[0], v[1]);
  }
  *reinterpret_cast<typename RawC<T, CPT>::type*>(p) = raw;
}

// CPT = 2 for bf16 (about 70 registers, 7 CTAs per SM: the kernel sits on the MUFU pipe and needs the warps),
// CPT = 4 for the fp32 parity path.
template <typename T, bool PRECISE, int CPT>
__global__ void __launch_bounds__(128)
conv_silu_kernel(const T* __restrict__ x, long long ldx, const float* __restrict__ w_f, const float* __restrict__ b_f,
                 const float* __restrict__ w_r, const float* __restrict__ b_r, T* __restrict__ out_f,
                 T* __restrict__ out_r, int L, int E) {
  typedef typename RawC<T, CPT>::type raw_t;
  const int e0 = (blockIdx.x * blockDim.x + threadIdx.x) * CPT;
  if (e0 >= E) return;
  const int t0 = blockIdx.y * kConvTT;
  const long long seq_row0 = static_cast<long long>(blockIdx.z) * L;
  float wf[CPT][4], wr[CPT][4], bf[CPT], br[CPT];
#pragma unroll
  for (int c = 0; c < CPT; ++c) {
    const float4 a = *reinterpret_cast<const float4*>(w_f + (e0 + c) * 4);
    const float4 b = *reinterpret_cast<const float4*>(w_r + (e0 + c) * 4);
    wf[c][0] = a.x; wf[c][1] = a.y; wf[c][2] = a.z; wf[c][3] = a.w;
    wr[c][0] = b.x; wr[c][1] = b.y; wr[c][2] = b.z; wr[c][3] = b.w;
    bf[c] = b_f[e0 + c];
    br[c] = b_r[e0 + c];
  }
  // Addressing: one 64-bit base per tensor and thread (row t0 of this sequence, this thread's channels) and 32-bit
  // element offsets that advance by a constant per step, so a step costs one IMAD.WIDE per access instead of a
  // 64-bit row * pitch product; blocks whose rows t0-3 .. t0+kConvTT+2 all lie inside the sequence (INTERIOR) skip
  // every bounds check.
  const T* xb = x + (seq_row0 + t0) * ldx + e0;
  T* ofb = out_f + (seq_row0 + t0) * E + e0;
  T* orb = out_r + (seq_row0 + t0) * E + e0;
  const int ldxi = static_cast<int>(ldx);
  raw_t zero_raw;
  memset(&zero_raw, 0, sizeof(zero_raw));
  auto body = [&](auto interior_tag) {
    constexpr bool INTERIOR = decltype(interior_tag)::value != 0;
    auto fetch = [&](int dt) -> raw_t {   // row t0 + dt of this sequence, zero outside [0, L)
      if (INTERIOR || (t0 + dt >= 0 && t0 + dt < L)) return *reinterpret_cast<const raw_t*>(xb + dt * ldxi);
      return zero_raw;
    };
    // win[j] holds x[t - 3 + j], j = 0..6, for the step being computed
    float win[7][CPT];
    raw_t nxt[kConvBlk];
#pragma unroll
    for (int j = 0; j < 6; ++j) cvtc(fetch(j - 3), win[j]);
#pragma unroll
    for (int i = 0; i < kConvBlk; ++i) nxt[i] = fetch(3 + i);
    int ooff = 0;   // element offset of the output row being written
#pragma unroll 1
    for (int blk = 0; blk < kConvTT; blk += kConvBlk) {
      if (!INTERIOR && t0 + blk >= L) break;
      raw_t cur[kConvBlk];
#pragma unroll
      for (int i = 0; i < kConvBlk; ++i) cur[i] = nxt[i];
      if (blk + kConvBlk < kConvTT) {   // next batch of rows: in flight while this batch is computed
#pragma unroll
        for (int i = 0; i < kConvBlk; ++i) nxt[i] = fetch(blk + kConvBlk + 3 + i);
      }
#pragma unroll
      for (int i = 0; i < kConvBlk; ++i) {
        cvtc(cur[i], win[6]);
        if (INTERIOR || t0 + blk + i < L) {
          float of[CPT], orv[CPT];
          if constexpr (!PRECISE && CPT == 2) {
            // bf16 fast path: the two channels of a thread ride in one fp32x2 register pair (FFMA2 / FMUL2 / FADD2: half
            // the issue slots), so the kernel is left with its MUFU work (ex2 + rcp per output) and its HBM traffic
            f32x2 a2 = pack2(bf[0], bf[1]), r2 = pack2(br[0], br[1]);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              a2 = fma2(pack2(wf[0][k], wf[1][k]), pack2(win[k][0], win[k][1]), a2);
              r2 = fma2(pack2(wr[0][k], wr[1][k]), pack2(win[6 - k][0], win[6 - k][1]), r2);
            }
            const f32x2 nl2 = pack2(-kLog2e, -kLog2e), one2 = pack2(1.0f, 1.0f);
            float xa0, xa1, xr0, xr1;
            unpack2(mul2(a2, nl2), xa0, xa1);
            unpack2(mul2(r2, nl2), xr0, xr1);
            const f32x2 da = add2(pack2(ex2_approx(xa0), ex2_approx(xa1)), one2);
            const f32x2 dr = add2(pack2(ex2_approx(xr0), ex2_approx(xr1)), one2);
            float da0, da1, dr0, dr1;
            unpack2(da, da0, da1);
            unpack2(dr, dr0, dr1);
            unpack2(mul2(a2, pack2(rcp_approx(da0), rcp_approx(da1))), of[0], of[1]);
            unpack2(mul2(r2, pack2(rcp_approx(dr0), rcp_approx(dr1))), orv[0], orv[1]);
          } else {
#pragma unroll
            for (int c = 0; c < CPT; ++c) {
              float a = bf[c];
              a = fmaf(wf[c][0], win[0][c], a);
              a = fmaf(wf[c][1], win[1][c], a);
              a = fmaf(wf[c][2], win[2][c], a);
              a = fmaf(wf[c][3], win[3][c], a);
              of[c] = silu<PRECISE>(a);
              float r = br[c];
              r = fmaf(wr[c][0], win[6][c], r);
              r = fmaf(wr[c][1], win[5][c], r);
              r = fmaf(wr[c][2], win[4][c], r);
              r = fmaf(wr[c][3], win[3][c], r);
              orv[c] = silu<PRECISE>(r);
            }
          }
          storec<T, CPT>(ofb + ooff, of);
          storec<T, CPT>(orb + ooff, orv);
        }
        ooff += E;
#pragma unroll
        for (int j = 0; j < 6; ++j)
#pragma unroll
          for (int c = 0; c < CPT; ++c) win[j][c] = win[j + 1][c];
      }
    }
  };
  if (t0 >= 3 && t0 + kConvTT + 3 <= L) body(ConvTag<1>());
  else body(ConvTag<0>());
}

// ---- RC LM head [EXT RCPSLMHead.forward + .float()] ---------------------------------------------
// logits[b, t, v] = <HF[b, t, :], W[v, :]> + <HR[b, L-1-t, :], W[comp[v], :]>, V = 8, fp32 out.
// One warp per requested position.  If pos != nullptr only positions pos[b*n_pos + i] are computed and
// only the 4 columns sel[0..3] (a,c,g,t) are written: out[(b*n_pos + i)*4 + k].
template <typename T>
__global__ void __launch_bounds__(256)
lm_head_kernel(const T* __restrict__ H, const float* __restrict__ W, const uint8_t* __restrict__ comp,
               const int* __restrict__ pos, int n_pos, const int* __restrict__ sel, float* __restrict__ out, int B,
               int L, int d) {
  const int lane = threadIdx.x & 31;
  const long long item = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long n_items = pos ? static_cast<long long>(B) * n_pos : static_cast<long long>(B) * L;
  if (item >= n_items) return;
  int b, t;
  if (pos) { b = static_cast<int>(item / n_pos); t = pos[item]; }
  else { b = static_cast<int>(item / L); t = static_cast<int>(item % L); }
  if (t < 0 || t >= L) {  // invalid position: write NaN so the caller notices
    if (lane < 4 && pos) out[item * 4 + lane] = __int_as_float(0x7fc00000);
    return;
  }
  const T* hf = H + (static_cast<long long>(b) * L + t) * d;
  const T* hr = H + (static_cast<long long>(B + b) * L + (L - 1 - t)) * d;
  float acc[8];
#pragma unroll
  for (int v = 0; v < 8; ++v) acc[v] = 0.f;
  for (int j = lane * 8; j < d; j += 256) {
    float a[8], r[8];
    load8<T>(hf + j, a);
    load8<T>(hr + j, r);
#pragma unroll
    for (int v = 0; v < 8; ++v) {
      const float* wv = W + v * d + j;
      const float* wc = W + static_cast<int>(comp[v]) * d + j;
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[v] = fmaf(a[i], wv[i], fmaf(r[i], wc[i], acc[v]));
    }
  }
#pragma unroll
  for (int v = 0; v < 8; ++v) acc[v] = warp_sum(acc[v]);
  if (lane == 0) {
    if (pos) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int v = sel[k];
        float val = 0.f;
#pragma unroll
        for (int u = 0; u < 8; ++u) val = (u == v) ? acc[u] : val;
        out[item * 4 + k] = val;
      }
    } else {
      float4* o = reinterpret_cast<float4*>(out + item * 8);
      o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
      o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    }
  }
}

// ---- hidden_states[-1] tap (reference train_XGBoost.py:104-105, notebooks/examples.ipynb:183) ----
// out[b, t, j]     = HF[b, t, j]                 j <  d
// out[b, t, d + j] = HR[b, L-1-t, d-1-j]         (RC half: sequence and channel reversed back)
template <typename T>
__global__ void hidden_tap_kernel(const T* __restrict__ H, T* __restrict__ out, int B, int L, int d) {
  const int vec_per_row = (2 * d) / 8;
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(B) * L * vec_per_row;
  if (gid >= total) return;
  const int v = static_cast<int>(gid % vec_per_row);
  const long long bt = gid / vec_per_row;
  const int t = static_cast<int>(bt % L);
  const int b = static_cast<int>(bt / L);
  const int j0 = v * 8;
  float x[8];
  if (j0 < d) {
    load8<T>(H + (static_cast<long long>(b) * L + t) * d + j0, x);
  } else {
    const int jj = j0 - d;  // out channels d+jj .. d+jj+7  <-  HR channels d-1-jj .. d-8-jj
    float y[8];
    load8<T>(H + (static_cast<long long>(B + b) * L + (L - 1 - t)) * d + (d - 8 - jj), y);
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = y[7 - i];
  }
  store8<T>(out + bt * (2 * d) + j0, x);
}

// The same tap at requested positions only (reference train_XGBoost.py:105: hidden_states[-1][:, tokenIdx, :]):
// out[b, i, :] = hidden_states[-1][b, pos[b*n_pos + i], :], without materialising [B, L, 2d].  Invalid positions give NaN.
template <typename T>
__global__ void hidden_tap_pos_kernel(const T* __restrict__ H, const int* __restrict__ pos, int n_pos, T* __restrict__ out,
                                      int B, int L, int d) {
  const int vec_per_row = (2 * d) / 8;
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(B) * n_pos * vec_per_row;
  if (gid >= total) return;
  const int v = static_cast<int>(gid % vec_per_row);
  const long long item = gid / vec_per_row;
  const int b = static_cast<int>(item / n_pos);
  const int t = pos[item];
  const int j0 = v * 8;
  float x[8];
  if (t < 0 || t >= L) {
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = __int_as_float(0x7fc00000);
  } else if (j0 < d) {
    load8<T>(H + (static_cast<long long>(b) * L + t) * d + j0, x);
  } else {
    const int jj = j0 - d;
    float y[8];
    load8<T>(H + (static_cast<long long>(B + b) * L + (L - 1 - t)) * d + (d - 8 - jj), y);
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = y[7 - i];
  }
  store8<T>(out + item * (2 * d) + j0, x);
}

// ---- mean of a hidden_states entry over a range of positions (pcad_hidden_mean_at_layers, pcad_op_hidden_mean) ----
// out[b, j] = mean over t in [s_b, e_b) of hidden_states[b, t, j] (the layout of hidden_tap_kernel), float32, with one
// fixed summation order: fp32 sums of kHiddenMeanChunk consecutive positions counted from s_b, each sequential in t, then
// the chunk partials summed sequentially in chunk order and divided by e_b - s_b (correctly rounded).  The order depends on
// neither B nor any other window, and there are no atomics.  ranges: int32 [B, 2] or nullptr for [0, L).  An invalid range
// (s < 0, e > L or s >= e) gives a NaN row.  part: float [B, ceil(L / kHiddenMeanChunk), 2d] scratch.
constexpr int kHiddenMeanChunk = 128;

__device__ __forceinline__ bool mean_range(const int* ranges, int b, int L, int& s, int& e) {
  s = ranges ? ranges[2 * b] : 0;
  e = ranges ? ranges[2 * b + 1] : L;
  return s >= 0 && e <= L && s < e;
}

// Stage 1: one thread per (window, chunk, 8 output channels) sums its chunk's rows.  The RC half of position t is row
// L-1-t of strand B+b with its channels reversed: the thread reads those rows in t order and reverses the 8 sums on store.
template <typename T>
__global__ void __launch_bounds__(128)
hidden_mean_partial_kernel(const T* __restrict__ H, const int* __restrict__ ranges, float* __restrict__ part, int B, int L,
                           int d, int n_chunks) {
  const int vec_per_row = (2 * d) / 8;
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= static_cast<long long>(B) * n_chunks * vec_per_row) return;
  const int v = static_cast<int>(gid % vec_per_row);
  const long long bc = gid / vec_per_row;
  const int c = static_cast<int>(bc % n_chunks);
  const int b = static_cast<int>(bc / n_chunks);
  int s, e;
  if (!mean_range(ranges, b, L, s, e)) return;
  const int t0 = s + c * kHiddenMeanChunk;
  if (t0 >= e) return;
  const int n = min(kHiddenMeanChunk, e - t0);
  const int j0 = v * 8;
  const bool fwd = j0 < d;
  const T* p = fwd ? H + (static_cast<long long>(b) * L + t0) * d + j0
                   : H + (static_cast<long long>(B + b) * L + (L - 1 - t0)) * d + (2 * d - 8 - j0);
  const long long step = fwd ? d : -static_cast<long long>(d);
  float acc[8];
  load8<T>(p, acc);
#pragma unroll 8
  for (int i = 1; i < n; ++i) {
    float x[8];
    load8<T>(p + i * step, x);
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] += x[k];
  }
  float o[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) o[k] = fwd ? acc[k] : acc[7 - k];
  float4* q = reinterpret_cast<float4*>(part + bc * (2 * d) + j0);
  q[0] = make_float4(o[0], o[1], o[2], o[3]);
  q[1] = make_float4(o[4], o[5], o[6], o[7]);
}

// Stage 2: one thread per (window, output channel) sums that window's chunk partials in chunk order and divides.
__global__ void __launch_bounds__(256)
hidden_mean_final_kernel(const float* __restrict__ part, const int* __restrict__ ranges, float* __restrict__ out, int B,
                         int L, int d, int n_chunks) {
  const int w = 2 * d;
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= static_cast<long long>(B) * w) return;
  const int j = static_cast<int>(gid % w);
  const int b = static_cast<int>(gid / w);
  int s, e;
  if (!mean_range(ranges, b, L, s, e)) {
    out[gid] = __int_as_float(0x7fc00000);
    return;
  }
  const int nc = (e - s + kHiddenMeanChunk - 1) / kHiddenMeanChunk;
  const float* q = part + static_cast<long long>(b) * n_chunks * w + j;
  float acc = q[0];
  int c = 1;
  for (; c + 8 <= nc; c += 8) {
    float x[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) x[u] = q[static_cast<long long>(c + u) * w];
#pragma unroll
    for (int u = 0; u < 8; ++u) acc += x[u];
  }
  for (; c < nc; ++c) acc += q[static_cast<long long>(c) * w];
  out[gid] = __fdiv_rn(acc, static_cast<float>(e - s));
}

}  // namespace pcad
