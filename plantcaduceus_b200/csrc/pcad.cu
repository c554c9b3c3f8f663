// libpcad: C ABI (include/pcad.h) over the sm_100a kernels.  Handle = weights + workspace + launch plan.
#include "../../include/pcad.h"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "elementwise.cuh"
#include "gemm_simt.cuh"
#include "gemm_tcgen05.cuh"
#include "scan.cuh"
#include "ssd.cuh"

using namespace pcad;

namespace {

char g_create_error[512] = "";

struct DirWeights {
  float* conv_w = nullptr;   // [E, 4]
  float* conv_b = nullptr;   // [E]
  void* x_proj = nullptr;    // [RP, E] act dtype, rows >= R+2N zero
  void* dt_proj = nullptr;   // [E, R] act dtype
  float* dt_bias = nullptr;  // [E]
  float* A = nullptr;        // [E, N] = -exp(A_log)
  float* D = nullptr;        // [E]
  float* gnorm_w = nullptr;  // Mamba-2: [E] weight of the mixer's gated RMSNorm (dt_bias, A, D are [H] there)
  bool has[8] = {false, false, false, false, false, false, false, false};
};

struct LayerWeights {
  void* in_proj = nullptr;   // [2E, d] act dtype
  void* in_proj_s = nullptr; // [2E, d] bf16, columns pre-multiplied by norm_w (fused-norm path only)
  void* out_proj = nullptr;  // [d, E] act dtype
  float* norm_w = nullptr;   // [d]
  DirWeights dir[2];
  bool has_in = false, has_out = false, has_norm = false;
};

struct Workspace {
  int B = 0, L = 0;
  size_t bytes = 0;
  uint8_t* base = nullptr;
  uint8_t* ids = nullptr;      // [B, L] u8
  void* hid = nullptr;         // [T, d]
  void* resid = nullptr;       // [T, d] (RT)
  void* normed = nullptr;      // [T, d]
  void* xz = nullptr;          // [T, 2E]
  void* xc[2] = {nullptr, nullptr};     // [T, E]
  void* dbc[2] = {nullptr, nullptr};    // [T, RP]
  void* delta[2] = {nullptr, nullptr};  // [T, E]
  void* y = nullptr;           // [T, E]
  float* sumsq[2] = {nullptr, nullptr};  // [T, parts] per-column-tile sums of squares of the residual stream (fused-norm path)
  float* seg_state = nullptr;  // time-parallel scan: [S*P, 2, E, 16] segment states
  float* seg_sumd = nullptr;   // time-parallel scan: [S*P, 2, E] sums of delta
  float* bcf = nullptr;        // Mamba-1 bf16: fp32 [B ln 2 | C] rows of both directions, [2][T][32] (scan.cuh kScanBcF32)
  uint8_t* ascii = nullptr;    // [B, L] staging for the host entry
  float* logits4 = nullptr;    // [B, 4] staging for the host entry
  int* pos = nullptr;          // [B] staging for the host entry
  int* pos0 = nullptr;         // [B] zeros: positions for the head over the compact (pruned) last layer
};

}  // namespace

struct pcad_handle {
  pcad_config cfg;
  int device = 0;
  int num_sms = 148;
  int d = 0, E = 0, N = 16, R = 0, RP = 0, V = 8;
  bool m2 = false;                     // Mamba-2 / SSD mixer (PlantCAD2)
  int ssd_impl = 0;                    // Mamba-2 bf16 A/B switch: 0 chunked SSD on tcgen05, 1 sequential recurrence
  int H = 0, CD = 0, DIP = 0, DIPP = 0;   // Mamba-2: heads, conv channels (x|B|C), in_proj width (z|x|B|C|dt) and its padded pitch
  bool f32 = false;
  bool fuse_dt = false;                // bf16: dt_proj computed inside the scan (tcgen05), no dt_proj launches, no delta in HBM
  bool bc_f32 = true;                  // bf16: B|C converted to fp32 rows once (bc_to_f32_kernel), scan in its one-barrier mode
  bool bc_f32_force = false;           // ... also below the size where it pays (tests)
  bool fuse_norm = false;   // bf16 activations + bf16 residual: add+RMSNorm folded into the out_proj / in_proj epilogues
  size_t act_size = 2;
  bool finalized = false;
  char err[512] = "";
  std::vector<LayerWeights> layers;
  void* emb = nullptr;        // [V, d] act dtype
  float* head_w = nullptr;    // [V, d] fp32
  float* norm_f = nullptr;    // [d]
  bool has_emb = false, has_norm_f = false;
  bool head_set = false;      // lm_head.lm_head.weight was set: otherwise every finalize derives the tied head from emb
  uint8_t* comp_dev = nullptr;   // [V]
  uint8_t* lut_dev = nullptr;    // [256]
  int* sel_dev = nullptr;        // [4] acgt ids
  int* bad_flag = nullptr;       // out-of-range-id flag: device alias of bad_flag_host (mapped pinned memory)
  volatile int* bad_flag_host = nullptr;
  int mask_id = 1;
  int acgt[4] = {3, 4, 5, 6};
  Workspace ws;
  std::vector<void*> allocs;
  // CUDA graphs of the score-only forward for small batches (launch-bound: ~260 launches of a few microseconds each):
  // one executable graph per (B, L, token_idx), captured on the second call with that shape, replayed afterwards.
  struct ScoreGraph { int B, L, token_idx; bool seen_only; cudaGraphExec_t exec; int64_t launches; };
  std::vector<ScoreGraph> graphs;
  bool prune_last = true;               // score-only calls: last layer computed only at the rows the head reads
  bool last_pruned = false;             // set by run_backbone: ws.normed holds the compact [2B, d] rows
  bool time_parallel = true;            // Mamba-1: segmented scan when the sequential kernel's grid leaves the SMs empty
  bool use_graphs = true;
  cudaStream_t gstream = nullptr;       // capture / replay stream (the caller's may be the legacy default stream, which cannot capture)
  cudaEvent_t g_in = nullptr, g_out = nullptr;
  long long graph_max_tokens = 65536;   // strand-tokens (2 B L) up to which a forward is replayed from a graph
  int64_t graph_replays = 0;            // calls served by a graph captured on an earlier call
  // profiling
  bool profiling = false;
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> prof_events;
  std::vector<cudaEvent_t> event_pool;
  float prof_ms[PCAD_ST_COUNT];
  int64_t prof_launches[PCAD_ST_COUNT];
  int64_t launch_count = 0;
};

namespace {

int fail(pcad_handle* h, int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  char* dst = h ? h->err : g_create_error;
  vsnprintf(dst, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(h, expr)                                                                          \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return fail((h), PCAD_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

template <typename T>
int dev_alloc(pcad_handle* h, T** p, size_t count) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T) > 0 ? count * sizeof(T) : 16);
  if (e != cudaSuccess) return fail(h, PCAD_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", count * sizeof(T), cudaGetErrorString(e));
  h->allocs.push_back(q);
  *p = static_cast<T*>(q);
  return PCAD_OK;
}

// ---- small conversion kernels used at weight-ingest time -------------------------------------
template <typename SrcT, typename DstT>
__global__ void convert_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v;
  if constexpr (sizeof(SrcT) == 2) v = __bfloat162float(src[i]); else v = src[i];
  if constexpr (sizeof(DstT) == 2) dst[i] = __float2bfloat16_rn(v); else dst[i] = v;
}
__global__ void half_to_float_kernel(const __half* __restrict__ src, float* __restrict__ dst, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __half2float(src[i]);
}
// W'[j, k] = W[j, k] * w[k]  (norm weight folded into in_proj's columns; fused-norm path)
__global__ void scale_columns_kernel(const bf16* __restrict__ W, const float* __restrict__ w, bf16* __restrict__ out,
                                     long long rows, int cols) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  out[i] = __float2bfloat16_rn(__bfloat162float(W[i]) * w[i % cols]);
}
// ss[row] = sum_j x[row, j]^2, one warp per row (layer 0 of the fused-norm path: the embedding output)
__global__ void row_sumsq_kernel(const bf16* __restrict__ x, float* __restrict__ ss, long long rows, int d, int parts) {
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float acc = 0.f;
  for (int j = lane * 8; j < d; j += 256) {
    float v[8];
    load16<bf16>(x + row * d + j, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) acc = fmaf(v[k], v[k], acc);
  }
  acc = warp_sum(acc);
  if (lane < parts) ss[row * parts + lane] = lane == 0 ? acc : 0.f;   // slot 0 holds the sum, the other slots are zero
}
__global__ void neg_exp_kernel(float* __restrict__ a, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) a[i] = -expf(a[i]);
}

// Copy `n` elements of src (host or device, src_dtype) into dst (device, fp32 or bf16).
int ingest(pcad_handle* h, const void* src, int src_dtype, void* dst, bool dst_f32, long long n) {
  const size_t src_size = (src_dtype == PCAD_F32) ? 4 : 2;
  void* stage = nullptr;
  CUDA_TRY(h, cudaMalloc(&stage, n * src_size));
  cudaError_t e = cudaMemcpy(stage, src, n * src_size, cudaMemcpyDefault);
  if (e != cudaSuccess) { cudaFree(stage); return fail(h, PCAD_ERR_CUDA, "weight copy failed: %s", cudaGetErrorString(e)); }
  float* f32_tmp = nullptr;
  const void* s = stage;
  int s_dtype = src_dtype;
  const int threads = 256;
  const unsigned blocks = static_cast<unsigned>((n + threads - 1) / threads);
  if (src_dtype == PCAD_F16) {
    e = cudaMalloc(reinterpret_cast<void**>(&f32_tmp), n * 4);
    if (e != cudaSuccess) { cudaFree(stage); return fail(h, PCAD_ERR_NOMEM, "cudaMalloc failed"); }
    half_to_float_kernel<<<blocks, threads>>>(static_cast<const __half*>(stage), f32_tmp, n);
    s = f32_tmp;
    s_dtype = PCAD_F32;
  }
  if (s_dtype == PCAD_F32) {
    if (dst_f32) convert_kernel<float, float><<<blocks, threads>>>(static_cast<const float*>(s), static_cast<float*>(dst), n);
    else convert_kernel<float, bf16><<<blocks, threads>>>(static_cast<const float*>(s), static_cast<bf16*>(dst), n);
  } else {
    if (dst_f32) convert_kernel<bf16, float><<<blocks, threads>>>(static_cast<const bf16*>(s), static_cast<float*>(dst), n);
    else convert_kernel<bf16, bf16><<<blocks, threads>>>(static_cast<const bf16*>(s), static_cast<bf16*>(dst), n);
  }
  e = cudaDeviceSynchronize();
  cudaFree(stage);
  if (f32_tmp) cudaFree(f32_tmp);
  if (e != cudaSuccess) return fail(h, PCAD_ERR_CUDA, "weight conversion failed: %s", cudaGetErrorString(e));
  return PCAD_OK;
}

bool shape_is(const int64_t* shape, int ndim, std::initializer_list<int64_t> want) {
  // compare after dropping size-1 dims from both (conv1d.weight is [E,1,4])
  std::vector<int64_t> a, b;
  for (int i = 0; i < ndim; ++i) if (shape[i] != 1) a.push_back(shape[i]);
  for (int64_t w : want) if (w != 1) b.push_back(w);
  return a == b;
}

// ---- profiling ----------------------------------------------------------------------------------
struct StageTimer {
  pcad_handle* h;
  cudaStream_t st;
  int stage;
  cudaEvent_t a = nullptr, b = nullptr;
  StageTimer(pcad_handle* h_, cudaStream_t st_, int stage_, int launches = 1) : h(h_), st(st_), stage(stage_) {
    h->launch_count += launches;
    if (!h->profiling) return;
    h->prof_launches[stage] += launches;
    auto get = [&]() {
      cudaEvent_t ev;
      if (!h->event_pool.empty()) { ev = h->event_pool.back(); h->event_pool.pop_back(); }
      else cudaEventCreate(&ev);
      return ev;
    };
    a = get(); b = get();
    cudaEventRecord(a, st);
  }
  ~StageTimer() {
    if (!a) return;
    cudaEventRecord(b, st);
    h->prof_events.push_back({stage, {a, b}});
  }
};

// ---- operator launchers (shared by the forward pass and the pcad_op_* entry points) -------------
// The CTA-pair (tcgen05 cta_group::2) GEMM is used for the wide GEMMs unless PCAD_GEMM_2CTA=0.
bool gemm_cta_pair_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("PCAD_GEMM_2CTA");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

int op_linear(pcad_handle* h, const void* A, const void* W, void* C, long long M, int N, int K, long long lda,
              long long ldw, long long ldc, bool f32, int num_sms, cudaStream_t st, int epi = kEpiPlain,
              const EpiParams& ep = EpiParams()) {
  if (f32) {
    if (epi != kEpiPlain) return fail(h, PCAD_ERR_INVALID, "fused GEMM epilogues exist for bf16 only");
    CUDA_TRY(h, gemm_f32_simt(static_cast<const float*>(A), static_cast<const float*>(W), static_cast<float*>(C), M, N, K, lda, ldw, ldc, st));
  } else {
    const char* why = nullptr;
    cudaError_t e = gemm_bf16_tcgen05(static_cast<const bf16*>(A), static_cast<const bf16*>(W), static_cast<bf16*>(C), M, N, K, lda, ldw, ldc, num_sms, st, &why, epi, ep, gemm_cta_pair_enabled());
    if (e != cudaSuccess) return fail(h, why ? PCAD_ERR_INVALID : PCAD_ERR_CUDA, "%s", why ? why : cudaGetErrorString(e));
  }
  return PCAD_OK;
}

template <typename T, typename RT>
int launch_norm_t(pcad_handle* h, const void* x, const void* res_in, const float* w, void* y, void* res_out,
                  long long rows, int d, float eps, cudaStream_t st) {
  const int nvec = d / 8;
  const int ch = (nvec + 31) / 32;
  const int warps = 8;
  const unsigned blocks = static_cast<unsigned>((rows + warps - 1) / warps);
#define NORM_CASE(CHV)                                                                                          \
  add_rmsnorm_kernel<T, RT, CHV><<<blocks, warps * 32, 0, st>>>(static_cast<const T*>(x), static_cast<const RT*>(res_in), w, \
                                                               static_cast<T*>(y), static_cast<RT*>(res_out), rows, d, eps)
  if (ch <= 1) NORM_CASE(1);
  else if (ch <= 2) NORM_CASE(2);
  else if (ch <= 4) NORM_CASE(4);
  else if (ch <= 8) NORM_CASE(8);
  else return fail(h, PCAD_ERR_INVALID, "add_rmsnorm: d=%d too large (max 2048)", d);
#undef NORM_CASE
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

int op_add_rmsnorm(pcad_handle* h, const void* x, const void* res_in, const float* w, void* y, void* res_out,
                   long long rows, int d, float eps, bool f32, bool res_f32, cudaStream_t st) {
  if (d % 8) return fail(h, PCAD_ERR_INVALID, "add_rmsnorm: d must be a multiple of 8");
  if (rows <= 0) return PCAD_OK;
  if (f32) return launch_norm_t<float, float>(h, x, res_in, w, y, res_out, rows, d, eps, st);
  if (res_f32) return launch_norm_t<bf16, float>(h, x, res_in, w, y, res_out, rows, d, eps, st);
  return launch_norm_t<bf16, bf16>(h, x, res_in, w, y, res_out, rows, d, eps, st);
}

int op_conv(pcad_handle* h, const void* x, long long ldx, const float* w_f, const float* b_f, const float* w_r,
            const float* b_r, void* out_f, void* out_r, int S, int L, int E, bool f32, cudaStream_t st) {
  if (E % 4) return fail(h, PCAD_ERR_INVALID, "conv: E must be a multiple of 4");
  if (S <= 0 || L <= 0) return PCAD_OK;
  const int cpt = f32 ? 4 : 2;   // channels per thread
  dim3 grid((E / cpt + 127) / 128, (L + kConvTT - 1) / kConvTT, S);
  if (f32) conv_silu_kernel<float, true, 4><<<grid, 128, 0, st>>>(static_cast<const float*>(x), ldx, w_f, b_f, w_r, b_r, static_cast<float*>(out_f), static_cast<float*>(out_r), L, E);
  else conv_silu_kernel<bf16, false, 2><<<grid, 128, 0, st>>>(static_cast<const bf16*>(x), ldx, w_f, b_f, w_r, b_r, static_cast<bf16*>(out_f), static_cast<bf16*>(out_r), L, E);
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

int op_biscan(pcad_handle* h, const void* u_f, const void* delta_f, const void* bc_f, const void* u_r,
              const void* delta_r, const void* bc_r, long long ldbc, int bc_off, const void* z, long long ldz,
              const float* A_f, const float* D_f, const float* bias_f, const float* A_r, const float* D_r,
              const float* bias_r, void* y, int S, int L, int E, bool f32, cudaStream_t st,
              const void* wdt_f = nullptr, const void* wdt_r = nullptr, long long ldw = 0, int R = 0, int segments = 1,
              float* seg_state = nullptr, float* seg_sumd = nullptr, int Lrun = 0, float* bcf = nullptr) {
  const int vec = f32 ? 4 : 8;
  if (E % vec || ldbc % vec || bc_off % vec || ldz % vec)
    return fail(h, PCAD_ERR_INVALID, "biscan: E, ldbc, bc_off, ldz must be multiples of %d elements", vec);
  if (S <= 0 || L <= 0) return PCAD_OK;
  if (S > 65535) return fail(h, PCAD_ERR_INVALID, "biscan: at most 65535 sequences per call");
  // rejected before anything is launched: these combinations used to be accepted with one argument silently ignored
  if (bcf && (f32 || wdt_f || wdt_r))
    return fail(h, PCAD_ERR_INVALID, "biscan: fp32 B|C rows are a mode of the bf16 scan without the in-kernel dt_proj");
  if (Lrun < 0 || Lrun > L || (Lrun > 0 && Lrun < (L + 1) / 2))
    return fail(h, PCAD_ERR_INVALID, "biscan: Lrun = %d must be 0 or in [(L+1)/2, L] = [%d, %d] (below, some rows are visited by neither direction)",
                Lrun, (L + 1) / 2, L);
  if (Lrun > 0 && Lrun < L && segments > 1)
    return fail(h, PCAD_ERR_INVALID, "biscan: an early-stopped scan (Lrun < L) cannot be time-parallel (segments > 1)");
  cudaError_t e;
#define PCAD_SCAN_ARGS(TT)                                                                                           \
  static_cast<const TT*>(u_f), static_cast<const TT*>(delta_f), static_cast<const TT*>(bc_f), static_cast<const TT*>(u_r), \
      static_cast<const TT*>(delta_r), static_cast<const TT*>(bc_r), ldbc, bc_off, static_cast<const TT*>(z), ldz, A_f, D_f, \
      bias_f, A_r, D_r, bias_r, static_cast<TT*>(y), S, L, E
  const bool fused_dt = wdt_f != nullptr || wdt_r != nullptr;
  // bcf (bf16, not fused): scratch for float [2][S*L][32]; B|C are converted once here and the scan runs its one-barrier mode
  const float* bcf_f = nullptr;
  const float* bcf_r = nullptr;
  if (bcf && !f32 && !fused_dt) {
    const long long rows = static_cast<long long>(S) * L;
    bc_to_f32_kernel<<<static_cast<unsigned>((rows * 8 + 255) / 256), 256, 0, st>>>(static_cast<const bf16*>(bc_f), static_cast<const bf16*>(bc_r),
                                                                                  ldbc, bc_off, bcf, rows);
    CUDA_TRY(h, cudaGetLastError());
    bcf_f = bcf;
    bcf_r = bcf + rows * 2 * kScanN;
  }
  if (segments > 1) {   // time-parallel: `segments` concurrent segments per sequence (scan.cuh)
    if (fused_dt || !seg_state || !seg_sumd || L % segments || static_cast<long long>(S) * segments > 65535)
      return fail(h, PCAD_ERR_INVALID, "biscan: the time-parallel scan needs L %% segments == 0, S * segments <= 65535 and its state buffers");
    if (f32) e = launch_biscan_time_parallel<float, true>(PCAD_SCAN_ARGS(float), segments, seg_state, seg_sumd, st);
    else e = launch_biscan_time_parallel<bf16, false>(PCAD_SCAN_ARGS(bf16), segments, seg_state, seg_sumd, st, bcf_f, bcf_r);
    CUDA_TRY(h, e);
    return PCAD_OK;
  }
  if (fused_dt) {   // delta_* are the x_proj outputs, dt_proj runs inside the kernel (tcgen05)
    if (f32 || !wdt_f || !wdt_r || ldbc < kScanDtK || R <= 0 || R > kScanDtK || ldw < R || ldw % 8)
      return fail(h, PCAD_ERR_INVALID, "biscan: the in-kernel dt_proj needs bf16, both weights (R <= 64, row pitch a multiple of 8) and ldbc >= 64");
    e = launch_biscan<bf16, false, kScanFusedDt>(PCAD_SCAN_ARGS(bf16), st, static_cast<const bf16*>(wdt_f), static_cast<const bf16*>(wdt_r),
                                                 ldw, R, nullptr, Lrun);
  } else if (f32) {
    e = launch_biscan<float, true, kScanPlain>(PCAD_SCAN_ARGS(float), st, nullptr, nullptr, 0, 0, nullptr, Lrun);
  } else if (bcf_f) {
    e = launch_biscan<bf16, false, kScanBcF32>(PCAD_SCAN_ARGS(bf16), st, nullptr, nullptr, 0, 0, nullptr, Lrun, bcf_f, bcf_r);
  } else {
    e = launch_biscan<bf16, false, kScanPlain>(PCAD_SCAN_ARGS(bf16), st, nullptr, nullptr, 0, 0, nullptr, Lrun);
  }
#undef PCAD_SCAN_ARGS
  CUDA_TRY(h, e);
  return PCAD_OK;
}

// ---- workspace ------------------------------------------------------------------------------------
size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
constexpr size_t kSegStateBytes = 16u << 20;   // time-parallel scan: room for S * P * 2 * E * 16 floats at low batch

size_t workspace_layout(const pcad_handle* h, int B, int L, Workspace* ws) {
  const size_t T = 2ull * B * L;
  const size_t a = h->act_size;
  const size_t rs = h->f32 ? 4 : (h->cfg.residual_in_fp32 ? 4 : 2);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
  const size_t o_ids = take(static_cast<size_t>(B) * L);
  const size_t o_hid = take(T * h->d * a);
  const size_t o_res = take(T * h->d * rs);
  const size_t o_nrm = take(T * h->d * a);
  // Mamba-2 reuses the slots: xz = in_proj output [T, DIPP], xc = conv outputs x|B|C [T, CD], delta = per-direction y [T, E]
  const size_t w_xz = h->m2 ? h->DIPP : 2 * h->E, w_xc = h->m2 ? h->CD : h->E, w_dbc = h->m2 ? 0 : h->RP;
  const size_t o_xz = take(T * w_xz * a);
  const size_t o_xc0 = take(T * w_xc * a), o_xc1 = take(T * w_xc * a);
  const size_t o_dbc0 = take(T * w_dbc * a), o_dbc1 = take(T * w_dbc * a);
  const size_t o_dl0 = take(T * h->E * a), o_dl1 = take(T * h->E * a);
  const size_t o_y = take(T * h->E * a);
  const size_t ss_parts = static_cast<size_t>(gemm_sumsq_parts(h->d));
  const size_t o_ss0 = take(T * ss_parts * sizeof(float)), o_ss1 = take(T * ss_parts * sizeof(float));
  const size_t o_segs = take(h->m2 ? 0 : kSegStateBytes), o_segd = take(h->m2 ? 0 : kSegStateBytes / 16);
  const size_t o_bcf = take((h->m2 || h->f32) ? 0 : T * 2 * 2 * kScanN * sizeof(float));   // fp32 [B ln 2 | C] rows, both directions
  const size_t o_ascii = take(static_cast<size_t>(B) * L);
  const size_t o_l4 = take(static_cast<size_t>(B) * 4 * sizeof(float));
  const size_t o_pos = take(static_cast<size_t>(B) * sizeof(int));
  const size_t o_pos0 = take(static_cast<size_t>(B) * sizeof(int));
  if (ws && ws->base) {
    uint8_t* p = ws->base;
    ws->ids = p + o_ids; ws->hid = p + o_hid; ws->resid = p + o_res; ws->normed = p + o_nrm; ws->xz = p + o_xz;
    ws->xc[0] = p + o_xc0; ws->xc[1] = p + o_xc1; ws->dbc[0] = p + o_dbc0; ws->dbc[1] = p + o_dbc1;
    ws->delta[0] = p + o_dl0; ws->delta[1] = p + o_dl1; ws->y = p + o_y;
    ws->sumsq[0] = reinterpret_cast<float*>(p + o_ss0); ws->sumsq[1] = reinterpret_cast<float*>(p + o_ss1);
    ws->seg_state = reinterpret_cast<float*>(p + o_segs); ws->seg_sumd = reinterpret_cast<float*>(p + o_segd);
    ws->bcf = (h->m2 || h->f32) ? nullptr : reinterpret_cast<float*>(p + o_bcf);
    ws->ascii = p + o_ascii; ws->logits4 = reinterpret_cast<float*>(p + o_l4); ws->pos = reinterpret_cast<int*>(p + o_pos);
    ws->pos0 = reinterpret_cast<int*>(p + o_pos0);
  }
  return off;
}

void clear_graphs(pcad_handle* h) {
  for (auto& g : h->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  h->graphs.clear();
}

int ensure_workspace(pcad_handle* h, int B, int L) {
  Workspace& ws = h->ws;
  const size_t need = workspace_layout(h, B, L, nullptr);
  if (ws.base == nullptr || need > ws.bytes) {
    clear_graphs(h);   // captured launches point into the old allocation
    if (ws.base) { cudaDeviceSynchronize(); cudaFree(ws.base); ws.base = nullptr; ws.bytes = 0; }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, need);
    if (e != cudaSuccess) return fail(h, PCAD_ERR_NOMEM, "workspace cudaMalloc(%zu bytes) for B=%d L=%d failed: %s", need, B, L, cudaGetErrorString(e));
    ws.base = static_cast<uint8_t*>(p);
    ws.bytes = need;
  }
  ws.B = B; ws.L = L;
  workspace_layout(h, B, L, &ws);
  return PCAD_OK;
}

// ---- Mamba-2 mixer between in_proj and out_proj: conv + SiLU over x|B|C, SSD scan per direction, gated norms + add ------
int op_ssd_scan(pcad_handle* h, const void* xbc_f, const void* xbc_r, long long ld_xbc, const void* dt_raw, long long ld_dt,
                const float* A_f, const float* D_f, const float* bias_f, const float* A_r, const float* D_r, const float* bias_r,
                void* y_f, void* y_r, int S, int L, int H, bool f32, int impl, cudaStream_t st) {
  // impl (bf16): 0 = chunked SSD on tcgen05 (ssd_chunk_tc_kernel), 1 = sequential recurrence
  const bool sequential = impl == 1;
  if (S <= 0 || L <= 0) return PCAD_OK;
  if (H <= 0 || S > 65535) return fail(h, PCAD_ERR_INVALID, "ssd_scan: need H > 0 and at most 65535 sequences per call");
  cudaError_t e;
  if (f32) {
    e = launch_ssd_seq<float>(static_cast<const float*>(xbc_f), static_cast<const float*>(xbc_r), ld_xbc, static_cast<const float*>(dt_raw),
                              ld_dt, A_f, D_f, bias_f, A_r, D_r, bias_r, static_cast<float*>(y_f), static_cast<float*>(y_r), S, L, H, st);
  } else if (sequential) {
    e = launch_ssd_seq<bf16>(static_cast<const bf16*>(xbc_f), static_cast<const bf16*>(xbc_r), ld_xbc, static_cast<const bf16*>(dt_raw),
                             ld_dt, A_f, D_f, bias_f, A_r, D_r, bias_r, static_cast<bf16*>(y_f), static_cast<bf16*>(y_r), S, L, H, st);
  } else {
    if ((H & 1) || (ld_xbc % 8) || (reinterpret_cast<uintptr_t>(xbc_f) & 15) || (reinterpret_cast<uintptr_t>(xbc_r) & 15) ||
        (reinterpret_cast<uintptr_t>(y_f) & 15) || (reinterpret_cast<uintptr_t>(y_r) & 15))
      return fail(h, PCAD_ERR_INVALID, "ssd_scan: the tensor-core kernel needs an even head count, 16-byte aligned tensors and ld_xbc %% 8 == 0");
    e = launch_ssd_tc(static_cast<const bf16*>(xbc_f), static_cast<const bf16*>(xbc_r), ld_xbc, static_cast<const bf16*>(dt_raw), ld_dt,
                      A_f, D_f, bias_f, A_r, D_r, bias_r, static_cast<bf16*>(y_f), static_cast<bf16*>(y_r), S, L, H, st);
  }
  CUDA_TRY(h, e);
  return PCAD_OK;
}

int op_gated_norm_sum(pcad_handle* h, const void* y_f, const void* y_r, const void* z, long long ldz, const float* w_f,
                      const float* w_r, void* out, long long rows, int E, float eps, bool f32, cudaStream_t st) {
  if (rows <= 0) return PCAD_OK;
  const int vec = f32 ? 4 : 8;
  if (E % vec || ldz % vec) return fail(h, PCAD_ERR_INVALID, "gated_norm_sum: E and ldz must be multiples of %d", vec);
  const unsigned blocks = static_cast<unsigned>((rows + 7) / 8);
  if (!f32 && E <= 256 * 12) {   // bf16: the row stays in registers between the statistics and the output
    const int ch = (E + 255) / 256;
#define GN_CASE(CHV)                                                                                                        \
  gated_norm_sum_regs_kernel<CHV><<<blocks, 256, 0, st>>>(static_cast<const bf16*>(y_f), static_cast<const bf16*>(y_r),        \
                                                          static_cast<const bf16*>(z), ldz, w_f, w_r, static_cast<bf16*>(out), rows, E, eps)
    if (ch <= 1) GN_CASE(1);
    else if (ch <= 2) GN_CASE(2);
    else if (ch <= 3) GN_CASE(3);
    else if (ch <= 4) GN_CASE(4);
    else if (ch <= 6) GN_CASE(6);
    else if (ch <= 8) GN_CASE(8);
    else GN_CASE(12);
#undef GN_CASE
    CUDA_TRY(h, cudaGetLastError());
    return PCAD_OK;
  }
  if (f32) gated_norm_sum_kernel<float, true><<<blocks, 256, 0, st>>>(static_cast<const float*>(y_f), static_cast<const float*>(y_r), static_cast<const float*>(z), ldz, w_f, w_r, static_cast<float*>(out), rows, E, eps);
  else gated_norm_sum_kernel<bf16, false><<<blocks, 256, 0, st>>>(static_cast<const bf16*>(y_f), static_cast<const bf16*>(y_r), static_cast<const bf16*>(z), ldz, w_f, w_r, static_cast<bf16*>(out), rows, E, eps);
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

static_assert(kHiddenMeanChunk == PCAD_HIDDEN_MEAN_CHUNK, "pcad.h states the chunk length of the pooled mean");

// Mean over each window's range of one hidden_states entry held as strand-major [2BL, d] rows -> out float [B, 2d] (two
// launches: chunk partials into `scratch`, float [B, ceil(L / kHiddenMeanChunk), 2d], then their sum in chunk order).
int op_hidden_mean(pcad_handle* h, const void* rows, const int32_t* ranges, float* scratch, float* out, int B, int L, int d,
                   bool f32, cudaStream_t st) {
  if (d <= 0 || d % 8) return fail(h, PCAD_ERR_INVALID, "hidden_mean: d must be a positive multiple of 8");
  if (B < 0 || L < 0) return fail(h, PCAD_ERR_INVALID, "hidden_mean: negative batch or length");
  if (B == 0 || L == 0) return PCAD_OK;
  const int n_chunks = (L + kHiddenMeanChunk - 1) / kHiddenMeanChunk;
  const long long items = static_cast<long long>(B) * n_chunks * (2 * d / 8);
  const unsigned blocks1 = static_cast<unsigned>((items + 127) / 128);
  if (f32) hidden_mean_partial_kernel<float><<<blocks1, 128, 0, st>>>(static_cast<const float*>(rows), ranges, scratch, B, L, d, n_chunks);
  else hidden_mean_partial_kernel<bf16><<<blocks1, 128, 0, st>>>(static_cast<const bf16*>(rows), ranges, scratch, B, L, d, n_chunks);
  const unsigned blocks2 = static_cast<unsigned>((static_cast<long long>(B) * 2 * d + 255) / 256);
  hidden_mean_final_kernel<<<blocks2, 256, 0, st>>>(scratch, ranges, out, B, L, d, n_chunks);
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

// ws.xz holds in_proj's output [T, DIPP]: z at [0, E), x|B|C at [E, E + CD), dt at [E + CD, E + CD + H).  Leaves the summed,
// normed y in ws.y.  [EXT mamba_ssm Mamba2.forward, non-fused branch; BiMambaWrapper "add" with tied projections]
int run_mixer_m2(pcad_handle* h, LayerWeights& lw, int S, int L, cudaStream_t st) {
  Workspace& ws = h->ws;
  const long long T = static_cast<long long>(S) * L;
  const int E = h->E, CD = h->CD, H = h->H;
  const bool f32 = h->f32;
  const size_t a = h->act_size;
  uint8_t* zx = static_cast<uint8_t*>(ws.xz);
  int rc;
  {
    StageTimer tm(h, st, PCAD_ST_CONV);
    rc = op_conv(h, zx + static_cast<size_t>(E) * a, h->DIPP, lw.dir[0].conv_w, lw.dir[0].conv_b, lw.dir[1].conv_w, lw.dir[1].conv_b,
                 ws.xc[0], ws.xc[1], S, L, CD, f32, st);
    if (rc) return rc;
  }
  {
    StageTimer tm(h, st, PCAD_ST_SCAN);
    rc = op_ssd_scan(h, ws.xc[0], ws.xc[1], CD, zx + static_cast<size_t>(E + CD) * a, h->DIPP, lw.dir[0].A, lw.dir[0].D, lw.dir[0].dt_bias,
                     lw.dir[1].A, lw.dir[1].D, lw.dir[1].dt_bias, ws.delta[0], ws.delta[1], S, L, H, f32, h->ssd_impl, st);
    if (rc) return rc;
  }
  {
    StageTimer tm(h, st, PCAD_ST_GNORM);
    rc = op_gated_norm_sum(h, ws.delta[0], ws.delta[1], zx, h->DIPP, lw.dir[0].gnorm_w, lw.dir[1].gnorm_w, ws.y, T, E, 1e-5f, f32, st);
    if (rc) return rc;
  }
  return PCAD_OK;
}

// Mamba-1, low batch / long context: cut every sequence into P concurrent segments while the sequential kernel's grid
// (E / 64 x S CTAs) would leave resident slots (4 per SM) empty and the segments stay >= 512 steps long.  (Measured:
// with shorter segments the two extra passes cost more than the parallelism returns -- B = 4, L = 512: 10.9 vs 6.5 ms;
// and 512-bp windows, the scoring workload, keep the property that a window scores the same bits alone or in a batch.)
int scan_segments(const pcad_handle* h, int S, int L) {
  int P = 1;
  if (!h->time_parallel) return P;
  const long long ctas = static_cast<long long>((h->E + kScanCH - 1) / kScanCH) * S, slots = 4LL * h->num_sms;
  while (P < 32 && ctas * P * 2 <= slots && L % (P * 2) == 0 && L / (P * 2) >= 512 &&
         static_cast<size_t>(S) * P * 2 * 2 * h->E * kScanN * sizeof(float) <= kSegStateBytes)
    P *= 2;
  return P;
}

// ws.xz holds in_proj's output [T, 2E]: x at [0, E), z at [E, 2E).  Leaves y in ws.y.  prune_idx >= 0: the scan may stop once
// both directions have reached row prune_idx; *pruned tells whether it did (y is then valid only at the rows the head reads).
int run_mixer_m1(pcad_handle* h, LayerWeights& lw, int S, int L, int prune_idx, bool* pruned, cudaStream_t st) {
  Workspace& ws = h->ws;
  const long long T = static_cast<long long>(S) * L;
  const int E = h->E, R = h->R, RP = h->RP;
  const bool f32 = h->f32;
  int rc;
  {
    StageTimer tm(h, st, PCAD_ST_CONV);
    rc = op_conv(h, ws.xz, 2 * E, lw.dir[0].conv_w, lw.dir[0].conv_b, lw.dir[1].conv_w, lw.dir[1].conv_b, ws.xc[0], ws.xc[1], S, L, E, f32, st);
    if (rc) return rc;
  }
  const int P = scan_segments(h, S, L);
  // dt_proj runs inside the scan kernel (tcgen05, scan.cuh) unless the time-parallel passes need delta in memory
  const bool fuse_dt = h->fuse_dt && P == 1;
  for (int dir = 0; dir < 2; ++dir) {
    {
      StageTimer tm(h, st, PCAD_ST_X_PROJ);
      rc = op_linear(h, ws.xc[dir], lw.dir[dir].x_proj, ws.dbc[dir], T, RP, E, E, E, RP, f32, h->num_sms, st);
      if (rc) return rc;
    }
    if (!fuse_dt) {
      StageTimer tm(h, st, PCAD_ST_DT_PROJ);
      rc = op_linear(h, ws.dbc[dir], lw.dir[dir].dt_proj, ws.delta[dir], T, E, R, RP, R, E, f32, h->num_sms, st);
      if (rc) return rc;
    }
  }
  StageTimer tm(h, st, PCAD_ST_SCAN);
  const uint8_t* zbase = static_cast<const uint8_t*>(ws.xz) + static_cast<size_t>(E) * h->act_size;
  *pruned = prune_idx >= 0 && P == 1 && L >= 8;
  const int Lrun = *pruned ? (prune_idx > L - 1 - prune_idx ? prune_idx : L - 1 - prune_idx) + 1 : 0;
  // fp32 B|C rows + one-barrier scan mode: one more (tiny) launch per layer, so only where the scan is long enough to
  // repay it (measured: -1 ms of 170 per step at T = 262 144; launch-bound small batches keep the in-kernel conversion)
  const bool use_bcf = h->bc_f32 && !f32 && (h->bc_f32_force || T >= 65536);
  if (fuse_dt)   // the scan reads the x_proj outputs (dt | B | C) and the dt_proj weights
    return op_biscan(h, ws.xc[0], ws.dbc[0], ws.dbc[0], ws.xc[1], ws.dbc[1], ws.dbc[1], RP, R, zbase, 2 * E,
                     lw.dir[0].A, lw.dir[0].D, lw.dir[0].dt_bias, lw.dir[1].A, lw.dir[1].D, lw.dir[1].dt_bias, ws.y, S, L, E, f32,
                     st, lw.dir[0].dt_proj, lw.dir[1].dt_proj, R, R, 1, nullptr, nullptr, Lrun);
  rc = op_biscan(h, ws.xc[0], ws.delta[0], ws.dbc[0], ws.xc[1], ws.delta[1], ws.dbc[1], RP, R, zbase, 2 * E,
                 lw.dir[0].A, lw.dir[0].D, lw.dir[0].dt_bias, lw.dir[1].A, lw.dir[1].D, lw.dir[1].dt_bias, ws.y, S, L, E, f32, st,
                 nullptr, nullptr, 0, 0, P, ws.seg_state, ws.seg_sumd, Lrun, use_bcf ? ws.bcf : nullptr);
  if (P > 1) h->launch_count += 2;
  if (use_bcf) h->launch_count += 1;
  return rc;
}

// Score-only last layer: rows (s, row_s) of a [S*L, width] tensor -> compact [S, width]; row_s = idx for the forward strands
// (s < B) and L-1-idx for the RC strands.  16-byte vectors.
__global__ void gather_rows_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int S, int B, int L, int idx, int vec_per_row) {
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= static_cast<long long>(S) * vec_per_row) return;
  const int s = static_cast<int>(gid / vec_per_row), v = static_cast<int>(gid % vec_per_row);
  const int row = s < B ? idx : L - 1 - idx;
  dst[gid] = src[(static_cast<long long>(s) * L + row) * vec_per_row + v];
}

// ---- hidden-state taps ---------------------------------------------------------------------------------
// Which entries of the reference's hidden_states tuple a forward emits, and where: idx[i] (strictly increasing, in
// [0, n_layer]) goes to dst[i], [B, L, 2d] in the model dtype; or, with pos, [B, n_pos, 2d] at the positions pos[b, :];
// or, with mean, float [B, 2d] at mean + i * B * 2d: the mean over each window's range (op_hidden_mean).
struct Taps {
  int n = 0;
  const int32_t* idx = nullptr;
  void* const* dst = nullptr;
  const int32_t* pos = nullptr;   // device, [B, n_pos]; nullptr: every position
  int n_pos = 0;
  float* mean = nullptr;          // device, [n, B, 2d]: pooled mode (dst and pos unused)
  const int32_t* ranges = nullptr;   // device, [B, 2] for the pooled mode; nullptr: [0, L) for every window
  int deepest() const { return n > 0 ? idx[n - 1] : -1; }
  int find(int k) const {   // i with idx[i] == k, or -1
    for (int i = 0; i < n; ++i)
      if (idx[i] == k) return i;
    return -1;
  }
};

// Writes hidden_states[k] from the strand-major [2BL, d] rows `src` into dst[i] if k is tap i (hidden_tap_kernel /
// hidden_tap_pos_kernel: the RC half reversed in time and channels), or its per-window mean in the pooled mode.
int emit_tap(pcad_handle* h, const Taps* taps, int k, const void* src, int B, int L, cudaStream_t st) {
  const int i = taps ? taps->find(k) : -1;
  if (i < 0) return PCAD_OK;
  StageTimer tm(h, st, PCAD_ST_MISC, taps->mean ? 2 : 1);
  const int d = h->d;
  if (taps->mean) {
    // the partials, 2B ceil(L / P) d floats, go to ws.delta[0] ([T, E] with E = 2d, so they fit): the scan has consumed it
    // whenever a tap is emitted, and the pruned last layer that reuses it never runs with taps
    return op_hidden_mean(h, src, taps->ranges, static_cast<float*>(h->ws.delta[0]), taps->mean + static_cast<size_t>(i) * B * 2 * d,
                          B, L, d, h->f32, st);
  }
  if (taps->pos) {
    const long long total = static_cast<long long>(B) * taps->n_pos * (2 * d / 8);
    const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
    if (h->f32) hidden_tap_pos_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(src), taps->pos, taps->n_pos, static_cast<float*>(taps->dst[i]), B, L, d);
    else hidden_tap_pos_kernel<bf16><<<blocks, 256, 0, st>>>(static_cast<const bf16*>(src), taps->pos, taps->n_pos, static_cast<bf16*>(taps->dst[i]), B, L, d);
  } else {
    const long long total = static_cast<long long>(B) * L * (2 * d / 8);
    const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
    if (h->f32) hidden_tap_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(src), static_cast<float*>(taps->dst[i]), B, L, d);
    else hidden_tap_kernel<bf16><<<blocks, 256, 0, st>>>(static_cast<const bf16*>(src), static_cast<bf16*>(taps->dst[i]), B, L, d);
  }
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

// ---- the forward pass over the strand-major layout --------------------------------------------------
// ids (u8 [B, L]) are already in ws.ids.  Leaves the final normed hidden state in ws.normed.
// prune_idx >= 0 (score-only calls with one scored position per window): the LAST layer is computed only as far as the head
// needs it -- the scan stops once both directions have reached the scored position (about half the steps at the window centre),
// out_proj / residual / final norm run on the 2B rows the head reads, and ws.normed comes back COMPACT as [2B, d] (the head is then
// called with L = 1, position 0).  Bit-identical to the full computation at those rows.
// taps (never with prune_idx): the hidden_states entries to emit as each comes into existence -- 0 the embedding, k in
// [1, n_layer) layer k-1's out_proj output before the residual add, n_layer the final norm.  With full = false the forward
// stops after the layer that produces the deepest requested entry, and runs the final norm only if n_layer is requested.
int run_backbone(pcad_handle* h, int B, int L, cudaStream_t st, int prune_idx = -1, const Taps* taps = nullptr, bool full = true) {
  Workspace& ws = h->ws;
  const long long T = 2LL * B * L;
  const int S = 2 * B;
  const int d = h->d, E = h->E;
  const bool f32 = h->f32;
  const bool res_f32 = f32 || h->cfg.residual_in_fp32;
  const bool fused = h->fuse_norm;
  // Fused-norm path (bf16 activations, bf16 residual): the residual stream lives in ws.resid, its row sums of
  // squares in ws.sumsq[cur]; out_proj's epilogue adds into it, in_proj's epilogue applies rstd.  Otherwise the
  // block is norm kernel -> in_proj ... out_proj -> ws.hid, exactly the reference's order of roundings.
  int cur = 0;
  h->last_pruned = false;
  const int parts = gemm_sumsq_parts(d);
  const int n_in = h->m2 ? h->DIP : 2 * E;          // in_proj output width and row pitch
  const long long ld_in = h->m2 ? h->DIPP : 2 * E;
  // The block tail: out_proj reads `rows` rows of y and writes x (adding the residual stream res in the fused path), the
  // final norm reads x and res.  All T rows, unless the last layer was pruned to the 2B rows the head reads.
  long long rows = T;
  void* y = ws.y;
  void* res = ws.resid;
  void* x = fused ? ws.resid : ws.hid;
  {
    StageTimer tm(h, st, PCAD_ST_EMBED, fused ? 2 : 1);
    const long long total = T * (d / 8);
    const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
    if (f32) embed_kernel<float><<<blocks, 256, 0, st>>>(ws.ids, static_cast<const float*>(h->emb), static_cast<float*>(ws.hid), B, L, d, h->comp_dev);
    else embed_kernel<bf16><<<blocks, 256, 0, st>>>(ws.ids, static_cast<const bf16*>(h->emb), static_cast<bf16*>(fused ? ws.resid : ws.hid), B, L, d, h->comp_dev);
    if (fused) row_sumsq_kernel<<<static_cast<unsigned>((T + 7) / 8), 256, 0, st>>>(static_cast<const bf16*>(ws.resid), ws.sumsq[cur], T, d, parts);
    CUDA_TRY(h, cudaGetLastError());
  }
  int rc = emit_tap(h, taps, 0, x, B, L, st);
  if (rc) return rc;
  const int n_layer = h->cfg.n_layer;
  const int n_run = full || !taps ? n_layer : (taps->deepest() < n_layer ? taps->deepest() : n_layer);
  for (int li = 0; li < n_run; ++li) {
    LayerWeights& lw = h->layers[li];
    if (!fused) {
      StageTimer tm(h, st, PCAD_ST_NORM);
      rc = op_add_rmsnorm(h, ws.hid, li == 0 ? nullptr : ws.resid, lw.norm_w, ws.normed, ws.resid, T, d, h->cfg.norm_eps, f32, res_f32, st);
      if (rc) return rc;
    }
    {
      StageTimer tm(h, st, PCAD_ST_IN_PROJ);
      if (fused) {
        EpiParams ep;
        ep.sumsq_in = ws.sumsq[cur];
        ep.sumsq_parts = parts;
        ep.inv_k = 1.0f / static_cast<float>(d);
        ep.eps = h->cfg.norm_eps;
        rc = op_linear(h, ws.resid, lw.in_proj_s, ws.xz, T, n_in, d, d, d, ld_in, false, h->num_sms, st, kEpiRowScale, ep);
      } else {
        rc = op_linear(h, ws.normed, lw.in_proj, ws.xz, T, n_in, d, d, d, ld_in, f32, h->num_sms, st);
      }
      if (rc) return rc;
    }
    bool pruned = false;
    rc = h->m2 ? run_mixer_m2(h, lw, S, L, st)
               : run_mixer_m1(h, lw, S, L, li == h->cfg.n_layer - 1 ? prune_idx : -1, &pruned, st);
    if (rc) return rc;
    if (pruned) {
      // compact tail: y and the residual stream at the 2B rows the head reads; out_proj and the final norm then run on those
      const size_t a = h->act_size, rs = res_f32 ? 4 : a;
      uint8_t* yc = static_cast<uint8_t*>(ws.delta[0]);                                  // [S, E]   (delta is dead after the scan)
      uint8_t* rc_in = static_cast<uint8_t*>(ws.delta[1]);                               // [S, d]   residual rows
      {
        StageTimer tm(h, st, PCAD_ST_MISC, 2);
        const int vy = static_cast<int>(E * a / 16), vr = static_cast<int>(d * rs / 16);
        gather_rows_kernel<<<static_cast<unsigned>((static_cast<long long>(S) * vy + 255) / 256), 256, 0, st>>>(
            static_cast<const uint4*>(ws.y), reinterpret_cast<uint4*>(yc), S, B, L, prune_idx, vy);
        gather_rows_kernel<<<static_cast<unsigned>((static_cast<long long>(S) * vr + 255) / 256), 256, 0, st>>>(
            static_cast<const uint4*>(ws.resid), reinterpret_cast<uint4*>(rc_in), S, B, L, prune_idx, vr);
        CUDA_TRY(h, cudaGetLastError());
      }
      h->last_pruned = true;
      rows = S;
      y = yc;
      res = rc_in;
      x = rc_in + align_up(static_cast<size_t>(S) * d * 4, 1024);                       // [S, d]   new residual / out_proj output
    }
    // hidden_states[li + 1] is this layer's out_proj output (the last layer's is not an entry: index n_layer is the final norm)
    const bool tap_here = taps && li + 1 < n_layer && taps->find(li + 1) >= 0;
    {
      StageTimer tm(h, st, PCAD_ST_OUT_PROJ);
      if (fused) {
        // the fused path never stores the pre-residual output, except as the tap: into ws.hid, which it does not otherwise use
        EpiParams ep;
        ep.resid = static_cast<const bf16*>(res);
        ep.ld_res = d;
        ep.sumsq_out = ws.sumsq[cur ^ 1];
        ep.sumsq_parts = parts;
        ep.tap = static_cast<bf16*>(ws.hid);
        ep.ld_tap = d;
        rc = op_linear(h, y, lw.out_proj, x, rows, d, E, E, E, d, false, h->num_sms, st, tap_here ? kEpiResidualTap : kEpiResidual, ep);
        cur ^= 1;
      } else {
        rc = op_linear(h, y, lw.out_proj, x, rows, d, E, E, E, d, f32, h->num_sms, st);
      }
      if (rc) return rc;
    }
    if (tap_here) {
      rc = emit_tap(h, taps, li + 1, ws.hid, B, L, st);
      if (rc) return rc;
    }
  }
  if (n_run < n_layer) return PCAD_OK;   // stopped early: the final norm is not requested
  {
    // the fused path has already added the residual in out_proj's epilogue; without a layer there is no residual yet
    StageTimer tm(h, st, PCAD_ST_NORM);
    rc = op_add_rmsnorm(h, x, fused || n_layer == 0 ? nullptr : res, h->norm_f, ws.normed, nullptr, rows, d, h->cfg.norm_eps,
                        f32, res_f32, st);
    if (rc) return rc;
  }
  return emit_tap(h, taps, n_layer, ws.normed, B, L, st);
}

int run_head(pcad_handle* h, int B, int L, const int* pos_dev, int n_pos, float* out, cudaStream_t st) {
  StageTimer tm(h, st, PCAD_ST_HEAD);
  const long long items = pos_dev ? static_cast<long long>(B) * n_pos : static_cast<long long>(B) * L;
  if (items <= 0) return PCAD_OK;
  const unsigned blocks = static_cast<unsigned>((items + 7) / 8);
  if (h->f32) lm_head_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(h->ws.normed), h->head_w, h->comp_dev, pos_dev, n_pos, h->sel_dev, out, B, L, h->d);
  else lm_head_kernel<bf16><<<blocks, 256, 0, st>>>(static_cast<const bf16*>(h->ws.normed), h->head_w, h->comp_dev, pos_dev, n_pos, h->sel_dev, out, B, L, h->d);
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

__global__ void fill_int_kernel(int* p, int n, int v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

constexpr int kNoWork = 1;   // begin_call: B, L or the count is 0, the call returns PCAD_OK without computing anything

// Start of every forward entry point: checks the handle and the shape, returns kNoWork for an empty call, then reports
// `args_msg` unless `args_ok` (the entry's own pointer and count checks) and checks token_idx (the default 0 is in range for
// every L > 0).  Returns PCAD_OK once the device is selected and the workspace fits B x L.
int begin_call(pcad_handle* h, int B, int L, int count, bool args_ok, const char* args_msg, int token_idx = 0) {
  if (!h) return PCAD_ERR_INVALID;
  if (!h->finalized) return fail(h, PCAD_ERR_STATE, "pcad_finalize must succeed before a forward call");
  if (B < 0 || L < 0) return fail(h, PCAD_ERR_INVALID, "negative batch or length");
  if (2LL * B > 65535) return fail(h, PCAD_ERR_INVALID, "B=%d too large for one call (max 32767)", B);
  if (B == 0 || L == 0 || count == 0) return kNoWork;
  if (!args_ok) return fail(h, PCAD_ERR_INVALID, "%s", args_msg);
  if (token_idx < 0 || token_idx >= L) return fail(h, PCAD_ERR_INVALID, "token_idx %d outside [0, %d)", token_idx, L);
  CUDA_TRY(h, cudaSetDevice(h->device));
  return ensure_workspace(h, B, L);
}

// ids (u8 [B, L], device) -> ws.ids, checked: ids >= vocab_size would index past the embedding table / complement map.
// token_idx >= 0 (score_at): also the head positions ws.pos = token_idx and ws.pos0 = 0.
int stage_ids(pcad_handle* h, const uint8_t* ids_dev, int B, int L, int token_idx, cudaStream_t st) {
  Workspace& ws = h->ws;
  StageTimer tm(h, st, PCAD_ST_MISC, token_idx >= 0 ? 3 : 1);
  const long long n = static_cast<long long>(B) * L;
  ids_u8_check_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(ids_dev, ws.ids, n, h->V, h->bad_flag);
  if (token_idx >= 0) {
    fill_int_kernel<<<(B + 255) / 256, 256, 0, st>>>(ws.pos, B, token_idx);
    fill_int_kernel<<<(B + 255) / 256, 256, 0, st>>>(ws.pos0, B, 0);
  }
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

// ids (int64 [B, L], device) -> ws.ids, checked as stage_ids does.
int stage_ids64(pcad_handle* h, const int64_t* ids_dev, int B, int L, cudaStream_t st) {
  StageTimer tm(h, st, PCAD_ST_MISC);
  const long long n = static_cast<long long>(B) * L;
  ids64_to_u8_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(reinterpret_cast<const long long*>(ids_dev), h->ws.ids, n, h->V, h->bad_flag);
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

// The tap list of pcad_forward_taps / pcad_hidden_at_layers, checked before anything is launched.
int check_taps(pcad_handle* h, int n_taps, const int32_t* tap_idx) {
  const int n_layer = h->cfg.n_layer;
  if (n_taps < 1 || n_taps > n_layer + 1) return fail(h, PCAD_ERR_INVALID, "n_taps = %d outside [1, n_layer + 1 = %d]", n_taps, n_layer + 1);
  if (!tap_idx) return fail(h, PCAD_ERR_INVALID, "tap_idx is null");
  for (int i = 0; i < n_taps; ++i) {
    if (tap_idx[i] < 0 || tap_idx[i] > n_layer) return fail(h, PCAD_ERR_INVALID, "tap_idx[%d] = %d outside [0, n_layer = %d]", i, tap_idx[i], n_layer);
    if (i > 0 && tap_idx[i] <= tap_idx[i - 1]) return fail(h, PCAD_ERR_INVALID, "tap_idx is not strictly increasing at %d", i);
  }
  return PCAD_OK;
}

// Backbone + head at token_idx -> out [B, 4]; ws.ids, ws.pos and ws.pos0 are staged.  One scored position, the same in every
// window: the last layer is computed only at the rows the head reads.
int score_at(pcad_handle* h, int B, int L, int token_idx, float* out, cudaStream_t st) {
  Workspace& ws = h->ws;
  const bool prune = h->prune_last && !h->m2 && h->cfg.n_layer > 0;
  int rc = run_backbone(h, B, L, st, prune ? token_idx : -1);
  if (rc) return rc;
  if (h->last_pruned) return run_head(h, B, 1, ws.pos0, 1, out, st);   // ws.normed is compact [2B, d]
  return run_head(h, B, L, ws.pos, 1, out, st);
}

}  // namespace

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

int pcad_abi_version(void) { return PCAD_ABI_VERSION; }

const char* pcad_last_error(const pcad_handle* h) { return h ? h->err : g_create_error; }

int pcad_create(const pcad_config* cfg, int device, pcad_handle** out) {
  if (!cfg || !out) return fail(nullptr, PCAD_ERR_INVALID, "null argument");
  *out = nullptr;
  const bool m2 = cfg->mixer == PCAD_MIXER_MAMBA2;
  if (cfg->mixer != PCAD_MIXER_MAMBA1 && !m2) return fail(nullptr, PCAD_ERR_INVALID, "unknown mixer %d", cfg->mixer);
  if (m2) {
    if (cfg->d_state != 64 || cfg->headdim != 64 || cfg->ngroups != 1)
      return fail(nullptr, PCAD_ERR_INVALID, "unsupported Mamba-2 shape d_state=%d headdim=%d ngroups=%d (engine is specialised for 64 / 64 / 1)",
                  cfg->d_state, cfg->headdim, cfg->ngroups);
    if ((cfg->expand * cfg->d_model / 64) % 2) return fail(nullptr, PCAD_ERR_INVALID, "Mamba-2 needs an even number of heads");
  } else if (cfg->d_state != 16) {
    return fail(nullptr, PCAD_ERR_INVALID, "unsupported d_state=%d (engine is specialised for 16)", cfg->d_state);
  }
  if (cfg->d_conv != 4) return fail(nullptr, PCAD_ERR_INVALID, "unsupported d_conv=%d (engine is specialised for 4)", cfg->d_conv);
  if (cfg->vocab_size != 8) return fail(nullptr, PCAD_ERR_INVALID, "unsupported vocab_size=%d (LM head is specialised for 8 rows)", cfg->vocab_size);
  if (cfg->d_model <= 0 || cfg->d_model % 128 != 0 || cfg->d_model > 2048)
    return fail(nullptr, PCAD_ERR_INVALID, "unsupported d_model=%d (need a multiple of 128, <= 2048)", cfg->d_model);
  if (cfg->expand != 2) return fail(nullptr, PCAD_ERR_INVALID, "unsupported expand=%d", cfg->expand);
  if (!m2 && (cfg->dt_rank <= 0 || cfg->dt_rank % 8 != 0)) return fail(nullptr, PCAD_ERR_INVALID, "unsupported dt_rank=%d (need a multiple of 8)", cfg->dt_rank);
  if (cfg->n_layer < 0) return fail(nullptr, PCAD_ERR_INVALID, "negative n_layer");
  if (cfg->dtype != PCAD_BF16 && cfg->dtype != PCAD_F32) return fail(nullptr, PCAD_ERR_INVALID, "dtype must be PCAD_BF16 or PCAD_F32");
  for (int i = 0; i < cfg->vocab_size; ++i)
    if (cfg->complement_map[i] < 0 || cfg->complement_map[i] >= cfg->vocab_size)
      return fail(nullptr, PCAD_ERR_INVALID, "complement_map[%d]=%d out of range", i, cfg->complement_map[i]);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, PCAD_ERR_CUDA, "no CUDA device available (%s); libpcad has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(nullptr, PCAD_ERR_INVALID, "device %d out of range (have %d)", device, ndev);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, PCAD_ERR_CUDA, "cudaSetDevice failed: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10)
    return fail(nullptr, PCAD_ERR_CUDA, "device %d is sm_%d%d; libpcad is built for sm_100a only", device, prop.major, prop.minor);

  pcad_handle* h = new pcad_handle();
  h->cfg = *cfg;
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  h->d = cfg->d_model;
  h->E = cfg->expand * cfg->d_model;
  h->N = cfg->d_state;
  h->R = cfg->dt_rank;
  h->RP = (h->R + 2 * h->N + 15) / 16 * 16;
  h->m2 = m2;
  if (m2) {
    h->H = h->E / 64;
    h->CD = h->E + 2 * h->N;
    h->DIP = h->E + h->CD + h->H;
    h->DIPP = (h->DIP + 7) / 8 * 8;
    h->R = 0;
    h->RP = 0;
    if (const char* sq = getenv("PCAD_SSD_SEQ")) h->ssd_impl = sq[0] == '1' ? 1 : 0;
  }
  h->V = cfg->vocab_size;
  h->f32 = cfg->dtype == PCAD_F32;
  h->act_size = h->f32 ? 4 : 2;
  h->fuse_norm = !h->f32 && !cfg->residual_in_fp32;
  // dt_proj inside the scan kernel (bf16; x_proj output rows must hold at least 64 columns for the TMA box).
  // Off by default: measured slower on B200 (scan +21 ms, dt_proj -12 ms per step; see scan.cuh).
  h->fuse_dt = false;
  if (const char* fd = getenv("PCAD_FUSED_DT"))
    h->fuse_dt = fd[0] == '1' && !m2 && !h->f32 && h->RP >= kScanDtK && h->R <= kScanDtK && (h->E % 8) == 0;
  if (const char* bq = getenv("PCAD_SCAN_BC_F32")) { h->bc_f32 = bq[0] != '0'; h->bc_f32_force = bq[0] == '1'; }   // A/B switch: 0 off, 1 always
  if (const char* pl = getenv("PCAD_NO_PRUNE")) h->prune_last = pl[0] != '1';
  if (const char* tp = getenv("PCAD_NO_TIME_PARALLEL")) h->time_parallel = tp[0] != '1';
  if (const char* ng = getenv("PCAD_NO_GRAPH")) h->use_graphs = ng[0] != '1';
  if (const char* gm = getenv("PCAD_GRAPH_MAX_TOKENS")) h->graph_max_tokens = atoll(gm);
  if (const char* nf = getenv("PCAD_NO_FUSED_NORM")) { if (nf[0] == '1') h->fuse_norm = false; }   // A/B switch for tests
  memset(h->prof_ms, 0, sizeof(h->prof_ms));
  memset(h->prof_launches, 0, sizeof(h->prof_launches));
  h->layers.resize(cfg->n_layer);
  int rc = PCAD_OK;
  const size_t a = h->act_size;
  auto A8 = [&](void** p, size_t bytes) { uint8_t* q; int r = dev_alloc<uint8_t>(h, &q, bytes); *p = q; return r; };
  rc |= A8(&h->emb, static_cast<size_t>(h->V) * h->d * a);
  rc |= dev_alloc(h, &h->head_w, static_cast<size_t>(h->V) * h->d);
  rc |= dev_alloc(h, &h->norm_f, h->d);
  rc |= dev_alloc(h, &h->comp_dev, 16);
  rc |= dev_alloc(h, &h->lut_dev, 256);
  rc |= dev_alloc(h, &h->sel_dev, 4);
  {
    // zero-copy flag: the id-validation kernels set it, pcad_take_id_error reads it without a device copy
    void* hp = nullptr;
    void* dp = nullptr;
    if (cudaHostAlloc(&hp, sizeof(int), cudaHostAllocMapped) != cudaSuccess || cudaHostGetDevicePointer(&dp, hp, 0) != cudaSuccess) {
      if (hp) cudaFreeHost(hp);
      rc |= fail(h, PCAD_ERR_NOMEM, "cudaHostAlloc for the id-error flag failed");
    } else {
      h->bad_flag_host = static_cast<volatile int*>(hp);
      *h->bad_flag_host = 0;
      h->bad_flag = static_cast<int*>(dp);
    }
  }
  const size_t n_in_rows = m2 ? static_cast<size_t>(h->DIP) : static_cast<size_t>(2) * h->E;
  for (auto& lw : h->layers) {
    rc |= A8(&lw.in_proj, n_in_rows * h->d * a);
    if (h->fuse_norm) rc |= A8(&lw.in_proj_s, n_in_rows * h->d * a);
    rc |= A8(&lw.out_proj, static_cast<size_t>(h->d) * h->E * a);
    rc |= dev_alloc(h, &lw.norm_w, h->d);
    for (int dir = 0; dir < 2; ++dir) {
      DirWeights& dw = lw.dir[dir];
      if (m2) {
        rc |= dev_alloc(h, &dw.conv_w, static_cast<size_t>(h->CD) * 4);
        rc |= dev_alloc(h, &dw.conv_b, h->CD);
        rc |= dev_alloc(h, &dw.dt_bias, h->H);
        rc |= dev_alloc(h, &dw.A, h->H);
        rc |= dev_alloc(h, &dw.D, h->H);
        rc |= dev_alloc(h, &dw.gnorm_w, h->E);
        continue;
      }
      rc |= dev_alloc(h, &dw.conv_w, static_cast<size_t>(h->E) * 4);
      rc |= dev_alloc(h, &dw.conv_b, h->E);
      rc |= A8(&dw.x_proj, static_cast<size_t>(h->RP) * h->E * a);
      rc |= A8(&dw.dt_proj, static_cast<size_t>(h->E) * h->R * a);
      rc |= dev_alloc(h, &dw.dt_bias, h->E);
      rc |= dev_alloc(h, &dw.A, static_cast<size_t>(h->E) * h->N);
      rc |= dev_alloc(h, &dw.D, h->E);
      if (rc == PCAD_OK) cudaMemset(dw.x_proj, 0, static_cast<size_t>(h->RP) * h->E * a);
    }
    if (rc != PCAD_OK) break;
  }
  if (rc != PCAD_OK) {
    snprintf(g_create_error, sizeof(g_create_error), "%.511s", h->err);
    pcad_destroy(h);
    return PCAD_ERR_NOMEM;
  }
  uint8_t comp8[16] = {0};
  for (int i = 0; i < h->V; ++i) comp8[i] = static_cast<uint8_t>(cfg->complement_map[i]);
  cudaMemcpy(h->comp_dev, comp8, 16, cudaMemcpyHostToDevice);
  // default tokenizer tables: [PAD]=0 [MASK]=1 [UNK]=2 a=3 c=4 g=5 t=6, case-folded, everything else UNK
  uint8_t lut[256];
  memset(lut, 2, sizeof(lut));
  lut['a'] = lut['A'] = 3; lut['c'] = lut['C'] = 4; lut['g'] = lut['G'] = 5; lut['t'] = lut['T'] = 6;
  const int32_t acgt[4] = {3, 4, 5, 6};
  *out = h;
  return pcad_set_tokenizer(h, lut, 1, acgt);
}

void pcad_destroy(pcad_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (auto& pe : h->prof_events) { cudaEventDestroy(pe.second.first); cudaEventDestroy(pe.second.second); }
  for (auto ev : h->event_pool) cudaEventDestroy(ev);
  clear_graphs(h);
  if (h->gstream) cudaStreamDestroy(h->gstream);
  if (h->g_in) cudaEventDestroy(h->g_in);
  if (h->g_out) cudaEventDestroy(h->g_out);
  if (h->ws.base) cudaFree(h->ws.base);
  if (h->bad_flag_host) cudaFreeHost(const_cast<int*>(h->bad_flag_host));
  for (void* p : h->allocs) cudaFree(p);
  delete h;
}

int pcad_set_tokenizer(pcad_handle* h, const uint8_t lut[256], int mask_id, const int32_t acgt_ids[4]) {
  if (!h || !lut || !acgt_ids) return PCAD_ERR_INVALID;
  if (mask_id < 0 || mask_id >= h->V) return fail(h, PCAD_ERR_INVALID, "mask_id %d out of range", mask_id);
  for (int i = 0; i < 256; ++i) if (lut[i] >= h->V) return fail(h, PCAD_ERR_INVALID, "lut[%d]=%d out of range", i, lut[i]);
  for (int k = 0; k < 4; ++k) if (acgt_ids[k] < 0 || acgt_ids[k] >= h->V) return fail(h, PCAD_ERR_INVALID, "acgt id out of range");
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaDeviceSynchronize());   // forwards and graph replays still queued on any stream read the old tables
  CUDA_TRY(h, cudaMemcpy(h->lut_dev, lut, 256, cudaMemcpyHostToDevice));
  int sel[4] = {acgt_ids[0], acgt_ids[1], acgt_ids[2], acgt_ids[3]};
  CUDA_TRY(h, cudaMemcpy(h->sel_dev, sel, sizeof(sel), cudaMemcpyHostToDevice));
  h->mask_id = mask_id;
  for (int k = 0; k < 4; ++k) h->acgt[k] = acgt_ids[k];
  clear_graphs(h);   // mask id and column selection are baked into captured launches
  return PCAD_OK;
}

int pcad_set_weight(pcad_handle* h, const char* name, const void* data, const int64_t* shape, int ndim, int src_dtype) {
  if (!h || !name || !data || !shape) return PCAD_ERR_INVALID;
  if (src_dtype != PCAD_BF16 && src_dtype != PCAD_F32 && src_dtype != PCAD_F16) return fail(h, PCAD_ERR_INVALID, "bad src_dtype for %s", name);
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaDeviceSynchronize());   // forwards and graph replays still queued on any stream read the old weights
  h->finalized = false;
  clear_graphs(h);
  const int d = h->d, E = h->E, N = h->N, R = h->R, V = h->V;
  const std::string s(name);
  auto bad_shape = [&]() { return fail(h, PCAD_ERR_INVALID, "unexpected shape for %s", name); };
  if (s == "caduceus.backbone.embeddings.word_embeddings.embedding.weight") {
    if (!shape_is(shape, ndim, {V, d})) return bad_shape();
    int rc = ingest(h, data, src_dtype, h->emb, h->f32, static_cast<long long>(V) * d);
    h->has_emb = rc == PCAD_OK;
    return rc;
  }
  if (s == "lm_head.lm_head.weight") {
    if (!shape_is(shape, ndim, {V, d})) return bad_shape();
    int rc = ingest(h, data, src_dtype, h->head_w, true, static_cast<long long>(V) * d);
    h->head_set = rc == PCAD_OK;
    return rc;
  }
  if (s == "caduceus.backbone.norm_f.weight") {
    if (!shape_is(shape, ndim, {d})) return bad_shape();
    int rc = ingest(h, data, src_dtype, h->norm_f, true, d);
    h->has_norm_f = rc == PCAD_OK;
    return rc;
  }
  const std::string lp = "caduceus.backbone.layers.";
  if (s.compare(0, lp.size(), lp) != 0) return fail(h, PCAD_ERR_INVALID, "unknown weight name %s", name);
  size_t dot = s.find('.', lp.size());
  if (dot == std::string::npos) return fail(h, PCAD_ERR_INVALID, "unknown weight name %s", name);
  const int li = atoi(s.substr(lp.size(), dot - lp.size()).c_str());
  if (li < 0 || li >= h->cfg.n_layer) return fail(h, PCAD_ERR_INVALID, "layer index out of range in %s", name);
  LayerWeights& lw = h->layers[li];
  const std::string rest = s.substr(dot + 1);
  if (rest == "norm.weight") {
    if (!shape_is(shape, ndim, {d})) return bad_shape();
    int rc = ingest(h, data, src_dtype, lw.norm_w, true, d);
    lw.has_norm = rc == PCAD_OK;
    return rc;
  }
  const std::string mp = "mixer.submodule.mamba_";
  if (rest.compare(0, mp.size(), mp) != 0) return fail(h, PCAD_ERR_INVALID, "unknown weight name %s", name);
  int dir;
  if (rest.compare(mp.size(), 4, "fwd.") == 0) dir = 0;
  else if (rest.compare(mp.size(), 4, "rev.") == 0) dir = 1;
  else return fail(h, PCAD_ERR_INVALID, "unknown weight name %s", name);
  const std::string leaf = rest.substr(mp.size() + 4);
  DirWeights& dw = lw.dir[dir];
  int rc;
  const int n_in = h->m2 ? h->DIP : 2 * E;        // in_proj rows
  const int CE = h->m2 ? h->CD : E;               // channels through the conv
  const int NH = h->m2 ? h->H : E;                // Mamba-2: dt_bias / A_log / D are per head
  if (leaf == "in_proj.weight") {
    if (!shape_is(shape, ndim, {n_in, d})) return bad_shape();
    // tied to mamba_fwd (bidirectional_weight_tie); a de-duplicated checkpoint may carry only the mamba_rev name
    if (dir == 1 && lw.has_in) return PCAD_OK;
    rc = ingest(h, data, src_dtype, lw.in_proj, h->f32, static_cast<long long>(n_in) * d);
    lw.has_in = rc == PCAD_OK;
  } else if (leaf == "out_proj.weight") {
    if (!shape_is(shape, ndim, {d, E})) return bad_shape();
    if (dir == 1 && lw.has_out) return PCAD_OK;
    rc = ingest(h, data, src_dtype, lw.out_proj, h->f32, static_cast<long long>(d) * E);
    lw.has_out = rc == PCAD_OK;
  } else if (leaf == "conv1d.weight") {
    if (!shape_is(shape, ndim, {CE, 4})) return bad_shape();
    rc = ingest(h, data, src_dtype, dw.conv_w, true, static_cast<long long>(CE) * 4);
    dw.has[0] = rc == PCAD_OK;
  } else if (leaf == "conv1d.bias") {
    if (!shape_is(shape, ndim, {CE})) return bad_shape();
    rc = ingest(h, data, src_dtype, dw.conv_b, true, CE);
    dw.has[1] = rc == PCAD_OK;
  } else if (leaf == "x_proj.weight" && !h->m2) {
    if (!shape_is(shape, ndim, {R + 2 * N, E})) return bad_shape();
    rc = ingest(h, data, src_dtype, dw.x_proj, h->f32, static_cast<long long>(R + 2 * N) * E);  // rows beyond stay zero
    dw.has[2] = rc == PCAD_OK;
  } else if (leaf == "dt_proj.weight" && !h->m2) {
    if (!shape_is(shape, ndim, {E, R})) return bad_shape();
    rc = ingest(h, data, src_dtype, dw.dt_proj, h->f32, static_cast<long long>(E) * R);
    dw.has[3] = rc == PCAD_OK;
  } else if ((leaf == "dt_proj.bias" && !h->m2) || (leaf == "dt_bias" && h->m2)) {
    if (!shape_is(shape, ndim, {NH})) return bad_shape();
    rc = ingest(h, data, src_dtype, dw.dt_bias, true, NH);
    dw.has[4] = rc == PCAD_OK;
  } else if (leaf == "A_log") {
    const long long n = h->m2 ? NH : static_cast<long long>(E) * N;
    if (h->m2 ? !shape_is(shape, ndim, {NH}) : !shape_is(shape, ndim, {E, N})) return bad_shape();
    rc = ingest(h, data, src_dtype, dw.A, true, n);
    if (rc == PCAD_OK) {
      neg_exp_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(dw.A, n);  // A = -exp(A_log), fp32
      CUDA_TRY(h, cudaDeviceSynchronize());
    }
    dw.has[5] = rc == PCAD_OK;
  } else if (leaf == "D") {
    if (!shape_is(shape, ndim, {NH})) return bad_shape();
    rc = ingest(h, data, src_dtype, dw.D, true, NH);
    dw.has[6] = rc == PCAD_OK;
  } else if (leaf == "norm.weight" && h->m2) {
    if (!shape_is(shape, ndim, {E})) return bad_shape();
    rc = ingest(h, data, src_dtype, dw.gnorm_w, true, E);
    dw.has[7] = rc == PCAD_OK;
  } else {
    return fail(h, PCAD_ERR_INVALID, "unknown weight name %s", name);
  }
  return rc;
}

int pcad_finalize(pcad_handle* h) {
  if (!h) return PCAD_ERR_INVALID;
  if (!h->has_emb) return fail(h, PCAD_ERR_MISSING, "missing weight: embedding");
  if (!h->has_norm_f) return fail(h, PCAD_ERR_MISSING, "missing weight: norm_f");
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaDeviceSynchronize());   // queued forwards read head_w and in_proj_s
  if (!h->head_set) {  // tied LM head (SURVEY.md Appendix A item 7): derive from the (possibly reloaded) embedding
    const long long n = static_cast<long long>(h->V) * h->d;
    if (h->f32) convert_kernel<float, float><<<static_cast<unsigned>((n + 255) / 256), 256>>>(static_cast<const float*>(h->emb), h->head_w, n);
    else convert_kernel<bf16, float><<<static_cast<unsigned>((n + 255) / 256), 256>>>(static_cast<const bf16*>(h->emb), h->head_w, n);
    CUDA_TRY(h, cudaDeviceSynchronize());
  }
  static const char* names1[8] = {"conv1d.weight", "conv1d.bias", "x_proj.weight", "dt_proj.weight", "dt_proj.bias", "A_log", "D", nullptr};
  static const char* names2[8] = {"conv1d.weight", "conv1d.bias", nullptr, nullptr, "dt_bias", "A_log", "D", "norm.weight"};
  const char** names = h->m2 ? names2 : names1;
  for (int li = 0; li < h->cfg.n_layer; ++li) {
    const LayerWeights& lw = h->layers[li];
    if (!lw.has_in) return fail(h, PCAD_ERR_MISSING, "missing weight: layers.%d in_proj.weight", li);
    if (!lw.has_out) return fail(h, PCAD_ERR_MISSING, "missing weight: layers.%d out_proj.weight", li);
    if (!lw.has_norm) return fail(h, PCAD_ERR_MISSING, "missing weight: layers.%d norm.weight", li);
    for (int dir = 0; dir < 2; ++dir)
      for (int k = 0; k < 8; ++k)
        if (names[k] && !lw.dir[dir].has[k]) return fail(h, PCAD_ERR_MISSING, "missing weight: layers.%d mamba_%s.%s", li, dir ? "rev" : "fwd", names[k]);
  }
  if (h->fuse_norm) {
    const long long rows = h->m2 ? h->DIP : 2LL * h->E, n = rows * h->d;
    for (auto& lw : h->layers)
      scale_columns_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(static_cast<const bf16*>(lw.in_proj), lw.norm_w,
                                                                           static_cast<bf16*>(lw.in_proj_s), rows, h->d);
    CUDA_TRY(h, cudaDeviceSynchronize());
  }
  h->finalized = true;
  return PCAD_OK;
}

int pcad_workspace_bytes(pcad_handle* h, int B, int L, size_t* out) {
  if (!h || !out || B < 0 || L < 0) return PCAD_ERR_INVALID;
  *out = workspace_layout(h, B, L, nullptr);
  return PCAD_OK;
}

int pcad_tokenize(pcad_handle* h, const uint8_t* ascii_dev, int64_t n, uint8_t* ids_dev, void* stream) {
  if (!h || (n > 0 && (!ascii_dev || !ids_dev))) return PCAD_ERR_INVALID;
  if (n <= 0) return PCAD_OK;
  CUDA_TRY(h, cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  StageTimer tm(h, st, PCAD_ST_MISC);
  tokenize_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(ascii_dev, ids_dev, n, h->lut_dev, 1, -1, 0);
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

int pcad_extract_windows(pcad_handle* h, const uint8_t* chrom_dev, int64_t chrom_len, const int64_t* pos0_dev, int B, int L,
                         int token_idx, uint8_t* ascii_out_dev, void* stream) {
  if (!h || B < 0 || L <= 0 || chrom_len < 0) return PCAD_ERR_INVALID;
  if (B == 0) return PCAD_OK;
  if (!chrom_dev || !pos0_dev || !ascii_out_dev) return fail(h, PCAD_ERR_INVALID, "null argument");
  if (token_idx < 0 || token_idx >= L) return fail(h, PCAD_ERR_INVALID, "token_idx %d outside [0, %d)", token_idx, L);
  CUDA_TRY(h, cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  StageTimer tm(h, st, PCAD_ST_MISC);
  const long long n = static_cast<long long>(B) * L;
  extract_windows_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(
      chrom_dev, chrom_len, reinterpret_cast<const long long*>(pos0_dev), ascii_out_dev, B, L, token_idx);
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

namespace {
// tokenise + mask (ws.ascii -> ws.ids), backbone, head at token_idx -> ws.logits4; everything on `st`, internal buffers only
int score_core(pcad_handle* h, int B, int L, int token_idx, cudaStream_t st) {
  Workspace& ws = h->ws;
  const long long n = static_cast<long long>(B) * L;
  {
    StageTimer tm(h, st, PCAD_ST_MISC, 3);
    tokenize_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(ws.ascii, ws.ids, n, h->lut_dev, L, token_idx, h->mask_id);
    fill_int_kernel<<<(B + 255) / 256, 256, 0, st>>>(ws.pos, B, token_idx);
    fill_int_kernel<<<(B + 255) / 256, 256, 0, st>>>(ws.pos0, B, 0);
    CUDA_TRY(h, cudaGetLastError());
  }
  return score_at(h, B, L, token_idx, ws.logits4, st);
}

// The same through a CUDA graph when the forward is small enough to be launch-bound.  First call with a shape: eager (also
// sets the kernels' shared-memory attributes, which must not happen inside a capture); second: capture + instantiate;
// then replay.  Profiling (per-stage events) always runs eagerly.
int score_core_graphed(pcad_handle* h, int B, int L, int token_idx, cudaStream_t st) {
  if (!h->use_graphs || h->profiling || 2LL * B * L > h->graph_max_tokens) return score_core(h, B, L, token_idx, st);
  pcad_handle::ScoreGraph* e = nullptr;
  for (auto& g : h->graphs)
    if (g.B == B && g.L == L && g.token_idx == token_idx) { e = &g; break; }
  if (!e) {
    h->graphs.push_back({B, L, token_idx, true, nullptr, 0});
    return score_core(h, B, L, token_idx, st);
  }
  if (!h->gstream) {
    if (cudaStreamCreateWithFlags(&h->gstream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->g_in, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->g_out, cudaEventDisableTiming) != cudaSuccess) {
      h->use_graphs = false;
      cudaGetLastError();
      return score_core(h, B, L, token_idx, st);
    }
  }
  const bool captured_before = !e->seen_only;
  if (e->seen_only) {
    const int64_t before = h->launch_count;
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamBeginCapture(h->gstream, cudaStreamCaptureModeThreadLocal);
    int rc = ce == cudaSuccess ? score_core(h, B, L, token_idx, h->gstream) : PCAD_ERR_CUDA;
    if (ce == cudaSuccess) ce = cudaStreamEndCapture(h->gstream, &graph);
    if (rc == PCAD_OK && ce == cudaSuccess && graph) ce = cudaGraphInstantiate(&e->exec, graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (rc != PCAD_OK || ce != cudaSuccess || !e->exec) {
      e->exec = nullptr;
      h->use_graphs = false;                       // fall back to eager launches for good; this call still has to run
      h->launch_count = before;
      cudaGetLastError();
      return score_core(h, B, L, token_idx, st);
    }
    e->launches = h->launch_count - before;
    h->launch_count = before;
    e->seen_only = false;
  }
  // replay on the capture stream, ordered after / before the caller's stream by events
  CUDA_TRY(h, cudaEventRecord(h->g_in, st));
  CUDA_TRY(h, cudaStreamWaitEvent(h->gstream, h->g_in, 0));
  CUDA_TRY(h, cudaGraphLaunch(e->exec, h->gstream));
  CUDA_TRY(h, cudaEventRecord(h->g_out, h->gstream));
  CUDA_TRY(h, cudaStreamWaitEvent(st, h->g_out, 0));
  h->launch_count += e->launches;
  if (captured_before) ++h->graph_replays;
  return PCAD_OK;
}
}  // namespace

int pcad_score_windows_dev(pcad_handle* h, const uint8_t* ascii_dev, int B, int L, int token_idx, float* logits4_dev, void* stream) {
  int rc = begin_call(h, B, L, 1, ascii_dev && logits4_dev, "null argument", token_idx);
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Workspace& ws = h->ws;
  const size_t n = static_cast<size_t>(B) * L;
  CUDA_TRY(h, cudaMemcpyAsync(ws.ascii, ascii_dev, n, cudaMemcpyDeviceToDevice, st));
  rc = score_core_graphed(h, B, L, token_idx, st);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(logits4_dev, ws.logits4, static_cast<size_t>(B) * 4 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return PCAD_OK;
}

int pcad_forward(pcad_handle* h, const int64_t* ids_dev, int B, int L, float* logits_dev, void* hidden_dev, void* stream) {
  int rc = begin_call(h, B, L, 1, ids_dev, "ids_dev is null");
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = stage_ids64(h, ids_dev, B, L, st);
  if (rc) return rc;
  rc = run_backbone(h, B, L, st);
  if (rc) return rc;
  if (logits_dev) {
    rc = run_head(h, B, L, nullptr, 0, logits_dev, st);
    if (rc) return rc;
  }
  if (hidden_dev) {
    StageTimer tm(h, st, PCAD_ST_MISC);
    const long long total = static_cast<long long>(B) * L * (2 * h->d / 8);
    const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
    if (h->f32) hidden_tap_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(h->ws.normed), static_cast<float*>(hidden_dev), B, L, h->d);
    else hidden_tap_kernel<bf16><<<blocks, 256, 0, st>>>(static_cast<const bf16*>(h->ws.normed), static_cast<bf16*>(hidden_dev), B, L, h->d);
    CUDA_TRY(h, cudaGetLastError());
  }
  return PCAD_OK;
}

int pcad_score_masked(pcad_handle* h, const uint8_t* ids_dev, const int32_t* pos_dev, int B, int L, int n_mask, float* logits4_dev, void* stream) {
  int rc = begin_call(h, B, L, n_mask, ids_dev && pos_dev && logits4_dev && n_mask >= 0, "null or negative argument");
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = stage_ids(h, ids_dev, B, L, -1, st);
  if (rc) return rc;
  rc = run_backbone(h, B, L, st);
  if (rc) return rc;
  return run_head(h, B, L, pos_dev, n_mask, logits4_dev, st);
}

int pcad_score_masked_at(pcad_handle* h, const uint8_t* ids_dev, int token_idx, int B, int L, float* logits4_dev, void* stream) {
  int rc = begin_call(h, B, L, 1, ids_dev && logits4_dev, "null argument", token_idx);
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = stage_ids(h, ids_dev, B, L, token_idx, st);
  if (rc) return rc;
  return score_at(h, B, L, token_idx, logits4_dev, st);
}

int pcad_hidden_at(pcad_handle* h, const uint8_t* ids_dev, const int32_t* pos_dev, int B, int L, int n_pos, void* hidden_dev, void* stream) {
  int rc = begin_call(h, B, L, n_pos, ids_dev && pos_dev && hidden_dev && n_pos >= 0, "null or negative argument");
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = stage_ids(h, ids_dev, B, L, -1, st);
  if (rc) return rc;
  rc = run_backbone(h, B, L, st);
  if (rc) return rc;
  StageTimer tm(h, st, PCAD_ST_MISC);
  const long long total = static_cast<long long>(B) * n_pos * (2 * h->d / 8);
  const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
  if (h->f32) hidden_tap_pos_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(h->ws.normed), pos_dev, n_pos, static_cast<float*>(hidden_dev), B, L, h->d);
  else hidden_tap_pos_kernel<bf16><<<blocks, 256, 0, st>>>(static_cast<const bf16*>(h->ws.normed), pos_dev, n_pos, static_cast<bf16*>(hidden_dev), B, L, h->d);
  CUDA_TRY(h, cudaGetLastError());
  return PCAD_OK;
}

int pcad_forward_taps(pcad_handle* h, const int64_t* ids_dev, int B, int L, float* logits_dev, int n_taps, const int32_t* tap_idx,
                      void* const* tap_dev, void* stream) {
  if (!h) return PCAD_ERR_INVALID;
  int rc = check_taps(h, n_taps, tap_idx);
  if (rc) return rc;
  if (!tap_dev) return fail(h, PCAD_ERR_INVALID, "tap_dev is null");
  for (int i = 0; i < n_taps; ++i)
    if (!tap_dev[i]) return fail(h, PCAD_ERR_INVALID, "tap_dev[%d] is null", i);
  rc = begin_call(h, B, L, 1, ids_dev, "ids_dev is null");
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = stage_ids64(h, ids_dev, B, L, st);
  if (rc) return rc;
  Taps taps;
  taps.n = n_taps;
  taps.idx = tap_idx;
  taps.dst = tap_dev;
  rc = run_backbone(h, B, L, st, -1, &taps, logits_dev != nullptr);
  if (rc || !logits_dev) return rc;
  return run_head(h, B, L, nullptr, 0, logits_dev, st);
}

int pcad_hidden_at_layers(pcad_handle* h, const uint8_t* ids_dev, const int32_t* pos_dev, int B, int L, int n_pos, int n_taps,
                          const int32_t* tap_idx, void* hidden_dev, void* stream) {
  if (!h) return PCAD_ERR_INVALID;
  int rc = check_taps(h, n_taps, tap_idx);
  if (rc) return rc;
  if (!hidden_dev) return fail(h, PCAD_ERR_INVALID, "hidden_dev is null");
  rc = begin_call(h, B, L, n_pos, ids_dev && pos_dev && n_pos >= 0, "null or negative argument");
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = stage_ids(h, ids_dev, B, L, -1, st);
  if (rc) return rc;
  // tap i occupies [B, n_pos, 2d] of hidden_dev, after the i taps before it
  const size_t tap_bytes = static_cast<size_t>(B) * n_pos * 2 * h->d * h->act_size;
  std::vector<void*> dst(n_taps);
  for (int i = 0; i < n_taps; ++i) dst[i] = static_cast<uint8_t*>(hidden_dev) + i * tap_bytes;
  Taps taps;
  taps.n = n_taps;
  taps.idx = tap_idx;
  taps.dst = dst.data();
  taps.pos = pos_dev;
  taps.n_pos = n_pos;
  return run_backbone(h, B, L, st, -1, &taps, false);
}

int pcad_hidden_mean_at_layers(pcad_handle* h, const uint8_t* ids_dev, const int32_t* ranges_dev, int B, int L, int n_taps,
                               const int32_t* tap_idx, float* out_dev, void* stream) {
  if (!h) return PCAD_ERR_INVALID;
  int rc = check_taps(h, n_taps, tap_idx);
  if (rc) return rc;
  if (!out_dev) return fail(h, PCAD_ERR_INVALID, "out_dev is null");
  rc = begin_call(h, B, L, 1, ids_dev != nullptr, "ids_dev is null");
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = stage_ids(h, ids_dev, B, L, -1, st);
  if (rc) return rc;
  Taps taps;
  taps.n = n_taps;
  taps.idx = tap_idx;
  taps.mean = out_dev;
  taps.ranges = ranges_dev;
  return run_backbone(h, B, L, st, -1, &taps, false);
}

int pcad_score_windows_host(pcad_handle* h, const uint8_t* ascii_host, int B, int L, int token_idx, float* logits4_host, void* stream) {
  int rc = begin_call(h, B, L, 1, ascii_host && logits4_host, "null argument", token_idx);
  if (rc) return rc == kNoWork ? PCAD_OK : rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Workspace& ws = h->ws;
  CUDA_TRY(h, cudaMemcpyAsync(ws.ascii, ascii_host, static_cast<size_t>(B) * L, cudaMemcpyHostToDevice, st));
  rc = score_core_graphed(h, B, L, token_idx, st);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(logits4_host, ws.logits4, static_cast<size_t>(B) * 4 * sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return PCAD_OK;
}

int pcad_take_id_error(pcad_handle* h, void* stream, int sync) {
  if (!h) return PCAD_ERR_INVALID;
  if (sync) {
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  }
  if (h->bad_flag_host && *h->bad_flag_host) {
    *h->bad_flag_host = 0;
    return fail(h, PCAD_ERR_INVALID, "token id outside [0, %d) in an earlier pcad_forward / pcad_score_masked call (the row was scored with id 0)", h->V);
  }
  return PCAD_OK;
}

int pcad_set_profiling(pcad_handle* h, int enabled) {
  if (!h) return PCAD_ERR_INVALID;
  for (auto& pe : h->prof_events) { h->event_pool.push_back(pe.second.first); h->event_pool.push_back(pe.second.second); }
  h->prof_events.clear();
  memset(h->prof_ms, 0, sizeof(h->prof_ms));
  memset(h->prof_launches, 0, sizeof(h->prof_launches));
  h->profiling = enabled != 0;
  return PCAD_OK;
}

int pcad_get_profile(pcad_handle* h, float ms[PCAD_ST_COUNT], int64_t launches[PCAD_ST_COUNT]) {
  if (!h || !ms || !launches) return PCAD_ERR_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  for (auto& pe : h->prof_events) {
    CUDA_TRY(h, cudaEventSynchronize(pe.second.second));
    float t = 0.f;
    CUDA_TRY(h, cudaEventElapsedTime(&t, pe.second.first, pe.second.second));
    h->prof_ms[pe.first] += t;
    h->event_pool.push_back(pe.second.first);
    h->event_pool.push_back(pe.second.second);
  }
  h->prof_events.clear();
  for (int i = 0; i < PCAD_ST_COUNT; ++i) { ms[i] = h->prof_ms[i]; launches[i] = h->prof_launches[i]; }
  return PCAD_OK;
}

int64_t pcad_launch_count(const pcad_handle* h) { return h ? h->launch_count : 0; }

int64_t pcad_graph_replays(const pcad_handle* h) { return h ? h->graph_replays : 0; }

int pcad_op_sumsq_parts(int N) { return N > 0 ? gemm_sumsq_parts(N) : 0; }

// ---- single-operator entry points ---------------------------------------------------------------------
static pcad_handle* op_scratch() {
  static pcad_handle scratch;  // only .err and .launch_count are used
  return &scratch;
}
static int op_fail_to_global(int rc) {
  if (rc != PCAD_OK) snprintf(g_create_error, sizeof(g_create_error), "%.511s", op_scratch()->err);
  return rc;
}
static int op_num_sms() {
  int dev = 0, n = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n;
}

int pcad_op_linear(const void* A, const void* W, void* C, int64_t M, int N, int K, int64_t lda, int64_t ldw, int64_t ldc, int dtype, void* stream) {
  if (dtype != PCAD_BF16 && dtype != PCAD_F32) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_linear(op_scratch(), A, W, C, M, N, K, lda, ldw, ldc, dtype == PCAD_F32, op_num_sms(), static_cast<cudaStream_t>(stream)));
}

int pcad_op_linear_residual(const void* A, const void* W, const void* resid_in, void* resid_out, float* sumsq_out, int64_t M, int N, int K,
                            int64_t lda, int64_t ldw, int64_t ld_res, int dtype, void* stream) {
  if (dtype != PCAD_BF16 || !resid_in || !sumsq_out) return PCAD_ERR_INVALID;
  EpiParams ep;
  ep.resid = static_cast<const bf16*>(resid_in);
  ep.ld_res = ld_res;
  ep.sumsq_out = sumsq_out;
  ep.sumsq_parts = gemm_sumsq_parts(N);
  return op_fail_to_global(op_linear(op_scratch(), A, W, resid_out, M, N, K, lda, ldw, ld_res, false, op_num_sms(), static_cast<cudaStream_t>(stream), kEpiResidual, ep));
}

int pcad_op_linear_residual_tap(const void* A, const void* W, const void* resid_in, void* resid_out, float* sumsq_out, void* tap_out,
                                int64_t M, int N, int K, int64_t lda, int64_t ldw, int64_t ld_res, int64_t ld_tap, int dtype, void* stream) {
  if (dtype != PCAD_BF16 || !resid_in || !sumsq_out || !tap_out) return PCAD_ERR_INVALID;
  EpiParams ep;
  ep.resid = static_cast<const bf16*>(resid_in);
  ep.ld_res = ld_res;
  ep.sumsq_out = sumsq_out;
  ep.sumsq_parts = gemm_sumsq_parts(N);
  ep.tap = static_cast<bf16*>(tap_out);
  ep.ld_tap = ld_tap;
  return op_fail_to_global(op_linear(op_scratch(), A, W, resid_out, M, N, K, lda, ldw, ld_res, false, op_num_sms(), static_cast<cudaStream_t>(stream), kEpiResidualTap, ep));
}

int pcad_op_linear_rowscale(const void* A, const void* W, const float* sumsq_in, int sumsq_parts, float eps, void* C, int64_t M, int N, int K,
                            int64_t lda, int64_t ldw, int64_t ldc, int dtype, void* stream) {
  if (dtype != PCAD_BF16 || !sumsq_in || sumsq_parts < 1) return PCAD_ERR_INVALID;
  EpiParams ep;
  ep.sumsq_in = sumsq_in;
  ep.sumsq_parts = sumsq_parts;
  ep.inv_k = 1.0f / static_cast<float>(K);
  ep.eps = eps;
  return op_fail_to_global(op_linear(op_scratch(), A, W, C, M, N, K, lda, ldw, ldc, false, op_num_sms(), static_cast<cudaStream_t>(stream), kEpiRowScale, ep));
}

int pcad_op_biscan_dt(const void* u_f, const void* dbc_f, const void* u_r, const void* dbc_r, int64_t ldbc, int bc_off,
                      const void* wdt_f, const void* wdt_r, int64_t ldw, int R, const void* z, int64_t ldz, const float* A_f,
                      const float* D_f, const float* dt_bias_f, const float* A_r, const float* D_r, const float* dt_bias_r, void* y,
                      int S, int L, int E, void* stream) {
  if (!wdt_f || !wdt_r) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_biscan(op_scratch(), u_f, dbc_f, dbc_f, u_r, dbc_r, dbc_r, ldbc, bc_off, z, ldz, A_f, D_f, dt_bias_f,
                                     A_r, D_r, dt_bias_r, y, S, L, E, false, static_cast<cudaStream_t>(stream), wdt_f, wdt_r, ldw, R));
}

int pcad_op_add_rmsnorm(const void* x, const void* res_in, const float* w, void* y, void* res_out, int64_t rows, int d, float eps, int dtype, int res_dtype, void* stream) {
  if (dtype != PCAD_BF16 && dtype != PCAD_F32) return PCAD_ERR_INVALID;
  if (dtype == PCAD_F32 && res_dtype != PCAD_F32) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_add_rmsnorm(op_scratch(), x, res_in, w, y, res_out, rows, d, eps, dtype == PCAD_F32, res_dtype == PCAD_F32, static_cast<cudaStream_t>(stream)));
}

int pcad_op_conv_silu(const void* x, int64_t ldx, const float* w_f, const float* b_f, const float* w_r, const float* b_r, void* out_f, void* out_r, int S, int L, int E, int dtype, void* stream) {
  if (dtype != PCAD_BF16 && dtype != PCAD_F32) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_conv(op_scratch(), x, ldx, w_f, b_f, w_r, b_r, out_f, out_r, S, L, E, dtype == PCAD_F32, static_cast<cudaStream_t>(stream)));
}

int pcad_op_biscan(const void* u_f, const void* delta_f, const void* bc_f, const void* u_r, const void* delta_r, const void* bc_r,
                   int64_t ldbc, int bc_off, const void* z, int64_t ldz, const float* A_f, const float* D_f, const float* dt_bias_f,
                   const float* A_r, const float* D_r, const float* dt_bias_r, void* y, int S, int L, int E, int dtype, void* stream) {
  if (dtype != PCAD_BF16 && dtype != PCAD_F32) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_biscan(op_scratch(), u_f, delta_f, bc_f, u_r, delta_r, bc_r, ldbc, bc_off, z, ldz, A_f, D_f, dt_bias_f,
                                     A_r, D_r, dt_bias_r, y, S, L, E, dtype == PCAD_F32, static_cast<cudaStream_t>(stream)));
}

int pcad_op_biscan_segmented(const void* u_f, const void* delta_f, const void* bc_f, const void* u_r, const void* delta_r, const void* bc_r,
                             int64_t ldbc, int bc_off, const void* z, int64_t ldz, const float* A_f, const float* D_f, const float* dt_bias_f,
                             const float* A_r, const float* D_r, const float* dt_bias_r, void* y, int S, int L, int E, int segments,
                             float* seg_state, float* seg_sumd, int dtype, void* stream) {
  if (dtype != PCAD_BF16 && dtype != PCAD_F32) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_biscan(op_scratch(), u_f, delta_f, bc_f, u_r, delta_r, bc_r, ldbc, bc_off, z, ldz, A_f, D_f, dt_bias_f,
                                     A_r, D_r, dt_bias_r, y, S, L, E, dtype == PCAD_F32, static_cast<cudaStream_t>(stream), nullptr,
                                     nullptr, 0, 0, segments, seg_state, seg_sumd));
}

int pcad_op_biscan_ex(const void* u_f, const void* delta_f, const void* bc_f, const void* u_r, const void* delta_r, const void* bc_r,
                      int64_t ldbc, int bc_off, const void* z, int64_t ldz, const float* A_f, const float* D_f, const float* dt_bias_f,
                      const float* A_r, const float* D_r, const float* dt_bias_r, void* y, int S, int L, int E, int segments,
                      float* seg_state, float* seg_sumd, float* bc_rows, int Lrun, int dtype, void* stream) {
  if (dtype != PCAD_BF16 && dtype != PCAD_F32) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_biscan(op_scratch(), u_f, delta_f, bc_f, u_r, delta_r, bc_r, ldbc, bc_off, z, ldz, A_f, D_f, dt_bias_f,
                                     A_r, D_r, dt_bias_r, y, S, L, E, dtype == PCAD_F32, static_cast<cudaStream_t>(stream), nullptr,
                                     nullptr, 0, 0, segments < 1 ? 1 : segments, seg_state, seg_sumd, Lrun, bc_rows));
}

int pcad_op_ssd_scan(const void* xbc_f, const void* xbc_r, int64_t ld_xbc, const void* dt_raw, int64_t ld_dt, const float* A_f,
                     const float* D_f, const float* dt_bias_f, const float* A_r, const float* D_r, const float* dt_bias_r, void* y_f,
                     void* y_r, int S, int L, int H, int dtype, int sequential, void* stream) {
  if (dtype != PCAD_BF16 && dtype != PCAD_F32) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_ssd_scan(op_scratch(), xbc_f, xbc_r, ld_xbc, dt_raw, ld_dt, A_f, D_f, dt_bias_f, A_r, D_r, dt_bias_r, y_f,
                                       y_r, S, L, H, dtype == PCAD_F32, sequential, static_cast<cudaStream_t>(stream)));
}

int pcad_op_gated_norm_sum(const void* y_f, const void* y_r, const void* z, int64_t ldz, const float* w_f, const float* w_r, void* out,
                           int64_t rows, int E, float eps, int dtype, void* stream) {
  if (dtype != PCAD_BF16 && dtype != PCAD_F32) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_gated_norm_sum(op_scratch(), y_f, y_r, z, ldz, w_f, w_r, out, rows, E, eps, dtype == PCAD_F32,
                                             static_cast<cudaStream_t>(stream)));
}

int pcad_op_hidden_mean(const void* rows, const int32_t* ranges_dev, float* scratch, float* out, int B, int L, int d, int dtype,
                        void* stream) {
  if ((dtype != PCAD_BF16 && dtype != PCAD_F32) || !rows || !scratch || !out) return PCAD_ERR_INVALID;
  return op_fail_to_global(op_hidden_mean(op_scratch(), rows, ranges_dev, scratch, out, B, L, d, dtype == PCAD_F32,
                                          static_cast<cudaStream_t>(stream)));
}

}  // extern "C"
