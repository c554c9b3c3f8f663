// C[M,N] (bf16) = A[M,K] (bf16, K-major) * W[N,K]^T (bf16, K-major), fp32 accumulation in TMEM.
//
// Persistent, warp-specialised sm_100a kernel:
//   warp 0     : TMA producer (one elected lane) -- cp.async.bulk.tensor 2D tiles, 128B swizzle,
//                STAGES-deep smem ring guarded by full/empty mbarriers
//   warp 1     : TMEM allocator + MMA issuer (one elected lane) -- tcgen05.mma.cta_group::1.kind::f16,
//                128 x BN x 16 per instruction, accumulator double-buffered in TMEM
//   warps 2..5 : epilogue -- tcgen05.ld 32x32b.x32, fp32 -> bf16, 128B-swizzled staging slab per warp in shared
//                memory (double-buffered), written back with cp.async.bulk.tensor (TMA store; M/N tails are
//                clipped by the tensor map)
// This is the F.linear of Mamba.in_proj / x_proj / dt_proj / out_proj ([EXT] mamba_ssm Mamba.forward),
// which the reference runs through cuBLAS.
#pragma once

#include "common.cuh"

namespace pcad {

constexpr int kGemmBM = 128;
constexpr int kGemmBK = 64;  // 64 bf16 = 128 bytes = one swizzle row

// EW = number of epilogue warps: 4 (one per TMEM lane quarter).
// CG = CTAs per tile: 1, or 2 = a CTA pair (cluster of two on one TPC) computing a 256 x BN tile with
// tcgen05.mma.cta_group::2 -- each CTA stages its own 128 rows of A and HALF of the B tile, so a stage is 32 KB
// instead of 48 KB (6 stages instead of 4) and B crosses shared memory once per 256 output rows.
template <int BN, int EW, int CG = 1>
struct GemmCfg {
  static constexpr int kThreads = 64 + 32 * EW;
  static constexpr int kABytes = kGemmBM * kGemmBK * 2;
  static constexpr int kBBytes = (BN / CG) * kGemmBK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  // B tiles must keep 1024-byte alignment inside the ring: pad each B slot to a multiple of 1024.
  static constexpr int kBSlot = (kBBytes + 1023) / 1024 * 1024;
  static constexpr int kSlot = kABytes + kBSlot;
  static constexpr int kStages = (EW == 8) ? 2 : ((BN >= 256 && CG == 1) ? 4 : 6);
  static constexpr int kAccStride = (BN <= 32) ? 32 : (BN <= 64) ? 64 : (BN <= 128) ? 128 : 256;
  static constexpr int kTmemCols = 2 * kAccStride;
  static constexpr int kBarBytes = 256;
  // epilogue staging: EW warps x 2 buffers x (32 rows x 64 bf16 = 4 KB), each slab 1024-byte aligned
  static constexpr int kEpiSlab = 32 * 64 * 2;
  static constexpr int kEpiBytes = EW * 2 * kEpiSlab;
  static constexpr int kSmemBytes = 1024 /*align slack*/ + kStages * kSlot + kEpiBytes + kBarBytes;
};

// Epilogues: kEpiPlain stores the accumulator.
//
// kEpiResidual / kEpiRowScale fold the block's fused residual-add RMSNorm ([EXT] rms_norm_fn(prenorm=True)) into the
// two GEMMs around it, so the bf16 forward has no norm kernel between layers:
//   out_proj, kEpiResidual:  r_new = acc + r_old (fp32), stored as the new residual stream (bf16), and
//                            sumsq[row][part] = sum over this tile's columns of r_new^2 (from the un-rounded fp32 sums,
//                            as the reference's stats); one slot per column tile, plain stores -- no atomics, so the
//                            forward is deterministic and the two strands stay bit-identical;
//   in_proj,  kEpiRowScale:  C = acc * rsqrt(sum_parts sumsq[row][.] / K + eps), with the norm weight pre-multiplied
//                            into the columns of W at load time: (r * rstd * w) W^T == rstd * (r (W diag(w))^T).
//   out_proj, kEpiResidualTap: kEpiResidual, and also tap[row] = bf16(acc), the block's mixer output before the residual
//                            add (the reference's intermediate hidden_states entry).  The same accumulator is rounded once
//                            for the tap and once, after the add, for the residual stream, so the stream and everything
//                            downstream are bit-identical to kEpiResidual's, and the tap to kEpiPlain's.  Each lane stores
//                            its row's 16-byte pieces straight to global memory, next to the residual loads it already
//                            makes: a TMA store would need a second tensor map in the kernel's arguments (changing every
//                            other instantiation) and a second staging slab in shared memory.
enum { kEpiPlain = 0, kEpiResidual = 2, kEpiRowScale = 3, kEpiResidualTap = 4 };

struct EpiParams {
  const bf16* resid = nullptr;        // kEpiResidual: [M, N] with row pitch ld_res (may alias C)
  long long ld_res = 0;
  float* sumsq_out = nullptr;         // kEpiResidual: [M, sumsq_parts]; slot = column-tile index (every slot is written)
  const float* sumsq_in = nullptr;    // kEpiRowScale: [M, sumsq_parts], summed in slot order
  int sumsq_parts = 1;
  float inv_k = 0.f;                  // kEpiRowScale: 1 / (row length the sum of squares was taken over)
  float eps = 0.f;
  bf16* tap = nullptr;                // kEpiResidualTap: [M, N] with row pitch ld_tap, bf16(acc) before the residual add
  long long ld_tap = 0;
};

template <int BN, int EPI, int EW, int CG>
__global__ void __launch_bounds__(GemmCfg<BN, EW, CG>::kThreads, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const __grid_constant__ CUtensorMap tmap_c, long long M, int N, int K, const EpiParams ep) {
  using Cfg = GemmCfg<BN, EW, CG>;
  constexpr int STAGES = Cfg::kStages;
  constexpr bool kResid = EPI == kEpiResidual || EPI == kEpiResidualTap;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;
  uint8_t* epi = smem + STAGES * Cfg::kSlot;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi + Cfg::kEpiBytes);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tiles_n = (N + BN - 1) / BN;
  const long long tiles_m = (M + kGemmBM * CG - 1) / (kGemmBM * CG);   // a tile is (128 * CG) x BN, one per CTA group
  const long long num_tiles = tiles_m * tiles_n;
  const int num_kb = (K + kGemmBK - 1) / kGemmBK;
  const int cta_rank = (CG == 2) ? static_cast<int>(cluster_ctarank()) : 0;   // 0 = leader (issues the MMAs)
  const long long group_id = blockIdx.x / CG, num_groups = gridDim.x / CG;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    tma_prefetch_desc(&tmap_c);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 32 * EW * CG);   // the leader's barrier collects both CTAs' epilogue warps
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (CG == 2) {
      tmem_alloc_cg2<Cfg::kTmemCols>(tmem_ptr);
      tmem_relinquish_cg2();
    } else {
      tmem_alloc<Cfg::kTmemCols>(tmem_ptr);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all();   // barrier inits of both CTAs visible before any remote arrive / TMA
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (long long tile = group_id; tile < num_tiles; tile += num_groups) {
        const int m0 = static_cast<int>(tile / tiles_n) * (kGemmBM * CG) + cta_rank * kGemmBM;   // this CTA's 128 rows
        const int n0 = static_cast<int>(tile % tiles_n) * BN + cta_rank * (BN / CG);             // this CTA's share of B
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* a_dst = ring + stage * Cfg::kSlot;
          uint8_t* b_dst = a_dst + Cfg::kABytes;
          if constexpr (CG == 2) {
            // both CTAs' bytes are credited to the leader's barrier, which alone is armed (with the pair's total)
            if (cta_rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
            tma_load_2d_cg2(a_dst, &tmap_a, &full_bar[stage], kb * kGemmBK, m0);
            tma_load_2d_cg2(b_dst, &tmap_b, &full_bar[stage], kb * kGemmBK, n0);
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes);
            tma_load_2d(a_dst, &tmap_a, &full_bar[stage], kb * kGemmBK, m0);
            tma_load_2d(b_dst, &tmap_b, &full_bar[stage], kb * kGemmBK, n0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (cta_rank == 0 && elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(kGemmBM * CG, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (long long tile = group_id; tile < num_tiles; tile += num_groups) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * Cfg::kAccStride;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(ring + stage * Cfg::kSlot);
          const uint32_t b_addr = a_addr + Cfg::kABytes;
          const uint64_t a_desc = make_smem_desc_sw128(a_addr);
          const uint64_t b_desc = make_smem_desc_sw128(b_addr);
#pragma unroll
          for (int k = 0; k < kGemmBK / 16; ++k) {
            // advance 16 bf16 = 32 bytes along K inside the swizzle row: +2 in 16-byte units
            if constexpr (CG == 2) umma_bf16_ss_cg2(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            else umma_bf16_ss(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          // frees this smem slot (in both CTAs of a pair) once the MMAs above have read it
          if constexpr (CG == 2) umma_commit_cg2(&empty_bar[stage]); else umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        // accumulator complete (each CTA's epilogue waits on its own barrier)
        if constexpr (CG == 2) umma_commit_cg2(&tmem_full[acc]); else umma_commit(&tmem_full[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // epilogue warps 2..(2+EW); TMEM lane quarter is fixed by warp id % 4; with EW = 8 the two warps of a quarter
    // take alternate 64-column chunks
    const int q = warp & 3;
    const int ew = warp - 2;
    constexpr int kChunkStep = 64 * (EW / 4);
    uint8_t* slab = epi + ew * 2 * Cfg::kEpiSlab;
    int buf = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (long long tile = group_id; tile < num_tiles; tile += num_groups) {
      const int m0 = static_cast<int>(tile / tiles_n) * (kGemmBM * CG) + cta_rank * kGemmBM;
      const int n0 = static_cast<int>(tile % tiles_n) * BN;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * Cfg::kAccStride;
      const long long grow = static_cast<long long>(m0) + q * 32 + lane;   // this lane's output row
      const bool row_ok = grow < M;
      float row_scale = 0.f, row_ss = 0.f;
      if constexpr (EPI == kEpiRowScale) {
        float ss = 0.f;
        if (row_ok)
          for (int pp = 0; pp < ep.sumsq_parts; ++pp) ss += ep.sumsq_in[grow * ep.sumsq_parts + pp];
        row_scale = row_ok ? rsqrtf(ss * ep.inv_k + ep.eps) : 0.f;
      }
#pragma unroll 1
      for (int c0 = (ew >> 2) * 64; c0 < BN; c0 += kChunkStep) {
        if (n0 + c0 >= N) break;  // warp-uniform
        uint8_t* dst = slab + buf * Cfg::kEpiSlab;
        // the TMA store that read this buffer two chunks ago must have drained it
        if (lane == 0) tma_store_wait_read<1>();
        __syncwarp();
        uint32_t r0[32], r1[32];
        uint4 res[8];
        if constexpr (kResid) {   // this row's 64 residual values: issued before the TMEM load returns
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int col = n0 + c0 + j * 8;
            res[j] = (row_ok && col + 8 <= N) ? *reinterpret_cast<const uint4*>(ep.resid + grow * ep.ld_res + col)
                                              : make_uint4(0u, 0u, 0u, 0u);
          }
        }
        tmem_ld_32x32b_x32(t_row + c0, r0);
        if (c0 + 32 < BN) tmem_ld_32x32b_x32(t_row + c0 + 32, r1);
        tmem_ld_wait();
        if constexpr (kResid) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            uint32_t* r = (j < 4) ? (r0 + j * 8) : (r1 + (j - 4) * 8);
            const uint32_t w[4] = {res[j].x, res[j].y, res[j].z, res[j].w};
            const bool col_ok = n0 + c0 + j * 8 + 8 <= N;
            if constexpr (EPI == kEpiResidualTap) {
              if (row_ok && col_ok) {
                uint4 t;
                t.x = pack_bf16x2(__uint_as_float(r[0]), __uint_as_float(r[1]));
                t.y = pack_bf16x2(__uint_as_float(r[2]), __uint_as_float(r[3]));
                t.z = pack_bf16x2(__uint_as_float(r[4]), __uint_as_float(r[5]));
                t.w = pack_bf16x2(__uint_as_float(r[6]), __uint_as_float(r[7]));
                *reinterpret_cast<uint4*>(ep.tap + grow * ep.ld_tap + n0 + c0 + j * 8) = t;
              }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float v0 = __uint_as_float(r[2 * k]) + __uint_as_float(w[k] << 16);
              const float v1 = __uint_as_float(r[2 * k + 1]) + __uint_as_float(w[k] & 0xffff0000u);
              r[2 * k] = __float_as_uint(v0);
              r[2 * k + 1] = __float_as_uint(v1);
              if (col_ok) row_ss = fmaf(v0, v0, fmaf(v1, v1, row_ss));
            }
          }
        }
        if constexpr (EPI == kEpiRowScale) {
#pragma unroll
          for (int k = 0; k < 32; ++k) {
            r0[k] = __float_as_uint(__uint_as_float(r0[k]) * row_scale);
            r1[k] = __float_as_uint(__uint_as_float(r1[k]) * row_scale);
          }
        }
        // row `lane` of the slab: 8 chunks of 16 bytes, chunk j stored at (j ^ (lane & 7)) -- the 128B swizzle
        uint8_t* row = dst + lane * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t* r = (j < 4) ? (r0 + j * 8) : (r1 + (j - 4) * 8);
          uint4 v;
          v.x = pack_bf16x2(__uint_as_float(r[0]), __uint_as_float(r[1]));
          v.y = pack_bf16x2(__uint_as_float(r[2]), __uint_as_float(r[3]));
          v.z = pack_bf16x2(__uint_as_float(r[4]), __uint_as_float(r[5]));
          v.w = pack_bf16x2(__uint_as_float(r[6]), __uint_as_float(r[7]));
          *reinterpret_cast<uint4*>(row + ((j ^ (lane & 7)) << 4)) = v;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmap_c, dst, n0 + c0, m0 + q * 32);
          tma_store_commit();
        }
        buf ^= 1;
      }
      tc_fence_before();
      if constexpr (CG == 2) mbar_arrive_leader(&tmem_empty[acc]); else mbar_arrive(&tmem_empty[acc]);
      if constexpr (kResid) {
        static_assert(!kResid || EW == 4, "one sum-of-squares slot per column tile assumes one warp per lane quarter");
        if (row_ok) ep.sumsq_out[grow * ep.sumsq_parts + (n0 / BN)] = row_ss;
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) tma_store_wait_read<0>();
  }

  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all();   // the peer may still be arriving on / reading this CTA's shared memory
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if constexpr (CG == 2) tmem_dealloc_cg2<Cfg::kTmemCols>(tmem_base);
    else tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// 2D bf16 row-major [rows, cols] with row pitch ld (elements); box = [box_rows, 64 cols], 128B swizzle.
// Loads (A, W) zero-fill out-of-range elements; stores (C) clip them.
inline bool make_tmap_bf16(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld,
                           int box_rows) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(kGemmBK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

inline int pick_bn(int N) {
  if (N <= 64) return 64;
  if (N <= 80) return 80;
  if (N <= 96) return 96;
  if (N <= 128) return 128;
  const int waste256 = (N + 255) / 256 * 256 - N;
  const int waste128 = (N + 127) / 128 * 128 - N;
  return waste128 < waste256 ? 128 : 256;
}

// Number of column tiles (= sum-of-squares slots per row) the residual epilogue produces for an N-column output.
inline int gemm_sumsq_parts(int N) {
  const int BN = pick_bn(N);
  return (N + BN - 1) / BN;
}

template <int BN, int EPI, int EW = 4, int CG = 1>
inline cudaError_t launch_gemm_bn(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, long long M, int N,
                                  int K, const EpiParams& ep, int num_sms, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, EW, CG>;
  static unsigned long long attr_done = 0;
  cudaError_t e = ensure_dynamic_smem(gemm_bf16_tcgen05_kernel<BN, EPI, EW, CG>, Cfg::kSmemBytes, attr_done);
  if (e != cudaSuccess) return e;
  const long long tiles = ((M + kGemmBM * CG - 1) / (kGemmBM * CG)) * ((N + BN - 1) / BN);
  const long long groups = num_sms / CG;
  const int grid = static_cast<int>(tiles < groups ? tiles : groups) * CG;
  if constexpr (CG == 1) {
    gemm_bf16_tcgen05_kernel<BN, EPI, EW, 1><<<grid, Cfg::kThreads, Cfg::kSmemBytes, stream>>>(ta, tb, tc, M, N, K, ep);
    return cudaGetLastError();
  } else {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(Cfg::kThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, gemm_bf16_tcgen05_kernel<BN, EPI, EW, CG>, ta, tb, tc, M, N, K, ep);
  }
}

// Returns cudaSuccess or an error; *why is set for non-CUDA failures.  `epi` selects the epilogue (EpiParams).
// cta_pair: use the 2-CTA (cta_group::2) kernel when the shape allows it (N a multiple of 256, K >= 256).
inline cudaError_t gemm_bf16_tcgen05(const bf16* A, const bf16* W, bf16* C, long long M, int N, int K, long long lda,
                                     long long ldw, long long ldc, int num_sms, cudaStream_t stream,
                                     const char** why, int epi = kEpiPlain, const EpiParams& ep = EpiParams(),
                                     bool cta_pair = false) {
  *why = nullptr;
  if (M <= 0 || N <= 0 || K <= 0) return cudaSuccess;
  if ((lda % 8) || (ldw % 8) || (ldc % 8) || (reinterpret_cast<uintptr_t>(A) & 15) ||
      (reinterpret_cast<uintptr_t>(W) & 15) || (reinterpret_cast<uintptr_t>(C) & 15)) {
    *why = "gemm: pointers must be 16-byte aligned and row pitches multiples of 8 elements";
    return cudaErrorInvalidValue;
  }
  const bool resid_epi = epi == kEpiResidual || epi == kEpiResidualTap;
  if (resid_epi && (!ep.resid || !ep.sumsq_out || (N % 8) || (ep.ld_res % 8) ||
                    (reinterpret_cast<uintptr_t>(ep.resid) & 15))) {
    *why = "gemm: the residual epilogue needs resid (16-byte aligned, pitch % 8 == 0), sumsq_out and N % 8 == 0";
    return cudaErrorInvalidValue;
  }
  if (epi == kEpiResidualTap && (!ep.tap || (ep.ld_tap % 8) || ep.ld_tap < N || (reinterpret_cast<uintptr_t>(ep.tap) & 15))) {
    *why = "gemm: the residual tap epilogue needs tap (16-byte aligned, pitch % 8 == 0 and >= N)";
    return cudaErrorInvalidValue;
  }
  if (resid_epi && ep.sumsq_parts != gemm_sumsq_parts(N)) {
    *why = "gemm: sumsq_parts must equal gemm_sumsq_parts(N)";
    return cudaErrorInvalidValue;
  }
  if (epi == kEpiRowScale && !ep.sumsq_in) {
    *why = "gemm: the row-scale epilogue needs sumsq_in";
    return cudaErrorInvalidValue;
  }
  const int BN = pick_bn(N);
  const bool pair = cta_pair && BN == 256 && (N % 256) == 0 && K >= 256 && num_sms >= 2;
  CUtensorMap ta, tb, tc;
  if (!make_tmap_bf16(&ta, A, M, K, lda, kGemmBM) || !make_tmap_bf16(&tb, W, N, K, ldw, pair ? BN / 2 : BN) ||
      !make_tmap_bf16(&tc, C, M, N, ldc, 32)) {
    *why = "gemm: cuTensorMapEncodeTiled failed";
    return cudaErrorInvalidValue;
  }
  if (pair) {
    switch (epi) {
      case kEpiResidual: return launch_gemm_bn<256, kEpiResidual, 4, 2>(ta, tb, tc, M, N, K, ep, num_sms, stream);
      case kEpiResidualTap: return launch_gemm_bn<256, kEpiResidualTap, 4, 2>(ta, tb, tc, M, N, K, ep, num_sms, stream);
      case kEpiRowScale: return launch_gemm_bn<256, kEpiRowScale, 4, 2>(ta, tb, tc, M, N, K, ep, num_sms, stream);
      default: return launch_gemm_bn<256, kEpiPlain, 4, 2>(ta, tb, tc, M, N, K, ep, num_sms, stream);
    }
  }
#define PCAD_GEMM_EPI(BNV)                                                                                  \
  switch (epi) {                                                                                            \
    case kEpiResidual: return launch_gemm_bn<BNV, kEpiResidual>(ta, tb, tc, M, N, K, ep, num_sms, stream);  \
    case kEpiResidualTap: return launch_gemm_bn<BNV, kEpiResidualTap>(ta, tb, tc, M, N, K, ep, num_sms, stream); \
    case kEpiRowScale: return launch_gemm_bn<BNV, kEpiRowScale>(ta, tb, tc, M, N, K, ep, num_sms, stream);  \
    default: return launch_gemm_bn<BNV, kEpiPlain>(ta, tb, tc, M, N, K, ep, num_sms, stream);               \
  }
  switch (BN) {
    case 64: PCAD_GEMM_EPI(64)
    case 80: PCAD_GEMM_EPI(80)
    case 96: PCAD_GEMM_EPI(96)
    case 128: PCAD_GEMM_EPI(128)
    default: PCAD_GEMM_EPI(256)
  }
#undef PCAD_GEMM_EPI
}

}  // namespace pcad
