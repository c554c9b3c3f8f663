/*
 * pcad.h -- C ABI of libpcad.so, the B200 (sm_100a) engine for the PlantCaduceus
 * (Caduceus / reverse-complement-equivariant BiMamba; Mamba-1 mixer for PlantCAD, Mamba-2 / SSD mixer for PlantCAD2)
 * masked-LM forward pass and its zero-shot variant-scoring path.
 *
 * The reference has no C/FFI boundary of its own: the boundary is the Hugging Face Python object
 * returned by AutoModelForMaskedLM.from_pretrained(..., trust_remote_code=True)
 * (reference src/zero_shot_score.py:91) and called as model(input_ids=...) (same file :115).
 * Each entry point below names the reference interface it replaces.  The Python shim in
 * plantcaduceus_b200/modeling.py binds these with ctypes; see INTEGRATION.md for the binding a
 * maintainer of the reference would add.
 *
 * Conventions: every function returns 0 on success or a negative pcad_status; nothing calls
 * exit()/abort() (contrast reference src/zero_shot_score.py:208-212).  All tensors are caller-owned
 * unless stated; device work is enqueued on the given CUDA stream (a cudaStream_t passed as void*,
 * NULL = legacy default stream) and is asynchronous unless the function name ends in _host.
 * One handle per device; a handle is not thread-safe; distinct handles are independent.
 * There is no CPU fallback: without a CUDA device pcad_create fails with PCAD_ERR_CUDA.
 */
#ifndef PCAD_H_
#define PCAD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCAD_ABI_VERSION 3

typedef enum {
  PCAD_OK = 0,
  PCAD_ERR_INVALID = -1,     /* bad argument / unsupported configuration */
  PCAD_ERR_CUDA = -2,        /* CUDA runtime or driver error (see pcad_last_error) */
  PCAD_ERR_STATE = -3,       /* call order violated (e.g. forward before finalize) */
  PCAD_ERR_MISSING = -4,     /* a required weight was never set */
  PCAD_ERR_NOMEM = -5
} pcad_status;

typedef enum { PCAD_BF16 = 0, PCAD_F32 = 1, PCAD_F16 = 2 } pcad_dtype;
/* ssm_cfg["layer"] of the checkpoint's config: "Mamba1" (PlantCaduceus_l20..l32) or "Mamba2" (PlantCAD2,
 * reference docs/PlantCAD2-overview.md:17-21, src/zero-shot-eval.py:54-72). */
typedef enum { PCAD_MIXER_MAMBA1 = 0, PCAD_MIXER_MAMBA2 = 1 } pcad_mixer;

/* Mirrors the keys of the checkpoint's config.json that the forward pass reads
 * (CaduceusConfig; SURVEY.md section 5).  complement_map[i] is the token id of the complement
 * of token i (reference pretrain/llmlib/architectures/models/mamba/caduceus.py:100-105). */
typedef struct {
  int32_t d_model;
  int32_t n_layer;
  int32_t vocab_size;        /* padded to a multiple of 8 (caduceus.py:124-125); engine requires 8 */
  int32_t d_state;           /* 16 (Mamba-1) / 64 (Mamba-2) */
  int32_t d_conv;            /* 4  */
  int32_t expand;            /* 2  */
  int32_t dt_rank;           /* ceil(d_model / 16); ignored for Mamba-2 */
  float   norm_eps;
  int32_t residual_in_fp32;
  int32_t dtype;             /* pcad_dtype of activations and GEMM operands: PCAD_BF16 or PCAD_F32 */
  int32_t complement_map[16];
  int32_t mixer;             /* pcad_mixer */
  int32_t headdim;           /* Mamba-2: 64 */
  int32_t ngroups;           /* Mamba-2: 1 */
} pcad_config;

typedef struct pcad_handle pcad_handle;

/* Replaces: AutoModelForMaskedLM.from_pretrained(...).to(device)  (zero_shot_score.py:91,97).
 * Validates the configuration; unsupported combinations fail here. */
int pcad_create(const pcad_config* cfg, int device, pcad_handle** out);
void pcad_destroy(pcad_handle* h);
const char* pcad_last_error(const pcad_handle* h);   /* h may be NULL: returns the last create error */
int pcad_abi_version(void);

/* Replaces: load_state_dict.  `name` is the checkpoint key (see plantcaduceus_b200/weights.py);
 * `data` may be a host or device pointer (unified addressing); src_dtype is a pcad_dtype.
 * The engine copies and re-lays-out; the caller keeps ownership. mamba_rev.{in,out}_proj alias
 * mamba_fwd's and are accepted and ignored.
 * A live handle may be reloaded: set_weight un-finalizes it and drops its CUDA graphs.  pcad_set_weight,
 * pcad_finalize and pcad_set_tokenizer are load-time calls: each first synchronises the handle's device, so work
 * already enqueued on any stream (forwards, graph replays) completes with the weights and tables it was enqueued with. */
int pcad_set_weight(pcad_handle* h, const char* name, const void* data,
                    const int64_t* shape, int ndim, int src_dtype);
/* Checks every weight is present, derives A = -exp(A_log) etc.  Must precede any forward.  Without
 * lm_head.lm_head.weight the LM head is tied: every finalize derives it from the embedding as it then is (a reloaded
 * embedding moves the head with it); once lm_head.lm_head.weight has been set on this handle, that is the head. */
int pcad_finalize(pcad_handle* h);

/* Tokeniser tables (replaces tokenizer.get_vocab() / mask_token_id, zero_shot_score.py:57,118):
 * lut[c] = token id of ASCII byte c (case already folded by the caller's table);
 * acgt_ids = ids of 'a','c','g','t'. */
int pcad_set_tokenizer(pcad_handle* h, const uint8_t lut[256], int mask_id, const int32_t acgt_ids[4]);

/* Replaces: model(input_ids=ids[, output_hidden_states=True])  (zero_shot_score.py:115,
 * train_XGBoost.py:104).  ids_dev: int64 [B, L] on the device.  logits_dev: float32 [B, L, V] or
 * NULL.  hidden_dev: [B, L, 2*d_model] in the model dtype (final normed hidden state,
 * hidden_states[-1]) or NULL. */
int pcad_forward(pcad_handle* h, const int64_t* ids_dev, int B, int L,
                 float* logits_dev, void* hidden_dev, void* stream);

/* Replaces: extract_logits' model call + logits[:, tokenIdx, [a,c,g,t]] (zero_shot_score.py:112-118)
 * and _masked_probs' gather (zero-shot-eval.py:129-140).  ids_dev: uint8 token ids [B, L], already
 * masked.  pos_dev: int32 [B, n_mask] positions whose logits are wanted.  Output float32
 * [B, n_mask, 4] in a,c,g,t order (raw logits; softmax / log-ratio are the caller's). */
int pcad_score_masked(pcad_handle* h, const uint8_t* ids_dev, const int32_t* pos_dev,
                      int B, int L, int n_mask, float* logits4_dev, void* stream);

/* pcad_score_masked for the reference's own case -- ONE scored position, the same index in every window
 * (extract_logits: logits[:, tokenIdx, [a,c,g,t]], zero_shot_score.py:117-118).  Knowing the position on the host lets the engine
 * compute the last layer only as far as the head needs it.  Output float32 [B, 4], bit-identical to pcad_score_masked. */
int pcad_score_masked_at(pcad_handle* h, const uint8_t* ids_dev, int token_idx, int B, int L,
                         float* logits4_dev, void* stream);

/* Replaces: model(input_ids, output_hidden_states=True).hidden_states[-1][:, tokenIdx, :]  (extract_embeddings,
 * train_XGBoost.py:104-105) without materialising [B, L, 2*d_model]: ids_dev uint8 [B, L] (masked or not, as the caller
 * wants), pos_dev int32 [B, n_pos]; hidden_dev receives [B, n_pos, 2*d_model] in the model dtype (forward half, then the
 * RC half with its channels in the reference's order -- the caller's `reverse[..., ::-1]` average applies as is). */
int pcad_hidden_at(pcad_handle* h, const uint8_t* ids_dev, const int32_t* pos_dev, int B, int L, int n_pos,
                   void* hidden_dev, void* stream);

/* Intermediate hidden states.  Replaces: model(input_ids, output_hidden_states=True).hidden_states[k], which has
 * n_layer + 1 entries, each [B, L, 2*d_model] in the model dtype and in the layout of pcad_forward's hidden_dev (forward
 * half, then the RC half with sequence and channels reversed back):
 *   k = 0                the RCPS embedding;
 *   k in [1, n_layer)    layer k-1's mixer output: out_proj's result before the residual add, the tensor layer k receives;
 *   k = n_layer          the final normed state (pcad_forward's hidden_dev).
 * tap_idx: n_taps host int32 indices, strictly increasing, in [0, n_layer]; tap_dev: host array of n_taps device pointers,
 * tap i receives hidden_states[tap_idx[i]].  The ids are checked as pcad_forward checks them.  Taps change no other output
 * bit: logits and every tap equal those of a call that requests any other set of taps, or none.  With logits_dev NULL the
 * forward stops after the layer that produces the deepest requested entry (about k / n_layer of the full cost) and runs
 * the final norm only if n_layer is requested.  Each tap is a caller buffer of B * L * 2 * d_model elements: with all
 * 33 entries of PlantCaduceus_l32 (d_model 1024, bf16) at B = 256, L = 512 that is 33 x 0.54 GB = 17.7 GB.
 * Returns PCAD_ERR_INVALID, before launching anything, for n_taps outside [1, n_layer + 1], an index outside
 * [0, n_layer], indices not strictly increasing, or a null tap pointer.  Never uses a CUDA graph. */
int pcad_forward_taps(pcad_handle* h, const int64_t* ids_dev, int B, int L, float* logits_dev, int n_taps,
                      const int32_t* tap_idx, void* const* tap_dev, void* stream);

/* Replaces: hidden_states[k][:, tokenIdx, :] for the n_taps indices tap_idx (as pcad_forward_taps) without [B, L, 2*d_model]
 * buffers: ids_dev uint8 [B, L], pos_dev int32 [B, n_pos]; hidden_dev receives [n_taps, B, n_pos, 2*d_model] in the model
 * dtype, bit-identical to the matching slices of pcad_forward_taps.  Always stops at the deepest requested entry.  Same
 * argument checks as pcad_forward_taps (hidden_dev is the tap pointer). */
int pcad_hidden_at_layers(pcad_handle* h, const uint8_t* ids_dev, const int32_t* pos_dev, int B, int L, int n_pos,
                          int n_taps, const int32_t* tap_idx, void* hidden_dev, void* stream);

/* Mean-pooled hidden states: one vector per window and per entry, the input of frozen-embedding classifiers and layer-wise
 * probes.  For uint8 ids_dev [B, L], the n_taps indices tap_idx (as pcad_forward_taps) and per-window ranges [s_b, e_b):
 *   out_dev[i, b, :] = mean over t in [s_b, e_b) of hidden_states[tap_idx[i]][b, t, :]        float32 [n_taps, B, 2*d_model]
 * in the layout of hidden_states (forward half, then the RC half with its channels in the reference's order, so the
 * caller's strand average applies as is).  ranges_dev: int32 [B, 2] on the device, (s_b, e_b) per window; NULL means
 * [0, L) for every window.  A window whose range is invalid (s < 0, e > L or s >= e) gets a NaN row; the other rows are
 * unaffected, and nothing waits on the host.  The states inside a range still see every position of the window, padding
 * included, through the bidirectional scans, as they do in the reference: a range selects what is averaged, not what the
 * model reads.
 * Summation order, fixed: entries are read in the model dtype and summed in fp32, positions in reference order
 * t = s, s+1, ...; sequentially within chunks of PCAD_HIDDEN_MEAN_CHUNK consecutive positions counted from s; the chunk
 * partials then sequentially in chunk order; the total divided by (float)(e - s) with a correctly rounded division.  So a
 * window's result depends neither on B, nor on the other windows, nor on which other entries are requested; it is
 * bit-identical run to run, and no atomics are used.  A one-position range (e = s + 1) equals pcad_hidden_at_layers at s
 * converted to fp32.
 * The entries are read once, in the engine's own workspace, as each comes into existence; the only caller buffer is the
 * result.  All 33 entries of PlantCaduceus_l32 at B = 256, L = 512 are 17.7 GB as pcad_forward_taps buffers and 69 MB
 * pooled; all 49 of PlantCAD2-Large at B = 16, L = 8192 are 39.5 GB and 9.6 MB.  The workspace is that of any forward
 * (pcad_workspace_bytes does not change).  Always stops at the deepest requested entry; never uses a CUDA graph.  Same
 * argument checks as pcad_forward_taps, and PCAD_ERR_INVALID for a null out_dev, all before launching anything.  With
 * B = 0 or L = 0 nothing is written. */
#define PCAD_HIDDEN_MEAN_CHUNK 128
int pcad_hidden_mean_at_layers(pcad_handle* h, const uint8_t* ids_dev, const int32_t* ranges_dev, int B, int L,
                               int n_taps, const int32_t* tap_idx, float* out_dev, void* stream);

/* Token ids outside [0, vocab_size) (the reference's nn.Embedding would raise) are detected on the device by
 * pcad_forward / pcad_score_masked: the offending position is scored as id 0 and a flag is raised in mapped host
 * memory.  pcad_take_id_error returns PCAD_ERR_INVALID and clears the flag if any call since the last take saw such an
 * id, PCAD_OK otherwise; sync != 0 synchronises `stream` first, so the answer covers every call enqueued on it. */
int pcad_take_id_error(pcad_handle* h, void* stream, int sync);

/* End-to-end host entry (SequenceDataset.__getitem__ + extract_logits, zero_shot_score.py:49-62,
 * 107-121): ascii_host = B windows of L ASCII bases (pinned memory recommended); position token_idx
 * of every window is masked; logits4_host receives float32 [B, 4] (a,c,g,t).  Copies H2D, tokenises
 * and masks on the device, runs the forward, copies D2H and synchronises the stream. */
int pcad_score_windows_host(pcad_handle* h, const uint8_t* ascii_host, int B, int L, int token_idx,
                            float* logits4_host, void* stream);

/* Window extraction on the device (seq_from_vcf's slice-and-pad rule, zero_shot_score.py:185-198), for genome-scale
 * runs where the chromosome is resident in HBM: chrom_dev = chrom_len ASCII bases, pos0_dev = int64 [B] 0-based variant
 * positions; ascii_out_dev receives uint8 [B, L] upper-cased windows with the variant at index token_idx, padded with
 * 'N' exactly as the reference pads (right-justified at the chromosome start, left-justified otherwise). */
int pcad_extract_windows(pcad_handle* h, const uint8_t* chrom_dev, int64_t chrom_len, const int64_t* pos0_dev,
                         int B, int L, int token_idx, uint8_t* ascii_out_dev, void* stream);

/* pcad_score_windows_host with device buffers: ascii_dev uint8 [B, L] (e.g. from pcad_extract_windows) ->
 * logits4_dev float32 [B, 4]; tokenise + mask + forward + head on the stream, no copies, no synchronisation. */
int pcad_score_windows_dev(pcad_handle* h, const uint8_t* ascii_dev, int B, int L, int token_idx,
                           float* logits4_dev, void* stream);

/* Device tokeniser on its own (bit-exact with the host LUT): ascii_dev [n] -> ids_dev uint8 [n]. */
int pcad_tokenize(pcad_handle* h, const uint8_t* ascii_dev, int64_t n, uint8_t* ids_dev, void* stream);

/* Bytes of device workspace the engine holds for a (B, L) call (activations, scratch). */
int pcad_workspace_bytes(pcad_handle* h, int B, int L, size_t* out);

/* Per-stage device timing (CUDA events on the launch stream), for bench.py's roofline block.
 * Stage ids are pcad_stage.  pcad_get_profile synchronises the recorded events and returns the
 * accumulated milliseconds and launch counts since the last pcad_set_profiling(h, 1). */
typedef enum {
  PCAD_ST_EMBED = 0, PCAD_ST_NORM, PCAD_ST_IN_PROJ, PCAD_ST_CONV, PCAD_ST_X_PROJ, PCAD_ST_DT_PROJ,
  PCAD_ST_SCAN, PCAD_ST_OUT_PROJ, PCAD_ST_HEAD, PCAD_ST_MISC, PCAD_ST_GNORM /* Mamba-2 gated norms + add */, PCAD_ST_COUNT
} pcad_stage;
int pcad_set_profiling(pcad_handle* h, int enabled);
int pcad_get_profile(pcad_handle* h, float ms[PCAD_ST_COUNT], int64_t launches[PCAD_ST_COUNT]);
/* Total kernels launched by this handle since creation. */
int64_t pcad_launch_count(const pcad_handle* h);
/* Score calls (pcad_score_windows_host / _dev) since creation that replayed a CUDA graph captured by an earlier call. */
int64_t pcad_graph_replays(const pcad_handle* h);

/* ---- single-operator entry points (device pointers; used by the parity tests and profiling) ----
 * All shapes are row-major, "token-major": activations are [rows, channels]. dtype is a pcad_dtype
 * (PCAD_BF16 or PCAD_F32) shared by all activation operands of the call. */

/* C[M,N] = A[M,K] * W[N,K]^T, fp32 accumulate.  lda/ldw/ldc are row pitches in elements.
 * bf16: tcgen05/TMEM GEMM fed by TMA.  f32: SIMT fp32 kernel (parity mode only).
 * Replaces F.linear in Mamba.in_proj / x_proj / dt_proj / out_proj [mamba_ssm Mamba.forward]. */
int pcad_op_linear(const void* A, const void* W, void* C, int64_t M, int N, int K,
                   int64_t lda, int64_t ldw, int64_t ldc, int dtype, void* stream);

/* The block's fused residual add + RMSNorm [mamba_ssm rms_norm_fn(prenorm=True)] folded into the two GEMMs around
 * it (bf16 only; what the bf16 forward runs when residual_in_fp32 = 0):
 *   pcad_op_linear_residual:  resid_out = A W^T + resid_in  (fp32 sum, stored bf16; resid_out may alias resid_in),
 *                             sumsq_out[row][p] = sum over column tile p of (fp32 sum)^2; float [M, pcad_op_sumsq_parts(N)],
 *                             every slot is written with a plain store (no atomics: results are deterministic)
 *   pcad_op_linear_residual_tap: pcad_op_linear_residual, and also tap_out = bf16(A W^T) (row pitch ld_tap, 16-byte
 *                             aligned, not aliasing the other operands), the sum before the residual add; tap_out equals
 *                             pcad_op_linear's C and resid_out / sumsq_out equal pcad_op_linear_residual's, bit for bit
 *   pcad_op_linear_rowscale:  C = (A W^T) * rsqrt(sum_p sumsq_in[row][p] / K + eps)   -- RMSNorm of A's rows applied
 *                             after the GEMM; the norm weight must be pre-multiplied into W's columns by the caller. */
int pcad_op_sumsq_parts(int N);
int pcad_op_linear_residual(const void* A, const void* W, const void* resid_in, void* resid_out, float* sumsq_out,
                            int64_t M, int N, int K, int64_t lda, int64_t ldw, int64_t ld_res, int dtype, void* stream);
int pcad_op_linear_residual_tap(const void* A, const void* W, const void* resid_in, void* resid_out, float* sumsq_out,
                                void* tap_out, int64_t M, int N, int K, int64_t lda, int64_t ldw, int64_t ld_res,
                                int64_t ld_tap, int dtype, void* stream);
int pcad_op_linear_rowscale(const void* A, const void* W, const float* sumsq_in, int sumsq_parts, float eps, void* C,
                            int64_t M, int N, int K, int64_t lda, int64_t ldw, int64_t ldc, int dtype, void* stream);

/* Fused residual add + RMSNorm [mamba_ssm rms_norm_fn, prenorm=True]:
 * res_out = x + res_in (res_in may be NULL); y = res_out * rsqrt(mean(res_out^2) + eps) * w.
 * res_dtype is the storage type of res_in/res_out (PCAD_F32 iff residual_in_fp32).  res_out may be
 * NULL (prenorm=False). */
int pcad_op_add_rmsnorm(const void* x, const void* res_in, const float* w, void* y, void* res_out,
                        int64_t rows, int d, float eps, int dtype, int res_dtype, void* stream);

/* Depthwise causal conv (k=4) + SiLU for both scan directions from one read of x
 * [causal_conv1d_fn, activation="silu"]: x is [S*L, E] with row pitch ldx; out_f uses taps
 * t-3..t with (w_f, b_f); out_r is the same operator applied to the time-reversed sequence,
 * written back at the original position (taps t..t+3).  w_*: float [E, 4], b_*: float [E]. */
int pcad_op_conv_silu(const void* x, int64_t ldx, const float* w_f, const float* b_f,
                      const float* w_r, const float* b_r, void* out_f, void* out_r,
                      int S, int L, int E, int dtype, void* stream);

/* Bidirectional selective scan with softplus(delta + bias), D skip and SiLU(z) gate
 * [selective_scan_fn(..., delta_softplus=True)], both directions summed before the gate
 * [BiMambaWrapper, strategy "add"]:
 *   u_*, delta_*: [S*L, E];  bc_*: [S*L, ldbc] with B at columns [bc_off, bc_off+16) and C at
 *   [bc_off+16, bc_off+32);  z: [S*L, E] with row pitch ldz;  A_*: float [E, 16] (= -exp(A_log));
 *   D_*, dt_bias_*: float [E];  y: [S*L, E].  delta_* are raw dt_proj outputs: the kernel applies
 *   softplus(delta + dt_bias) itself (the reference's order of operations). */
int pcad_op_biscan(const void* u_f, const void* delta_f, const void* bc_f,
                   const void* u_r, const void* delta_r, const void* bc_r,
                   int64_t ldbc, int bc_off, const void* z, int64_t ldz,
                   const float* A_f, const float* D_f, const float* dt_bias_f,
                   const float* A_r, const float* D_r, const float* dt_bias_r,
                   void* y, int S, int L, int E, int dtype, void* stream);

/* pcad_op_biscan as a TIME-PARALLEL scan (low batch / long context): every sequence is cut into `segments` pieces of
 * L / segments positions (L % segments == 0, segments >= 2) that are scanned concurrently -- each from a zero state to get
 * its end state, the end states combined in scan order into every segment's start state, then the segments scanned again from
 * those states.  Exact up to fp32 rounding of the carry.  seg_state: float [S * segments * 2 * E * 16] scratch, seg_sumd: float
 * [S * segments * 2 * E] scratch.  The forward selects this by itself when E / 64 * S CTAs would leave the GPU mostly idle. */
int pcad_op_biscan_segmented(const void* u_f, const void* delta_f, const void* bc_f,
                             const void* u_r, const void* delta_r, const void* bc_r,
                             int64_t ldbc, int bc_off, const void* z, int64_t ldz,
                             const float* A_f, const float* D_f, const float* dt_bias_f,
                             const float* A_r, const float* D_r, const float* dt_bias_r,
                             void* y, int S, int L, int E, int segments, float* seg_state, float* seg_sumd,
                             int dtype, void* stream);

/* pcad_op_biscan with the scan modes the forward picks for itself, for testing them one operator at a time (the forward
 * runs the same host function):
 *   segments <= 1:  the sequential scan.  segments >= 2: time-parallel, as pcad_op_biscan_segmented (same scratch).
 *   bc_rows NULL:   B|C are converted to fp32 inside the scan kernel.  Otherwise (bf16 only) float [2][S*L][32] scratch:
 *                   rows [B ln 2 | C] of the forward direction, then of the reverse direction, written by a conversion
 *                   kernel before the scan, which then reads them by TMA.  What the bf16 forward runs at S*L >= 65536.
 *   Lrun 0 or L:    every row of y holds its final value.  (L+1)/2 <= Lrun < L (sequential only): each direction stops
 *                   after Lrun steps, as the forward's score-only last layer does; only rows [L-Lrun, Lrun) of every
 *                   sequence hold final values, the other rows hold one direction's parked partial.
 * Returns PCAD_ERR_INVALID, before launching anything, for bc_rows with fp32, Lrun < 0, Lrun > L, 0 < Lrun < (L+1)/2
 * (some rows would be visited by neither direction), and Lrun < L with segments >= 2. */
int pcad_op_biscan_ex(const void* u_f, const void* delta_f, const void* bc_f,
                      const void* u_r, const void* delta_r, const void* bc_r,
                      int64_t ldbc, int bc_off, const void* z, int64_t ldz,
                      const float* A_f, const float* D_f, const float* dt_bias_f,
                      const float* A_r, const float* D_r, const float* dt_bias_r,
                      void* y, int S, int L, int E, int segments, float* seg_state, float* seg_sumd,
                      float* bc_rows, int Lrun, int dtype, void* stream);

/* The same with Mamba.dt_proj [F.linear(dt, dt_proj.weight)] computed inside the scan kernel on the tensor core (bf16 only):
 * dbc_* are the x_proj outputs [S*L, ldbc] (dt in columns [0, R), B at [bc_off, bc_off+16), C at [bc_off+16, bc_off+32);
 * ldbc >= 64), wdt_* the dt_proj weights [E, R] with row pitch ldw (elements, a multiple of 8; R <= 64).  Delta is rounded
 * to bf16 where the GEMM would have rounded it, so the result matches pcad_op_linear + pcad_op_biscan. */
int pcad_op_biscan_dt(const void* u_f, const void* dbc_f, const void* u_r, const void* dbc_r, int64_t ldbc, int bc_off,
                      const void* wdt_f, const void* wdt_r, int64_t ldw, int R, const void* z, int64_t ldz,
                      const float* A_f, const float* D_f, const float* dt_bias_f,
                      const float* A_r, const float* D_r, const float* dt_bias_r,
                      void* y, int S, int L, int E, void* stream);

/* Mamba-2 / SSD selective scan [mamba_chunk_scan_combined(x, dt, A, B, C, D=D, z=None, dt_bias, dt_softplus=True)] for
 * both time directions (direction by index math): xbc_f / xbc_r are the two directions' conv + SiLU outputs
 * [S*L, ld_xbc] with x at columns [0, 64 H), B at [64 H, 64 H + 64), C at [64 H + 64, 64 H + 128) (64-wide heads, 64
 * states, one B/C group); dt_raw [S*L, ld_dt] holds the raw dt, one column per head (shared by the directions: in_proj is
 * tied); A_* (= -exp(A_log)), D_*, dt_bias_*: float [H]; y_f / y_r: [S*L, 64 H], y_r written at the original positions.
 * bf16: chunked SSD on tcgen05 (H even), or the sequential recurrence when sequential != 0; f32: sequential recurrence. */
int pcad_op_ssd_scan(const void* xbc_f, const void* xbc_r, int64_t ld_xbc, const void* dt_raw, int64_t ld_dt,
                     const float* A_f, const float* D_f, const float* dt_bias_f,
                     const float* A_r, const float* D_r, const float* dt_bias_r,
                     void* y_f, void* y_r, int S, int L, int H, int dtype, int sequential, void* stream);

/* Mamba2's RMSNormGated(norm_before_gate=False, one group) of each direction followed by BiMambaWrapper's "add":
 * out = rms(y_f * silu(z)) * w_f + rms(y_r * silu(z)) * w_r, rows of E channels; z has row pitch ldz. */
int pcad_op_gated_norm_sum(const void* y_f, const void* y_r, const void* z, int64_t ldz, const float* w_f,
                           const float* w_r, void* out, int64_t rows, int E, float eps, int dtype, void* stream);

/* The pooled mean of pcad_hidden_mean_at_layers for one entry, from the engine's strand-major rows: rows [2*B*L, d] (the
 * B forward strands, then the B RC strands, each L rows of d channels; RC strand b's row t is position L-1-t of window b,
 * channels reversed) -> out float32 [B, 2*d], with the same ranges, NaN rows and summation order.  scratch: float
 * [B * ceil(L / PCAD_HIDDEN_MEAN_CHUNK) * 2 * d] (the chunk partials).  d a multiple of 8; rows 16-byte aligned. */
int pcad_op_hidden_mean(const void* rows, const int32_t* ranges_dev, float* scratch, float* out, int B, int L, int d,
                        int dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PCAD_H_ */
