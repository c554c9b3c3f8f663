"""Forward parity at the benchmark's shapes: the engine's forward, bit for bit, against a replay of it through the verified
operators, one call at a time.

tests/test_kernel_bounds_gpu.py proves each pcad_op_* kernel against float64 at the published presets' shapes.  What sits
between those kernels in csrc/pcad.cu -- the workspace carving, the pitches and column offsets handed from call to call,
which direction's buffers and weights go to which call, the sum-of-squares ping-pong of the fused norm, the embedding's
row_sumsq_kernel, the mode decisions made from the shape (fp32 B|C rows, time-parallel segments, the pruned last layer)
and the hidden tap -- is checked here.  `replay` computes the forward from a CaduceusConfig, a state dict, a dtype and the
ids using only the public operator entry points and exact torch operations (gathers, flips, copies, zero padding), in the
order run_backbone / run_mixer_m1 / run_mixer_m2 launch them.  Every operator is deterministic, so the engine's
hidden_states[-1] must equal the replay's hidden tap exactly.  The logits must equal `lm_head`, the RC LM head in
lm_head_kernel's own order of fp32 operations, on that hidden state, and lie within the a-priori error bound of the float64
RC head.

The replay is tied to the model's semantics separately (`test_replay_matches_the_oracle`: fp32 replay against the CPU
oracle at a small shape), and `test_wiring_errors_are_rejected` shows that single wiring errors in the replay break the
equality.  The replay's plan of calls and modes, and the row_sumsq and lm_head emulations, are checked without a device.

Run with -s to see one line per case with its mode flags, and the file's wall time and peak device memory."""
import ctypes as C
import dataclasses
import time

import pytest
import torch

from plantcaduceus_b200.configuration import CaduceusConfig, preset
from plantcaduceus_b200.weights import EMB_KEY, HEAD_KEY, NORM_F_KEY, layer_key, norm_key, random_init_state_dict
from test_kernel_bounds_gpu import (ALL_PRESETS, BF16, DEV, F32, TD, U32, Call, Guarded, Stats, assert_guards, forward_calls,
                                    forward_lrun, model_dims, scan_segments, sumsq_parts)

NS = 16                      # Mamba-1 d_state
SSD_EPS = 1e-5               # the Mamba-2 mixer's gated RMSNorm epsilon (run_mixer_m2)
B200_SMS = 148
RAGGED = (13, 301)           # T = 7826: ragged row and time tiles, below the fp32 B|C-row threshold
SNP = (256, 512)             # bench.py --workload snp
LONG = (16, 8192)            # bench.py --workload long
BC_ROWS_MIN_T = 65536        # run_mixer_m1: fp32 B|C rows from this many rows on (bf16)
SWITCHES = ("PCAD_SCAN_BC_F32", "PCAD_NO_PRUNE", "PCAD_NO_TIME_PARALLEL", "PCAD_FUSED_DT", "PCAD_NO_FUSED_NORM", "PCAD_SSD_SEQ")


# ---- the plan: modes the forward picks from the shape ------------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class Modes:
    fused: bool        # bf16 activations and residual: add+RMSNorm folded into the in_proj / out_proj epilogues
    res32: bool        # residual stream in fp32 (residual_in_fp32, or fp32 activations)
    f32: bool
    bc_rows: bool      # Mamba-1 bf16: B|C converted to fp32 rows before the scan
    P: int             # Mamba-1: time-parallel segments per sequence
    ssd_seq: bool      # Mamba-2: sequential SSD recurrence instead of the chunked tcgen05 kernel

    def lrun(self, cfg, L, idx):
        """Steps per direction of the last layer's scan when only position idx is scored (0: not pruned), as score_at
        decides it: Mamba-1 only, with at least one layer."""
        if idx is None or cfg.is_mamba2 or cfg.n_layer == 0:
            return 0
        return forward_lrun(L, idx, self.P)

    def flags(self):
        norm = "fused" if self.fused else ("res32" if not self.f32 else "f32")
        return f"{norm:5s} bc_rows={int(self.bc_rows)} P={self.P:2d}" + (" ssd=seq" if self.ssd_seq else "")


def forward_modes(cfg, B, L, dtype, sms, ssd_seq_env=False):
    """What pcad_create and run_mixer_m1 decide for this model and shape with no PCAD_* switch set (PCAD_SSD_SEQ=1 when
    ssd_seq_env)."""
    f32 = dtype == F32
    res32 = f32 or bool(cfg.residual_in_fp32)
    T = 2 * B * L
    if cfg.is_mamba2:
        return Modes(fused=not res32, res32=res32, f32=f32, bc_rows=False, P=1, ssd_seq=f32 or ssd_seq_env)
    return Modes(fused=not res32, res32=res32, f32=f32, bc_rows=not f32 and T >= BC_ROWS_MIN_T,
                 P=scan_segments(cfg.d_inner, 2 * B, L, sms), ssd_seq=False)


# ---- the row sums of squares of the embedding (row_sumsq_kernel) --------------------------------------------------------
def row_sumsq(x, parts):
    """row_sumsq_kernel on bf16 rows x [rows, d] -> fp32 [rows, parts], bit for bit.  Lane l of the row's warp adds, in
    order, the squares of x[8l + 256k + i] for k = 0, 1, ... and i = 0..7 (a bf16 square is exact in fp32, so its fmaf is an
    fp32 add); the 32 lane sums are combined by warp_sum's xor butterfly (16, 8, 4, 2, 1).  Slot 0 holds the sum, the others
    are zero.  Zero padding to a multiple of 256 columns adds exact zeros to lanes that have no element there."""
    rows, d = x.shape
    chunks = -(-d // 256)
    sq = torch.nn.functional.pad(x.float(), (0, chunks * 256 - d)).pow(2).view(rows, chunks, 32, 8)
    acc = torch.zeros(rows, 32, dtype=torch.float32, device=x.device)
    for k in range(chunks):
        for i in range(8):
            acc = acc + sq[:, k, :, i]
    lanes = torch.arange(32, device=x.device)
    for o in (16, 8, 4, 2, 1):
        acc = acc + acc[:, lanes ^ o]
    out = torch.zeros(rows, parts, dtype=torch.float32, device=x.device)
    out[:, 0] = acc[:, 0]
    return out


# ---- the RC LM head (lm_head_kernel) -----------------------------------------------------------------------------------
def fma32(x, y, z):
    """fmaf(x, y, z) on fp32 tensors: x y + z rounded once to fp32.  x y is exact in float64 (48 bits); the float64 sum s
    and its exact error e come from TwoSum.  Rounding s to fp32 gives the correctly rounded result unless s is itself the
    midpoint of two fp32 neighbours and e != 0 (no fp32 midpoint can lie strictly between the exact value and its nearest
    float64); then the exact value lies on e's side of the midpoint."""
    p = x.double() * y.double()
    zd = z.double()
    s = p + zd
    bb = s - p
    e = (p - (s - bb)) + (zd - bb)
    r = s.float()
    n = torch.nextafter(r, torch.where(s > r.double(), torch.full_like(r, float("inf")), torch.full_like(r, -float("inf"))))
    mid = (s != r.double()) & (s == (r.double() + n.double()) * 0.5) & (e != 0)
    beyond = (e > 0) == (n.double() > r.double())       # e points from the midpoint towards n
    return torch.where(mid & beyond, n, r)


def lm_head(hid, W, comp):
    """lm_head_kernel over hidden_states[-1] [rows, 2d] -> fp32 logits [rows, 8], bit for bit.  The kernel reads the forward
    row hf = hid[:d] and the RC strand's row hr = flip(hid[d:]); lane l takes columns j = 8l + 256k + i (k = 0, 1, ...,
    i = 0..7) and accumulates, for every v, acc = fmaf(hf[j], W[v, j], fmaf(hr[j], W[comp[v], j], acc)); the lanes are then
    combined by warp_sum's xor butterfly.  Columns past d are zero-padded: fmaf(0, 0, acc) = acc."""
    rows, d = hid.shape[0], hid.shape[1] // 2
    chunks = -(-d // 256)
    pad = chunks * 256 - d

    def lanes(t):                                    # [n, d] -> [n, chunks, 32, 8]
        return torch.nn.functional.pad(t.float(), (0, pad)).view(t.shape[0], chunks, 32, 8)
    hf, hr = lanes(hid[:, :d]), lanes(hid[:, d:].flip(-1))
    wv = lanes(W)                                    # [8, chunks, 32, 8]
    wc = lanes(W[comp])
    acc = torch.zeros(rows, 32, 8, dtype=torch.float32, device=hid.device)        # [row, lane, v]
    for k in range(chunks):
        for i in range(8):
            acc = fma32(hr[:, k, :, i, None], wc[:, k, :, i].t()[None], acc)
            acc = fma32(hf[:, k, :, i, None], wv[:, k, :, i].t()[None], acc)
    ln = torch.arange(32, device=hid.device)
    for o in (16, 8, 4, 2, 1):
        acc = acc + acc[:, ln ^ o]
    return acc[:, 0]


# ---- executors: the operator entry points, or a record of the calls -----------------------------------------------------
class Recorder:
    """Records every operator call of a replay as the parity file's `Call` (plus the scan's mode arguments) and launches
    nothing: with tensors on the meta device the replay's plan runs without a GPU."""

    def __init__(self):
        self.calls, self.extra = [], []

    def _rec(self, call, **extra):
        self.calls.append(call)
        self.extra.append(extra)

    def linear(self, name, A, W, Cm, M, N, K, lda, ldw, ldc, dtype, A_off=0):
        self._rec(Call("linear", name, M=M, N=N, K=K, lda=lda, ldw=ldw, ldc=ldc, dtype=dtype))

    def linear_residual(self, name, A, W, res_in, res_out, ss_out, M, N, K, lda, ldw, ld_res):
        self._rec(Call("linear_residual", name, M=M, N=N, K=K, lda=lda, ldw=ldw, ldc=ld_res, parts=ss_out.shape[1]))

    def linear_rowscale(self, name, A, W, ss_in, eps, Cm, M, N, K, lda, ldw, ldc):
        self._rec(Call("linear_rowscale", name, M=M, N=N, K=K, lda=lda, ldw=ldw, ldc=ldc, parts=ss_in.shape[1]))

    def add_rmsnorm(self, name, x, res_in, w, y, res_out, rows, d, eps, dtype, res_dtype):
        self._rec(Call("add_rmsnorm", name, M=rows, N=d, dtype=dtype, res_dtype=res_dtype, res_in=res_in is not None,
                       res_out=res_out is not None))

    def conv_silu(self, x, x_off, ldx, wf, bf_, wr, br, out_f, out_r, S, L, E, dtype):
        self._rec(Call("conv_silu", "conv", S=S, L=L, E=E, ld_in=ldx, dtype=dtype), x_off=x_off)

    def biscan_ex(self, uf, df, bcf, ur, dr, bcr, ldbc, bc_off, z, z_off, ldz, dirs, y, S, L, E, segments, seg_state,
                  seg_sumd, bc_rows, Lrun, dtype):
        self._rec(Call("biscan", "scan", S=S, L=L, E=E, ld_in=ldbc, off=bc_off, ld_z=ldz, dtype=dtype), z_off=z_off,
                  segments=segments, bc_rows=bc_rows is not None, Lrun=Lrun)

    def ssd_scan(self, xf, xr, ld_x, dt, dt_off, ld_dt, dirs, yf, yr, S, L, H, dtype, sequential):
        self._rec(Call("ssd_scan", "scan", S=S, L=L, H=H, E=yf.shape[1], ld_in=ld_x, ld_z=ld_dt, dtype=dtype),
                  dt_off=dt_off, sequential=sequential)

    def gated_norm_sum(self, yf, yr, z, z_off, ldz, wf, wr, out, rows, E, eps, dtype):
        self._rec(Call("gated_norm_sum", "gnorm", M=rows, E=E, ld_z=ldz, dtype=dtype), z_off=z_off)


class Launcher(Recorder):
    """Records, and runs each call through its pcad_op_* entry point on the current stream."""

    def __init__(self, lib):
        super().__init__()
        self.lib = lib

    def _ok(self, rc):
        assert rc == 0, self.lib.pcad_last_error(None)

    @staticmethod
    def _p(t, off=0):
        return None if t is None else C.c_void_p(t.data_ptr() + off * t.element_size())

    @staticmethod
    def _s():
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def linear(self, name, A, W, Cm, M, N, K, lda, ldw, ldc, dtype, A_off=0):
        super().linear(name, A, W, Cm, M, N, K, lda, ldw, ldc, dtype)
        self._ok(self.lib.pcad_op_linear(self._p(A, A_off), self._p(W), self._p(Cm), M, N, K, lda, ldw, ldc, dtype, self._s()))

    def linear_residual(self, name, A, W, res_in, res_out, ss_out, M, N, K, lda, ldw, ld_res):
        super().linear_residual(name, A, W, res_in, res_out, ss_out, M, N, K, lda, ldw, ld_res)
        self._ok(self.lib.pcad_op_linear_residual(self._p(A), self._p(W), self._p(res_in), self._p(res_out), self._p(ss_out),
                                                  M, N, K, lda, ldw, ld_res, BF16, self._s()))

    def linear_rowscale(self, name, A, W, ss_in, eps, Cm, M, N, K, lda, ldw, ldc):
        super().linear_rowscale(name, A, W, ss_in, eps, Cm, M, N, K, lda, ldw, ldc)
        self._ok(self.lib.pcad_op_linear_rowscale(self._p(A), self._p(W), self._p(ss_in), ss_in.shape[1], C.c_float(eps),
                                                  self._p(Cm), M, N, K, lda, ldw, ldc, BF16, self._s()))

    def add_rmsnorm(self, name, x, res_in, w, y, res_out, rows, d, eps, dtype, res_dtype):
        super().add_rmsnorm(name, x, res_in, w, y, res_out, rows, d, eps, dtype, res_dtype)
        self._ok(self.lib.pcad_op_add_rmsnorm(self._p(x), self._p(res_in), self._p(w), self._p(y), self._p(res_out), rows, d,
                                              C.c_float(eps), dtype, res_dtype, self._s()))

    def conv_silu(self, x, x_off, ldx, wf, bf_, wr, br, out_f, out_r, S, L, E, dtype):
        super().conv_silu(x, x_off, ldx, wf, bf_, wr, br, out_f, out_r, S, L, E, dtype)
        self._ok(self.lib.pcad_op_conv_silu(self._p(x, x_off), ldx, self._p(wf), self._p(bf_), self._p(wr), self._p(br),
                                            self._p(out_f), self._p(out_r), S, L, E, dtype, self._s()))

    def biscan_ex(self, uf, df, bcf, ur, dr, bcr, ldbc, bc_off, z, z_off, ldz, dirs, y, S, L, E, segments, seg_state,
                  seg_sumd, bc_rows, Lrun, dtype):
        super().biscan_ex(uf, df, bcf, ur, dr, bcr, ldbc, bc_off, z, z_off, ldz, dirs, y, S, L, E, segments, seg_state,
                          seg_sumd, bc_rows, Lrun, dtype)
        (A0, D0, b0), (A1, D1, b1) = dirs
        p = self._p
        self._ok(self.lib.pcad_op_biscan_ex(p(uf), p(df), p(bcf), p(ur), p(dr), p(bcr), ldbc, bc_off, p(z, z_off), ldz,
                                            p(A0), p(D0), p(b0), p(A1), p(D1), p(b1), p(y), S, L, E, segments, p(seg_state),
                                            p(seg_sumd), p(bc_rows), Lrun, dtype, self._s()))

    def ssd_scan(self, xf, xr, ld_x, dt, dt_off, ld_dt, dirs, yf, yr, S, L, H, dtype, sequential):
        super().ssd_scan(xf, xr, ld_x, dt, dt_off, ld_dt, dirs, yf, yr, S, L, H, dtype, sequential)
        (A0, D0, b0), (A1, D1, b1) = dirs
        p = self._p
        self._ok(self.lib.pcad_op_ssd_scan(p(xf), p(xr), ld_x, p(dt, dt_off), ld_dt, p(A0), p(D0), p(b0), p(A1), p(D1), p(b1),
                                           p(yf), p(yr), S, L, H, dtype, int(sequential), self._s()))

    def gated_norm_sum(self, yf, yr, z, z_off, ldz, wf, wr, out, rows, E, eps, dtype):
        super().gated_norm_sum(yf, yr, z, z_off, ldz, wf, wr, out, rows, E, eps, dtype)
        self._ok(self.lib.pcad_op_gated_norm_sum(self._p(yf), self._p(yr), self._p(z, z_off), ldz, self._p(wf), self._p(wr),
                                                 self._p(out), rows, E, C.c_float(eps), dtype, self._s()))


# ---- the replay --------------------------------------------------------------------------------------------------------
def engine_weights(cfg, sd, dtype, device):
    """The weights as pcad_set_weight / pcad_finalize hold them: every floating tensor first cast to the model dtype (as
    modeling.py does), then GEMM weights and the embedding in the activation dtype and everything else in fp32;
    A = -exp(A_log) in fp32 on the device; x_proj zero-padded to RP rows; in the fused-norm path in_proj_s =
    bf16(float(in_proj) * norm_w[col])."""
    td = TD[dtype]
    D = model_dims(cfg)
    fused = dtype == BF16 and not cfg.residual_in_fp32

    def act(k):
        return sd[k].to(td).contiguous().to(device)

    def f32(k):
        return sd[k].to(td).float().contiguous().to(device)

    w = {"emb": act(EMB_KEY), "head": f32(HEAD_KEY if HEAD_KEY in sd else EMB_KEY), "norm_f": f32(NORM_F_KEY), "layers": []}
    for i in range(cfg.n_layer):
        lw = {"in_proj": act(layer_key(i, "mamba_fwd", "in_proj.weight")), "out_proj": act(layer_key(i, "mamba_fwd", "out_proj.weight")),
              "norm_w": f32(norm_key(i)), "dir": []}
        if fused:
            lw["in_proj_s"] = (lw["in_proj"].float() * lw["norm_w"][None, :]).to(torch.bfloat16)
        for direction in ("mamba_fwd", "mamba_rev"):
            def k(leaf):
                return layer_key(i, direction, leaf)
            dw = {"conv_w": f32(k("conv1d.weight")).reshape(-1, 4).contiguous(), "conv_b": f32(k("conv1d.bias")),
                  "A": -torch.exp(f32(k("A_log"))), "D": f32(k("D"))}
            if cfg.is_mamba2:
                dw.update(dt_bias=f32(k("dt_bias")), gnorm_w=f32(k("norm.weight")))
            else:
                R, RP = D["R"], D["RP"]
                xp = act(k("x_proj.weight"))
                dw["x_proj"] = torch.cat((xp, torch.zeros(RP - R - 2 * NS, xp.shape[1], dtype=td, device=device)))
                dw.update(dt_proj=act(k("dt_proj.weight")), dt_bias=f32(k("dt_proj.bias")))
            lw["dir"].append(dw)
        w["layers"].append(lw)
    return w


def gather_rows(t, B, L, idx):
    """gather_rows_kernel: row idx of every forward strand, row L-1-idx of every RC strand -> compact [2B, width]."""
    S = 2 * B
    rows = torch.tensor([idx] * B + [L - 1 - idx] * B, device=t.device)
    return t.view(S, L, -1)[torch.arange(S, device=t.device), rows].contiguous()


def strand_ids(ids, comp):
    """The strand-major ids of the embedding: forward strands ids[b, t], then RC strands comp[ids[b, L-1-t]]."""
    return torch.cat((ids, comp[ids.flip(1)])).reshape(-1)


def hidden_tap(normed, B, L, d):
    """hidden_states[-1] [B, L, 2d] from the strand-major [2BL, d] final norm: the RC half reversed in time and channels."""
    n = normed.view(2, B, L, d)
    return torch.cat((n[0], n[1].flip(1).flip(2)), dim=-1)


WIRING_ERRORS = ("swap_conv_l1", "stale_sumsq_l1", "z_from_x", "lrun_short")


def replay(ex, cfg, w, dtype, ids, modes, prune_idx=None, error=None):
    """The engine's forward over ids [B, L] (int64, on the weights' device), as run_backbone launches it, through the
    executor `ex`.  Returns the final normed rows: [2BL, d] strand-major, or with prune_idx (Mamba-1, score-only last layer)
    the compact [2B, d] rows the head reads (forward strands at prune_idx, RC strands at L-1-prune_idx).  `error` injects
    one of WIRING_ERRORS (the negative controls)."""
    dev = w["emb"].device
    B, L = ids.shape
    T, S = 2 * B * L, 2 * B
    D = model_dims(cfg)
    d, E = D["d"], D["E"]
    td = TD[dtype]
    rdtype = F32 if modes.res32 else BF16
    rd = TD[rdtype]
    eps = float(cfg.norm_epsilon)
    m2 = cfg.is_mamba2
    n_in, ld_in = (D["DIP"], D["DIPP"]) if m2 else (2 * E, 2 * E)
    parts = sumsq_parts(d)
    Lrun = modes.lrun(cfg, L, prune_idx)
    if error == "lrun_short":
        assert Lrun > 0
        Lrun -= 1
    comp = torch.tensor([cfg.complement_map[i] for i in range(cfg.vocab_size)], device=dev)
    h0 = w["emb"][strand_ids(ids, comp)]                                  # embed_kernel: [T, d] act dtype
    if modes.fused:
        resid = h0
        ss = [row_sumsq(resid, parts), torch.empty(T, parts, dtype=torch.float32, device=dev)]
    else:
        hid, resid = h0, torch.empty(T, d, dtype=rd, device=dev)
    cur = 0
    rows, x, res = T, None, None
    for li, lw in enumerate(w["layers"]):
        last = li == cfg.n_layer - 1
        xz = torch.zeros(T, ld_in, dtype=td, device=dev)
        if modes.fused:
            slot = cur ^ 1 if (error == "stale_sumsq_l1" and li == 1) else cur
            ex.linear_rowscale("in_proj", resid, lw["in_proj_s"], ss[slot], eps, xz, T, n_in, d, d, d, ld_in)
        else:
            normed = torch.empty(T, d, dtype=td, device=dev)
            ex.add_rmsnorm("norm", hid, resid if li > 0 else None, lw["norm_w"], normed, resid, T, d, eps, dtype, rdtype)
            ex.linear("in_proj", normed, lw["in_proj"], xz, T, n_in, d, d, d, ld_in, dtype)
            del normed
        dirs = lw["dir"][::-1] if (error == "swap_conv_l1" and li == 1) else lw["dir"]
        conv = [(dirs[k]["conv_w"], dirs[k]["conv_b"]) for k in range(2)]
        if m2:
            CD, H, DIPP = D["CD"], D["H"], D["DIPP"]
            xc = [torch.empty(T, CD, dtype=td, device=dev) for _ in range(2)]
            ex.conv_silu(xz, E, DIPP, *conv[0], *conv[1], xc[0], xc[1], S, L, CD, dtype)
            yd = [torch.empty(T, E, dtype=td, device=dev) for _ in range(2)]
            ex.ssd_scan(xc[0], xc[1], CD, xz, E + CD, DIPP, [(dw["A"], dw["D"], dw["dt_bias"]) for dw in lw["dir"]],
                        yd[0], yd[1], S, L, H, dtype, modes.ssd_seq)
            del xc
            y = torch.empty(T, E, dtype=td, device=dev)
            ex.gated_norm_sum(yd[0], yd[1], xz, E if error == "z_from_x" else 0, DIPP, lw["dir"][0]["gnorm_w"],
                              lw["dir"][1]["gnorm_w"], y, T, E, SSD_EPS, dtype)
            del yd
        else:
            R, RP, P = D["R"], D["RP"], modes.P
            xc = [torch.empty(T, E, dtype=td, device=dev) for _ in range(2)]
            ex.conv_silu(xz, 0, 2 * E, *conv[0], *conv[1], xc[0], xc[1], S, L, E, dtype)
            dbc = [torch.empty(T, RP, dtype=td, device=dev) for _ in range(2)]
            delta = [torch.empty(T, E, dtype=td, device=dev) for _ in range(2)]
            for k in range(2):
                ex.linear("x_proj", xc[k], lw["dir"][k]["x_proj"], dbc[k], T, RP, E, E, E, RP, dtype)
                ex.linear("dt_proj", dbc[k], lw["dir"][k]["dt_proj"], delta[k], T, E, R, RP, R, E, dtype)
            y = torch.empty(T, E, dtype=td, device=dev)
            seg_state = torch.empty(S * P * 2 * E, NS, dtype=torch.float32, device=dev) if P > 1 else None
            seg_sumd = torch.empty(S * P * 2, E, dtype=torch.float32, device=dev) if P > 1 else None
            bcr = torch.empty(2 * T, 2 * NS, dtype=torch.float32, device=dev) if modes.bc_rows else None
            ex.biscan_ex(xc[0], delta[0], dbc[0], xc[1], delta[1], dbc[1], RP, R, xz, 0 if error == "z_from_x" else E, 2 * E,
                         [(dw["A"], dw["D"], dw["dt_bias"]) for dw in lw["dir"]], y, S, L, E, P, seg_state, seg_sumd, bcr,
                         Lrun if last else 0, dtype)
            del xc, dbc, delta, seg_state, seg_sumd, bcr
        del xz
        if last and Lrun > 0:
            # the score-only tail: y and the residual stream at the 2B rows the head reads, then out_proj and the norm there
            rows, y = S, gather_rows(y, B, L, prune_idx)
            res = gather_rows(resid, B, L, prune_idx)
            x = torch.empty(S, d, dtype=rd if modes.fused else td, device=dev)
            if modes.fused:
                ex.linear_residual("out_proj", y, lw["out_proj"], res, x, torch.empty(S, parts, dtype=torch.float32, device=dev),
                                   S, d, E, E, E, d)
            else:
                ex.linear("out_proj", y, lw["out_proj"], x, S, d, E, E, E, d, dtype)
        elif modes.fused:
            ex.linear_residual("out_proj", y, lw["out_proj"], resid, resid, ss[cur ^ 1], T, d, E, E, E, d)
            cur ^= 1
            x = resid
        else:
            ex.linear("out_proj", y, lw["out_proj"], hid, T, d, E, E, E, d, dtype)
            x, res = hid, resid
        del y
    if cfg.n_layer == 0:
        x = resid if modes.fused else hid
    normed = torch.empty(rows, d, dtype=td, device=dev)
    ex.add_rmsnorm("norm_f", x, None if modes.fused or cfg.n_layer == 0 else res, w["norm_f"], normed, None, rows, d, eps, dtype,
                   rdtype)
    return normed


# ---- device-free: the plan and the row_sumsq emulation ------------------------------------------------------------------
META_SD = {}


def meta_replay(cfg, B, L, dtype, modes, prune_idx=None):
    key = (cfg.d_model, cfg.n_layer, cfg.mixer)
    if key not in META_SD:
        META_SD[key] = {k: torch.empty(v.shape, device="meta") for k, v in random_init_state_dict(cfg).items()}
    w = engine_weights(cfg, META_SD[key], dtype, "meta")
    rec = Recorder()
    out = replay(rec, cfg, w, dtype, torch.empty(B, L, dtype=torch.int64, device="meta"), modes, prune_idx)
    return rec, out


def expected_calls(cfg, B, L, dtype):
    """forward_calls (the parity file's derivation of one layer) expanded to a whole forward: the first layer's norm has no
    residual in, x_proj and dt_proj run once per direction, the final norm once."""
    per_layer = forward_calls(cfg, B, L, dtype)
    tail = per_layer.pop()
    layer = []
    for c in per_layer:
        layer.append(c)
        if c.name == "dt_proj":                   # x_proj, dt_proj of the forward direction, then of the reverse one
            layer += layer[-2:]
    first = [dataclasses.replace(c, res_in=False) if c.name == "norm" else c for c in layer]
    return first + layer * (cfg.n_layer - 1) + [tail]


PLAN_CASES = [(name, RAGGED) for name in ALL_PRESETS] + [(name, shape) for name in ("PlantCaduceus_l32", "PlantCAD2-Large-l48-d1536")
                                                           for shape in (SNP, LONG)]


@pytest.mark.parametrize("name,shape", PLAN_CASES, ids=[f"{n}-B{s[0]}-L{s[1]}" for n, s in PLAN_CASES])
def test_replay_plan_matches_forward_calls(name, shape):
    """Needs no device: the replay, run on meta tensors, makes exactly the calls forward_calls derives for the preset, in all
    three modes, with the scan's own arguments (z / dt column, segments, fp32 B|C rows, Lrun) as the forward picks them."""
    B, L = shape
    for dtype, res32 in ((BF16, False), (BF16, True), (F32, False)):
        cfg = dataclasses.replace(preset(name, residual_in_fp32=res32), n_layer=2)
        modes = forward_modes(cfg, B, L, dtype, B200_SMS)
        rec, out = meta_replay(cfg, B, L, dtype, modes)
        assert out.shape == (2 * B * L, cfg.d_model)
        assert rec.calls == expected_calls(cfg, B, L, dtype), (name, dtype, res32)
        E = cfg.d_inner
        for c, ex in zip(rec.calls, rec.extra):
            if c.op == "biscan":
                assert ex == dict(z_off=E, segments=modes.P, bc_rows=modes.bc_rows, Lrun=0)
            elif c.op == "conv_silu":
                assert ex == dict(x_off=E if cfg.is_mamba2 else 0)
            elif c.op == "ssd_scan":
                assert ex == dict(dt_off=E + cfg.conv_dim, sequential=dtype == F32)
            elif c.op == "gated_norm_sum":
                assert ex == dict(z_off=0)
        if cfg.is_mamba2:
            continue
        # the score-only last layer at the benchmark's position: the first layer runs in full, the last one stops early
        # and its out_proj and the final norm run on the 2B gathered rows
        idx = L // 2 - 1
        Lrun = modes.lrun(cfg, L, idx)
        rec, out = meta_replay(cfg, B, L, dtype, modes, prune_idx=idx)
        assert out.shape == (2 * B, cfg.d_model)
        scans = [ex["Lrun"] for c, ex in zip(rec.calls, rec.extra) if c.op == "biscan"]
        assert scans == [0, Lrun]
        assert [c.M for c in rec.calls if c.name in ("out_proj", "norm_f")] == [2 * B * L, 2 * B, 2 * B]


def test_forward_modes_match_hand_derived_values():
    """Needs no device: the modes of the case matrix below, worked out by hand for a 148-SM B200."""
    def m(name, B, L, dtype=BF16, **kw):
        return forward_modes(preset(name, **kw), B, L, dtype, B200_SMS)
    l20, l24, l32, small = "PlantCaduceus_l20", "PlantCaduceus_l24", "PlantCaduceus_l32", "PlantCAD2-Small-l24-d0768"
    assert m(l32, *SNP) == Modes(fused=True, res32=False, f32=False, bc_rows=True, P=1, ssd_seq=False)
    assert m(l32, *SNP, residual_in_fp32=True) == Modes(False, True, False, True, 1, False)
    assert m(l32, *SNP, dtype=F32) == Modes(False, True, True, False, 1, False)
    assert m(l32, *LONG).bc_rows and m(l32, *LONG).P == 1                 # 32 strands x 32 channel blocks fill the GPU
    assert m(l24, *RAGGED) == Modes(True, False, False, False, 1, False)   # T = 7826: B|C converted inside the scan
    # one window: 12 (l20) or 32 (l32) channel blocks per strand, 2 strands; segments of at least 512 steps
    assert (m(l20, 1, 8192).P, m(l20, 1, 8192).bc_rows) == (16, False)
    assert (m(l20, 1, 32768).P, m(l20, 1, 32768).bc_rows) == (16, True)   # T = 65536: time-parallel with fp32 rows
    assert m(l32, 1, 8192).P == 8
    assert m(small, *RAGGED) == Modes(True, False, False, False, 1, False)
    assert forward_modes(preset(small), *RAGGED, BF16, B200_SMS, ssd_seq_env=True).ssd_seq
    assert m(small, *RAGGED, dtype=F32).ssd_seq
    # the last layer's scan when one position is scored: max(p, L-1-p) + 1 steps; not for Mamba-2 or a segmented scan
    cfg = preset(l32)
    assert [m(l32, *SNP).lrun(cfg, 512, p) for p in (255, 0, 511, 101)] == [257, 512, 512, 411]
    assert [m(l24, *RAGGED).lrun(preset(l24), 301, p) for p in (149, 0, 300, 101)] == [152, 301, 301, 200]
    assert m(l20, 1, 8192).lrun(preset(l20), 8192, 4095) == 0
    assert m(small, *RAGGED).lrun(preset(small), 301, 149) == 0


def test_row_sumsq_emulation():
    """Needs no device: the emulation of row_sumsq_kernel.  Lane 0 holds 2^12 and seven ones: in the kernel's order
    2^24 + 1 rounds back to 2^24 seven times, where a float64 sum rounded once gives 2^24 + 8.  Elsewhere the emulation is
    within the fp32 rounding of the float64 sum, at every published width."""
    for d in (384, 512, 768, 1024, 1536):
        x = torch.zeros(3, d, dtype=torch.bfloat16)
        x[0, 0] = 2.0 ** 12
        x[0, 1:8] = 1.0
        x[1, :] = 1.0
        x[2, 8] = 3.0                                             # lane 1
        x[2, d - 1] = 2.0                                         # the last lane that holds an element
        parts = sumsq_parts(d)
        ss = row_sumsq(x, parts)
        assert ss.shape == (3, parts) and not ss[:, 1:].any()
        assert ss[:, 0].tolist() == [2.0 ** 24, float(d), 13.0], d
        g = torch.Generator().manual_seed(d)
        xr = (torch.randn(64, d, generator=g) * torch.exp(torch.randn(64, 1, generator=g))).to(torch.bfloat16)
        ref = xr.double().pow(2).sum(-1)
        got = row_sumsq(xr, parts)[:, 0].double()
        assert ((got - ref).abs() <= 2.0 ** -24 * d * ref).all(), d


def test_fma32_rounds_once():
    """Needs no device: fma32 against values worked out by hand where rounding x y + z first to float64 and then to fp32
    lands on a tie and picks the wrong neighbour; and equal to that double rounding on random values, where a tie is
    improbable."""
    u = 2.0 ** -23
    t = lambda *v: torch.tensor(v, dtype=torch.float32)
    # x y = -2^-24 + 2^-70: the exact sum lies 2^-70 above the midpoint of 1 + 2u and 1 + 3u
    x, y, z = t(-(2.0 ** -24) * (1 + u)), t(1 - u), t(1 + 3 * u)
    assert fma32(x, y, z).item() == 1 + 3 * u
    assert (x.double() * y.double() + z.double()).float().item() == 1 + 2 * u      # the tie went to the even neighbour
    # x y = 2^-24 - 2^-70: the exact sum lies 2^-70 below the midpoint of 1 + u and 1 + 2u
    x, y, z = t(2.0 ** -24 * (1 + u)), t(1 - u), t(1 + u)
    assert fma32(x, y, z).item() == 1 + u
    assert (x.double() * y.double() + z.double()).float().item() == 1 + 2 * u
    g = torch.Generator().manual_seed(3)
    x, y, z = (torch.randn(100000, generator=g) for _ in range(3))
    assert torch.equal(fma32(x, y, z), (x.double() * y.double() + z.double()).float())


def test_lm_head_emulation():
    """Needs no device: lm_head on small integers, where every operation is exact, against the integer RC head (the flip of
    the RC half, the complement map and the lane layout all show); on random rows within one rounding per term of float64."""
    cfg = preset("PlantCaduceus_l20")
    comp = torch.tensor([cfg.complement_map[i] for i in range(8)])
    for d in (384, 768, 1536):
        g = torch.Generator().manual_seed(d)
        hid = torch.randint(-8, 9, (17, 2 * d), generator=g).float()
        W = torch.randint(-8, 9, (8, d), generator=g).float()
        want = hid[:, :d].long() @ W.long().t() + hid[:, d:].flip(-1).long() @ W[comp].long().t()
        assert torch.equal(lm_head(hid.to(torch.bfloat16), W, comp), want.float()), d
        hid = torch.randn(64, 2 * d, generator=g).to(torch.bfloat16)
        W = torch.randn(8, d, generator=g)
        ref = hid[:, :d].double() @ W.double().t() + hid[:, d:].flip(-1).double() @ W[comp].double().t()
        mag = hid[:, :d].double().abs() @ W.double().abs().t() + hid[:, d:].flip(-1).double().abs() @ W[comp].double().abs().t()
        assert ((lm_head(hid, W, comp).double() - ref).abs() <= U32 * (ref.abs() + 2 * d * mag)).all(), d


# ---- on the GPU -----------------------------------------------------------------------------------------------------------
WORKSPACE = {"max": 0}


@pytest.fixture(scope="module")
def lib(cuda_device):
    from plantcaduceus_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def budget():
    """Wall time and peak device memory of the file's GPU tests (printed with -s): torch's own allocations (the replay, the
    outputs, the float64 checks) and, beside them, the largest engine workspace, which libpcad allocates itself.  The engine
    is destroyed before its replay runs, so the two never add up."""
    if not torch.cuda.is_available():
        yield
        return
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    torch.cuda.synchronize()
    print(f"\n[replay] file: wall {time.time() - t0:.1f} s, peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB "
          f"in torch, largest engine workspace {WORKSPACE['max'] / 2 ** 30:.2f} GiB")
    torch.backends.cuda.matmul.allow_tf32 = tf32


@pytest.fixture
def switches(monkeypatch, budget):
    """No PCAD_* switch set: the engine picks its modes from the shape, as forward_modes does."""
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    yield monkeypatch
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def make_ids(B, L, seed):
    """Mostly a/c/g/t, with every other id (PAD, mask, N, 7) at a few positions."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(3, 7, (B, L), generator=g)
    spots = torch.rand(B, L, generator=g) < 0.05
    ids[spots] = torch.tensor([0, 1, 2, 7])[torch.randint(0, 4, (int(spots.sum()),), generator=g)]
    return ids


def two_layers(name, **kw):
    return dataclasses.replace(preset(name, **kw), n_layer=2)


def score_positions(L):
    """The score-only positions: the benchmark's (window centre), both edges, and an odd off-centre one."""
    return [L // 2 - 1, 0, L - 1, (L // 3) | 1]


def first_difference(got, want):
    diff = (got != want) & ~(torch.isnan(got) & torch.isnan(want))
    n = int(diff.sum())
    if not n:
        return "none"
    i = int(diff.reshape(-1).nonzero()[0])
    return (f"{n} of {got.numel()} values differ, first at flat index {i} (got {float(got.reshape(-1)[i]):.6g}, "
            f"want {float(want.reshape(-1)[i]):.6g})")


HEAD_A_PRIORI = 1.0   # k of the float64 head check: an fp32 fmaf chain of at most 2d terms is within 2d 2^-24 mag, plus one rounding


def head_stats(hid, logits, W, comp, d):
    """float64 RC head on the engine's own hidden output, logits[b, t] = h[:d] W^T + flip(h[d:]) W[comp]^T, with the
    a-priori unit 2^-24 |ref| + 2d 2^-24 mag per element."""
    W = W.double()
    Wc = W[comp]
    rows = hid.shape[0] * hid.shape[1]
    h, lg = hid.reshape(rows, 2 * d), logits.reshape(rows, -1)
    st = Stats()
    for r0 in range(0, rows, 8192):
        r1 = min(rows, r0 + 8192)
        hf, hr = h[r0:r1, :d].double(), h[r0:r1, d:].flip(-1).double()
        ref = hf @ W.t() + hr @ Wc.t()
        mag = hf.abs() @ W.abs().t() + hr.abs() @ Wc.abs().t()
        st.add(lg[r0:r1], ref, mag, U32, U32 * 2 * d, row0=r0)
    return st


def head_matches(hid, logits, W, comp, d):
    """pcad_forward's logits against lm_head (the kernel's own order of fp32 operations) on its hidden output, bit for bit."""
    rows = hid.shape[0] * hid.shape[1]
    h, lg = hid.reshape(rows, 2 * d), logits.reshape(rows, -1)
    for r0 in range(0, rows, 32768):
        want = lm_head(h[r0:r0 + 32768], W, comp)
        if not torch.equal(lg[r0:r0 + 32768], want):
            return f"rows from {r0}: {first_difference(lg[r0:r0 + 32768], want)}"
    return None


def run_engine(lib, cfg, sd, dtype, ids, entry_points=True):
    """pcad_forward into Guarded buffers, then the scoring and tap entry points against slices of its outputs.  Destroys
    the engine before returning: (hidden [B, L, 2d], logits [B, L, 8])."""
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    from plantcaduceus_b200.tokenizer import CharDNATokenizer
    B, L = ids.shape
    d, V = cfg.d_model, cfg.vocab_size
    model = CaduceusForMaskedLM.from_pretrained(sd, config=cfg, torch_dtype=TD[dtype]).to(DEV)
    WORKSPACE["max"] = max(WORKSPACE["max"], model.workspace_bytes(B, L))
    ids_dev = ids.to(DEV)
    logits = Guarded(B * L, V, torch.float32)
    hidden = Guarded(B * L, 2 * d, TD[dtype])
    rc = lib.pcad_forward(model._handle, C.c_void_p(ids_dev.data_ptr()), B, L, logits.ptr, hidden.ptr,
                          C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.pcad_last_error(model._handle)
    torch.cuda.synchronize()
    assert_guards("pcad_forward", logits=logits, hidden=hidden)
    hid, lg = hidden.t.view(B, L, 2 * d).clone(), logits.t.view(B, L, V).clone()
    del logits, hidden
    if entry_points:
        ids_u8 = ids_dev.to(torch.uint8)
        vocab = CharDNATokenizer().get_vocab()
        acgt = torch.tensor([vocab[c] for c in "acgt"], device=DEV)
        g = torch.Generator().manual_seed(L)
        pos = torch.stack([torch.randperm(L, generator=g)[:3] for _ in range(B)]).to(DEV, torch.int32)
        b_idx = torch.arange(B, device=DEV)[:, None]
        checks = {f"score_masked_at({p})": (model.score_masked(ids_u8, p)[:, 0], lg[:, p][:, acgt]) for p in score_positions(L)}
        checks["score_masked"] = (model.score_masked(ids_u8, pos), lg[b_idx, pos.long()][..., acgt])
        checks["hidden_at"] = (model.hidden_at(ids_u8, pos), hid[b_idx, pos.long()])
        torch.cuda.synchronize()
        bad = {k: first_difference(got, want) for k, (got, want) in checks.items() if not torch.equal(got, want)}
        assert not bad, f"entry points differ from the matching slice of pcad_forward's outputs: {bad}"
    model._release()
    return hid, lg


def check_case(lib, cfg, dtype, B, L, label, ssd_seq_env=False, seed=0):
    sd = random_init_state_dict(cfg, seed=seed)
    ids = make_ids(B, L, seed=B * 100003 + L)
    modes = forward_modes(cfg, B, L, dtype, torch.cuda.get_device_properties(0).multi_processor_count, ssd_seq_env)
    t0 = time.time()
    hid, logits = run_engine(lib, cfg, sd, dtype, ids)
    w = engine_weights(cfg, sd, dtype, DEV)
    ex = Launcher(lib)
    ids_dev = ids.to(DEV)
    want = hidden_tap(replay(ex, cfg, w, dtype, ids_dev, modes), B, L, cfg.d_model)
    torch.cuda.synchronize()
    assert all(c.op != "biscan" or e["segments"] == modes.P for c, e in zip(ex.calls, ex.extra))
    assert torch.equal(hid, want), f"{label}: hidden_states[-1] differs from the replay: {first_difference(hid, want)}"
    del want
    comp = torch.tensor([cfg.complement_map[i] for i in range(cfg.vocab_size)], device=DEV)
    bad = head_matches(hid, logits, w["head"], comp, cfg.d_model)
    assert bad is None, f"{label}: logits differ from lm_head on the forward's hidden output: {bad}"
    st = head_stats(hid, logits, w["head"], comp, cfg.d_model)
    # the score-only tail (Mamba-1): compact rows of the pruned replay against the full forward's rows at the scored position
    lruns = []
    for p in score_positions(L):
        Lrun = modes.lrun(cfg, L, p)
        if not Lrun:
            continue
        lruns.append(f"{p}:{Lrun}")
        compact = replay(Launcher(lib), cfg, w, dtype, ids_dev, modes, prune_idx=p)
        got = torch.cat((compact[:B], compact[B:].flip(-1)), dim=-1)
        assert torch.equal(got, hid[:, p]), f"{label}: pruned tail at {p} (Lrun {Lrun}): {first_difference(got, hid[:, p])}"
        del compact, got
    print(f"[replay] {label:58s} {modes.flags()} Lrun {','.join(lruns) or '-':26s} bit-identical, logits bit-identical; "
          f"float64 head err/bound {st.ratio / HEAD_A_PRIORI:.3g} ({len(ex.calls)} calls, {time.time() - t0:.1f} s)")
    assert st.ratio <= HEAD_A_PRIORI and st.bad == 0, f"{label}: logits against the float64 RC head: {st.worst}"


def case(name, shape, mode, ssd_seq=False):
    kw = {"residual_in_fp32": True} if mode == "bf16-res32" else {}
    dtype = F32 if mode == "f32" else BF16
    tag = f"{name}-B{shape[0]}-L{shape[1]}-{mode}" + ("-ssdseq" if ssd_seq else "")
    return pytest.param(name, kw, dtype, shape, ssd_seq, id=tag)


MODES3 = ("bf16", "bf16-res32", "f32")
CASES = ([case(n, RAGGED, m) for n in ALL_PRESETS for m in MODES3]
         + [case(n, SNP, m) for n in ("PlantCaduceus_l32", "PlantCAD2-Large-l48-d1536") for m in MODES3]
         + [case(n, LONG, m) for n in ("PlantCaduceus_l32", "PlantCAD2-Large-l48-d1536") for m in ("bf16", "f32")]
         + [case("PlantCaduceus_l20", (1, 8192), "bf16"), case("PlantCaduceus_l32", (1, 8192), "bf16"),
            case("PlantCaduceus_l20", (1, 32768), "bf16"), case("PlantCAD2-Small-l24-d0768", RAGGED, "bf16", ssd_seq=True)])


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw,dtype,shape,ssd_seq", CASES)
def test_engine_equals_replay(lib, switches, name, kw, dtype, shape, ssd_seq):
    """pcad_forward's hidden_states[-1] is bit-identical to the replay; its logits are within K["head"] of the float64 RC
    head on that hidden state; score_masked_at (pruned for Mamba-1), score_masked and hidden_at return the matching slices
    of the forward's outputs, and the pruned replay's compact rows equal the forward's rows at the scored position."""
    if ssd_seq:
        switches.setenv("PCAD_SSD_SEQ", "1")
    cfg = two_layers(name, **kw)
    mode = "f32" if dtype == F32 else ("bf16-res32" if kw else "bf16")
    check_case(lib, cfg, dtype, *shape, f"{name} B={shape[0]} L={shape[1]} {mode}", ssd_seq_env=ssd_seq)


def small_config(mixer):
    if mixer == "mamba1":
        return CaduceusConfig(d_model=256, n_layer=2)
    return CaduceusConfig(d_model=256, n_layer=2, ssm_cfg=dict(layer="Mamba2", d_state=64, d_conv=4, expand=2, headdim=64,
                                                              ngroups=1, conv_bias=True, bias=False))


@pytest.mark.gpu
@pytest.mark.parametrize("mixer", ["mamba1", "mamba2"])
def test_replay_matches_the_oracle(lib, switches, mixer):
    """The replay is the model, not a copy of pcad.cu: in fp32 it is within 1e-4 (relative to the largest value) of the CPU
    oracle's hidden_states[-1], and the engine equals it bit for bit at the same shape, in both dtypes."""
    from oracle import caduceus_oracle as O
    cfg = small_config(mixer)
    B, L = 3, 200
    sd = random_init_state_dict(cfg, seed=5)
    ids = make_ids(B, L, seed=7)
    _, hs = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32, output_hidden_states=True)
    ref = hs[-1]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    w = engine_weights(cfg, sd, F32, DEV)
    got = hidden_tap(replay(Launcher(lib), cfg, w, F32, ids.to(DEV), forward_modes(cfg, B, L, F32, sms)), B, L, cfg.d_model).cpu()
    rel = float((got - ref).abs().max() / ref.abs().max())
    print(f"[replay] {mixer} d=256 B={B} L={L} fp32 replay vs oracle: max |diff| / max |ref| = {rel:.3g}")
    assert rel <= 1e-4
    for dtype in (F32, BF16):
        check_case(lib, cfg, dtype, B, L, f"{mixer} d=256 B={B} L={L} {'f32' if dtype == F32 else 'bf16'}", seed=5)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["PlantCaduceus_l24", "PlantCAD2-Small-l24-d0768"])
def test_wiring_errors_are_rejected(lib, switches, name):
    """The equality is not blind: each single wiring error in the replay -- layer 1's forward and reverse conv weights
    swapped, layer 1's in_proj reading layer 0's sum-of-squares slot, z read from x's columns, the pruned layer's scan one
    step short (Mamba-1) -- makes it fail, while the replay without an error matches."""
    cfg = two_layers(name)
    B, L = RAGGED
    sd = random_init_state_dict(cfg, seed=11)
    ids = make_ids(B, L, seed=12)
    hid, _ = run_engine(lib, cfg, sd, BF16, ids, entry_points=False)
    modes = forward_modes(cfg, B, L, BF16, torch.cuda.get_device_properties(0).multi_processor_count)
    assert modes.fused
    w = engine_weights(cfg, sd, BF16, DEV)
    ids_dev = ids.to(DEV)
    p = L // 2 - 1

    def matches(error, prune_idx=None):
        out = replay(Launcher(lib), cfg, w, BF16, ids_dev, modes, prune_idx=prune_idx, error=error)
        if prune_idx is None:
            return torch.equal(hidden_tap(out, B, L, cfg.d_model), hid)
        return torch.equal(torch.cat((out[:B], out[B:].flip(-1)), dim=-1), hid[:, prune_idx])
    assert matches(None)
    errors = ["swap_conv_l1", "stale_sumsq_l1", "z_from_x"]
    if not cfg.is_mamba2:
        assert matches(None, prune_idx=p)
        errors.append("lrun_short")
    for e in errors:
        still = matches(e, prune_idx=p if e == "lrun_short" else None)
        print(f"[replay] negative control {name} {e:15s}: {'MATCHES (blind check)' if still else 'rejected'}")
        assert not still, f"{name}: the replay with wiring error {e} still equals the engine"
