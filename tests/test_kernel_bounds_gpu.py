"""Kernel parity at the published models' shapes: every pcad_op_* kernel against a float64 reference of the same operation,
element by element, with guard bands around every output.

The operator calls are derived from the model (`forward_calls`: what run_backbone / run_mixer_m1 / run_mixer_m2 in
csrc/pcad.cu launch for a CaduceusConfig), so the GEMM, norm, conv and scan shapes below are the ones the seven published
presets run.  The check is per element:

    |got - ref64| <= k * (u_out * |ref64| + u_acc * mag)

where ref64 is the float64 result on the kernel's own (rounded) inputs and mag is the same float64 computation run on
absolute values (|A| |W|^T for a GEMM; |u|, |B|, |C|, |D| with the same decays for a scan; |w| |x| + |b| for the conv).
Every operator is linear in its data inputs once the decays are fixed, so mag is, per element, the scale that rounding
errors are proportional to.  u_out is the unit roundoff of the stored output, i.e. one rounding (2^-8 for bf16, 2^-24 for
fp32); u_acc that of the accumulation (2^-24 per term summed in fp32, or 2^-8 where an intermediate is stored as bf16).  k is a
per-kernel constant set from a B200 run (`K` below: at most twice the measured maximum of err / (u_out |ref| + u_acc mag)).
A kernel that drops a K block, mis-scales a channel or a row tile, or mis-rounds one element fails here even when the
element is far below the largest output.

Each output sits between sentinel-filled guard rows (1024-byte aligned), and where the entry point takes a row pitch the
output also has pad columns; after every call every byte outside the logical output must be bit-unchanged.

Run with -s to see, per case, the maximum err / bound ratio and the maximum absolute error."""
import ctypes as C
import math
import time
import zlib
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

from plantcaduceus_b200.configuration import PRESETS, preset

pytestmark = pytest.mark.gpu

BF16, F32 = 0, 1
TD = {BF16: torch.bfloat16, F32: torch.float32}
U_OUT = {BF16: 2.0 ** -8, F32: 2.0 ** -24}    # unit roundoff of the stored output: one rounding
U32 = 2.0 ** -24                              # fp32 unit roundoff
T_PROD = 2 * 256 * 512                        # bench.py snp (B = 256, L = 512) and long (B = 16, L = 8192): 262 144 rows
M_RAGGED = 2 * 13 * 301                       # 7826 = 30 * 256 + 146: a full and a partial CTA pair at the end
CONV_TT = 64                                  # kConvTT (csrc/elementwise.cuh): timesteps per conv thread
DEV = "cuda"
SP_THRESHOLD = 20.0                           # softplus is the identity above this (mamba_ssm, F.softplus)

# k per checker, from the first B200 run (max err / unit bound, times at most 2).  See the module docstring.
K = {
    "gemm": 1.5, "gemm_residual": 1.5, "gemm_sumsq": 0.006, "gemm_rowscale": 1.5,
    "norm_bf16": 1.5, "norm_f32": 1.0, "conv_bf16": 1.5, "conv_f32": 2.0,
    "scan_bf16": 1.25, "scan_f32": 0.375, "segscan_bf16": 1.25, "segscan_f32": 0.45,
    "softplus_bf16": 1.5, "softplus_f32": 12.0, "decay_bf16": 1.5, "decay_f32": 4.0,
    "ssd_tc": 1.3, "ssd_seq_bf16": 1.0, "ssd_seq_f32": 0.7, "gnorm_bf16": 2.0, "gnorm_f32": 0.2,
    "head": 4e-4,     # measured maximum 1.85e-4 (fp32, PlantCaduceus_l32 widths, B = 256, L = 512)

    "bc_rows": 1.0,   # a priori, not measured: one rounding of the product and one of ln 2 (2^-24 |ref| each) bound it by 1
}

PLANTCADUCEUS = ["PlantCaduceus_l20", "PlantCaduceus_l24", "PlantCaduceus_l28", "PlantCaduceus_l32"]
PLANTCAD2 = ["PlantCAD2-Small-l24-d0768", "PlantCAD2-Medium-l48-d1024", "PlantCAD2-Large-l48-d1536"]
ALL_PRESETS = PLANTCADUCEUS + PLANTCAD2
LARGEST = ("PlantCaduceus_l32", "PlantCAD2-Large-l48-d1536")   # run at the production row count


# ---- the operator calls of one layer, derived from the model ------------------------------------------------------------
def pick_bn(N):
    """The GEMM's column tile width (csrc/gemm_tcgen05.cuh pick_bn)."""
    if N <= 64:
        return 64
    if N <= 80:
        return 80
    if N <= 96:
        return 96
    if N <= 128:
        return 128
    waste256 = -(-N // 256) * 256 - N
    waste128 = -(-N // 128) * 128 - N
    return 128 if waste128 < waste256 else 256


def sumsq_parts(N):
    """Sum-of-squares slots per row of the residual epilogue: one per column tile."""
    return -(-N // pick_bn(N))


def uses_cta_pair(N, K):
    return pick_bn(N) == 256 and N % 256 == 0 and K >= 256


@dataclass(frozen=True)
class Call:
    op: str                 # pcad_op_<op>
    name: str               # the forward's name for it
    M: int = 0              # GEMM rows / norm rows
    N: int = 0
    K: int = 0
    lda: int = 0
    ldw: int = 0
    ldc: int = 0            # output pitch (linear, rowscale); ld_res (residual)
    parts: int = 0          # sum-of-squares slots (residual out, row scale in)
    dtype: int = BF16
    res_dtype: int = BF16   # add_rmsnorm: residual stream dtype
    res_in: bool = False    # add_rmsnorm: a residual is added
    res_out: bool = False   # add_rmsnorm: the sum is stored
    S: int = 0              # sequences (2B: forward and RC strands)
    L: int = 0
    E: int = 0              # channels (conv, scans, gated norm)
    ld_in: int = 0          # conv ldx, biscan ldbc, ssd ld_xbc
    ld_z: int = 0           # biscan / gated norm z pitch, ssd ld_dt
    off: int = 0            # biscan bc_off (= R)
    H: int = 0


def model_dims(cfg):
    d, E, N = cfg.d_model, cfg.d_inner, cfg.d_state
    dims = dict(d=d, E=E, N=N)
    if cfg.is_mamba2:
        H = E // cfg.headdim
        CD = E + 2 * cfg.ngroups * N
        DIP = E + CD + H
        dims.update(H=H, CD=CD, DIP=DIP, DIPP=-(-DIP // 8) * 8)
    else:
        R = cfg.dt_rank
        dims.update(R=R, RP=-(-(R + 2 * N) // 16) * 16)
    return dims


def forward_calls(cfg, B, L, dtype=BF16):
    """The pcad_op_* calls one layer of the forward over B windows of length L makes (plus the final norm), in order.
    The bf16 forward with a bf16 residual stream fuses the add+RMSNorm into the GEMM epilogues (out_proj: residual add and
    row sums of squares; in_proj: the row scale); fp32 activations or residual_in_fp32 run the norm kernel instead."""
    D = model_dims(cfg)
    d, E = D["d"], D["E"]
    T, S = 2 * B * L, 2 * B
    res_f32 = dtype == F32 or cfg.residual_in_fp32
    res_dtype = F32 if res_f32 else BF16
    fused = not res_f32
    parts = sumsq_parts(d)
    if cfg.is_mamba2:
        n_in, ld_in = D["DIP"], D["DIPP"]
    else:
        n_in, ld_in = 2 * E, 2 * E
    calls = []
    if fused:
        calls.append(Call("linear_rowscale", "in_proj", M=T, N=n_in, K=d, lda=d, ldw=d, ldc=ld_in, parts=parts))
    else:
        calls.append(Call("add_rmsnorm", "norm", M=T, N=d, dtype=dtype, res_dtype=res_dtype, res_in=True, res_out=True))
        calls.append(Call("linear", "in_proj", M=T, N=n_in, K=d, lda=d, ldw=d, ldc=ld_in, dtype=dtype))
    if cfg.is_mamba2:
        E_, CD, H, DIPP = D["E"], D["CD"], D["H"], D["DIPP"]
        calls.append(Call("conv_silu", "conv", S=S, L=L, E=CD, ld_in=DIPP, dtype=dtype))
        calls.append(Call("ssd_scan", "scan", S=S, L=L, H=H, E=E_, ld_in=CD, ld_z=DIPP, dtype=dtype))
        calls.append(Call("gated_norm_sum", "gnorm", M=T, E=E_, ld_z=DIPP, dtype=dtype))
    else:
        R, RP = D["R"], D["RP"]
        calls.append(Call("conv_silu", "conv", S=S, L=L, E=E, ld_in=2 * E, dtype=dtype))
        calls.append(Call("linear", "x_proj", M=T, N=RP, K=E, lda=E, ldw=E, ldc=RP, dtype=dtype))
        calls.append(Call("linear", "dt_proj", M=T, N=E, K=R, lda=RP, ldw=R, ldc=E, dtype=dtype))
        calls.append(Call("biscan", "scan", S=S, L=L, E=E, ld_in=RP, off=R, ld_z=2 * E, dtype=dtype))
    if fused:
        calls.append(Call("linear_residual", "out_proj", M=T, N=d, K=E, lda=E, ldw=E, ldc=d, parts=parts))
    else:
        calls.append(Call("linear", "out_proj", M=T, N=d, K=E, lda=E, ldw=E, ldc=d, dtype=dtype))
    calls.append(Call("add_rmsnorm", "norm_f", M=T, N=d, dtype=dtype, res_dtype=res_dtype, res_in=not fused))
    return calls


def gemm_calls(name):
    return [c for c in forward_calls(preset(name), 256, 512) if c.op.startswith("linear")]


# ---- plumbing ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib(cuda_device):
    from plantcaduceus_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module", autouse=True)
def budget(request):
    """Wall time and peak device memory of the whole file (printed with -s); no TF32 in any fp32 matmul."""
    if not torch.cuda.is_available():
        yield
        return
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    torch.cuda.synchronize()
    print(f"\n[bounds] file: wall {time.time() - t0:.1f} s, peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")
    torch.backends.cuda.matmul.allow_tf32 = tf32


@pytest.fixture(autouse=True)
def release_memory():
    yield
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def vp(t, elem_offset=0):
    return C.c_void_p(t.data_ptr() + elem_offset * t.element_size())


def ok(lib, rc):
    assert rc == 0, lib.pcad_last_error(None)


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def randn(g, *shape, dtype=torch.float32, scale=1.0, shift=0.0):
    return (torch.randn(*shape, generator=g, device=DEV) * scale + shift).to(dtype)


def rand(g, *shape, lo=0.0, hi=1.0):
    return torch.rand(*shape, generator=g, device=DEV, dtype=torch.float64) * (hi - lo) + lo


SENTINEL = 0x7FA5   # int16; as bf16 a NaN, two of them an fp32 NaN


class Guarded:
    """A [rows, cols] output with row pitch ld inside a sentinel-filled allocation: guard rows before and after (at
    1024-byte aligned offsets) and, if ld > cols, pad columns.  `intact()` says whether every byte outside the logical
    output still holds the sentinel."""

    def __init__(self, rows, cols, dtype, ld=None):
        self.rows, self.cols, self.ld = rows, cols, ld or cols
        self.esz = torch.empty((), dtype=dtype).element_size()
        self.nbytes = rows * self.ld * self.esz
        self.guard = max(-(-4 * self.ld * self.esz // 1024) * 1024, 1024)
        total = 1024 + self.guard + -(-self.nbytes // 1024) * 1024 + self.guard
        self.raw = torch.full((total // 2,), SENTINEL, dtype=torch.int16, device=DEV).view(torch.uint8)
        self.start = (-self.raw.data_ptr()) % 1024 + self.guard
        self.mat = self.raw[self.start:self.start + self.nbytes].view(dtype).view(rows, self.ld)
        self.t = self.mat[:, :cols]

    @property
    def ptr(self):
        return C.c_void_p(self.mat.data_ptr())

    def intact(self):
        r16 = self.raw.view(torch.int16)
        a, b = self.start // 2, (self.start + self.nbytes) // 2
        good = bool((r16[:a] == SENTINEL).all()) and bool((r16[b:] == SENTINEL).all())
        if self.ld > self.cols:
            pad = self.mat.view(torch.int16)[:, self.cols * self.esz // 2:]
            good = good and bool((pad == SENTINEL).all())
        return good


def assert_guards(label, **bufs):
    bad = [name for name, g in bufs.items() if not g.intact()]
    assert not bad, f"{label}: bytes outside the output changed in {bad}"


class Stats:
    """Running maximum of err / (u_out |ref| + u_acc mag) and of |err| over chunks of one output."""

    def __init__(self):
        self.ratio, self.err, self.n, self.bad = 0.0, 0.0, 0, 0
        self.worst = ""

    def add(self, got, ref, mag, u_out, u_acc, floor=0.0, row0=0):
        got = got.double()
        err = (got - ref).abs()
        unit = u_out * ref.abs() + u_acc * mag + floor
        nan = ~torch.isfinite(got)
        self.bad += int(nan.sum())
        err = torch.where(nan, torch.full_like(err, math.inf), err)
        r = err / unit
        r = torch.where(unit > 0, r, torch.where(err > 0, torch.full_like(r, math.inf), torch.zeros_like(r)))
        rmax = float(r.max())
        if rmax > self.ratio or not self.worst:
            i = int(r.argmax())
            row, col = divmod(i, got.shape[-1]) if got.dim() > 1 else (0, i)
            self.worst = (f"worst at [{row0 + row}, {col}]: got {float(got.flatten()[i]):.6g} ref {float(ref.flatten()[i]):.6g} "
                          f"mag {float(mag.flatten()[i]):.6g}")
        self.ratio = max(self.ratio, rmax)
        self.err = max(self.err, float(err.max()))
        self.n += got.numel()
        return self


def verdict(family, case, *stats_and_labels):
    """Print one line per checked output and assert each within K[family]."""
    k = K[family]
    fails = []
    for label, st in stats_and_labels:
        print(f"[bounds] {family:14s} {case + ' ' + label:62s} max err/unit {st.ratio:9.4g}  err/bound {st.ratio / k:7.3g}"
              f"  max|err| {st.err:9.3g}  ({st.n} values; {st.worst})")
        if not st.ratio <= k:
            fails.append(f"{label}: max err/unit {st.ratio:.4g} > k = {k} ({st.bad} non-finite)")
    assert not fails, f"{family} {case}: " + "; ".join(fails)


def rejects(family, st):
    return not st.ratio <= K[family]


def softplus64(x):
    return torch.where(x > SP_THRESHOLD, x, torch.log1p(torch.exp(torch.clamp(x, max=SP_THRESHOLD))))


def silu64(x):
    return x * torch.sigmoid(x)


def checkpoint_dt_bias(g, n):
    """dt_bias as Mamba initialises it: the inverse softplus of dt ~ log-uniform in [1e-3, 1e-1]."""
    dt = torch.exp(rand(g, n, lo=math.log(1e-3), hi=math.log(1e-1)))
    return (dt + torch.log(-torch.expm1(-dt))).float()


# ---- GEMM --------------------------------------------------------------------------------------------------------------
CHUNK_ROWS = 4096


def gemm_reference_stats(got, A, W, K_, rowscale=None, resid=None, sumsq=None, bn=0):
    """float64 A[:, :K] W[:, :K]^T (times rowscale, plus resid) in row chunks; sumsq: also check the per-column-tile sums
    of squares of the result (the residual epilogue's second output)."""
    W64 = W[:, :K_].double()
    Wa = W64.abs()
    st, ss_st = Stats(), Stats()
    M, N = got.shape
    for r0 in range(0, M, CHUNK_ROWS):
        r1 = min(M, r0 + CHUNK_ROWS)
        a = A[r0:r1, :K_].double()
        ref = a @ W64.t()
        mag = a.abs() @ Wa.t()
        if rowscale is not None:
            ref *= rowscale[r0:r1, None]
            mag *= rowscale[r0:r1, None]
        if resid is not None:
            rr = resid[r0:r1].double()
            ref += rr
            mag += rr.abs()
        st.add(got[r0:r1], ref, mag, U_OUT[BF16], U32 * K_, row0=r0)
        if sumsq is not None:
            P = sumsq.shape[1]
            pad = P * bn - N
            refp = F.pad(ref, (0, pad)).view(r1 - r0, P, bn)
            magp = F.pad(mag, (0, pad)).view(r1 - r0, P, bn)
            ss_ref = refp.pow(2).sum(-1)
            # each v carries <= 2^-24 K mag of accumulation error, v^2 twice that relative; plus the fp32 sum of bn squares
            ss_mag = 2 * K_ * (refp.abs() * magp).sum(-1) + bn * ss_ref
            ss_st.add(sumsq[r0:r1], ss_ref, ss_mag, 0.0, U32, row0=r0)
        del a, ref, mag
    return st, ss_st


def make_gemm_operands(g, call, M, lda_fill=True):
    """A [M, lda] (every column filled: a GEMM that reads past K is caught) with per-row scales exp(N(0,1)); W [N, ldw]."""
    A = randn(g, M, call.lda, dtype=torch.bfloat16)
    A.mul_(torch.exp(randn(g, M, 1)).to(torch.bfloat16))
    W = randn(g, call.N, call.ldw, dtype=torch.bfloat16, scale=call.K ** -0.5)
    return A, W


PAD = 16   # pad columns on every pitched GEMM output (ld = the forward's pitch + PAD)


def run_gemm_case(lib, call, M, seed):
    """One forward GEMM call at M rows, checked against float64; returns [(family, label, Stats)]."""
    g = gen(seed)
    A, W = make_gemm_operands(g, call, M)
    N, K_ = call.N, call.K
    if call.op == "linear":
        out = Guarded(M, N, torch.bfloat16, ld=call.ldc + PAD)
        ok(lib, lib.pcad_op_linear(vp(A), vp(W), out.ptr, M, N, K_, call.lda, call.ldw, out.ld, BF16, stream()))
        torch.cuda.synchronize()
        assert_guards(f"linear {call.name}", C=out)
        st, _ = gemm_reference_stats(out.t, A, W, K_)
        return [("gemm", "C", st)]
    if call.op == "linear_residual":
        # in place, as the forward runs it: resid_in == resid_out, pitch ld_res
        res = Guarded(M, N, torch.bfloat16, ld=call.ldc + PAD)
        res.t.copy_(randn(g, M, N, dtype=torch.bfloat16, scale=2.0))
        res0 = res.t.clone()
        ss = Guarded(M, call.parts, torch.float32)
        ok(lib, lib.pcad_op_linear_residual(vp(A), vp(W), res.ptr, res.ptr, ss.ptr, M, N, K_, call.lda, call.ldw, res.ld, BF16, stream()))
        torch.cuda.synchronize()
        assert_guards(f"linear_residual {call.name}", resid=res, sumsq=ss)
        st, ss_st = gemm_reference_stats(res.t, A, W, K_, resid=res0, sumsq=ss.t, bn=pick_bn(N))
        return [("gemm_residual", "resid_out", st), ("gemm_sumsq", "sumsq_out", ss_st)]
    assert call.op == "linear_rowscale"
    # C = rsqrt(sum_parts sumsq / K + eps) * (A Ws^T): the float64 norm (from the same fp32 sums) followed by the matmul
    eps = 1e-5
    bn = pick_bn(K_)
    ssq = torch.cat([F.pad(A[r0:r0 + CHUNK_ROWS, :K_].double().pow(2), (0, call.parts * bn - K_)).view(-1, call.parts, bn).sum(-1)
                     for r0 in range(0, M, CHUNK_ROWS)]).float()
    rstd = 1.0 / torch.sqrt(ssq.double().sum(-1) / K_ + eps)
    out = Guarded(M, N, torch.bfloat16, ld=call.ldc + PAD)
    ok(lib, lib.pcad_op_linear_rowscale(vp(A), vp(W), vp(ssq), call.parts, C.c_float(eps), out.ptr, M, N, K_, call.lda, call.ldw,
                                        out.ld, BF16, stream()))
    torch.cuda.synchronize()
    assert_guards(f"linear_rowscale {call.name}", C=out)
    st, _ = gemm_reference_stats(out.t, A, W, K_, rowscale=rstd)
    return [("gemm_rowscale", "C", st)]


def gemm_cases():
    cases = []
    for name in ALL_PRESETS:
        M = T_PROD if name in LARGEST else M_RAGGED
        for c in gemm_calls(name):
            cases.append(pytest.param(name, c.name, M, id=f"{name}-{c.name}-M{M}"))
    # the four tail classes of the CTA-pair kernel: the last pair's second CTA empty (1, 127, 128) or holding one row (129)
    for c in ("in_proj", "out_proj"):
        for tail in (1, 127, 128, 129):
            M = 3 * 256 + tail
            cases.append(pytest.param("PlantCaduceus_l32", c, M, id=f"PlantCaduceus_l32-{c}-M{M}"))
    return cases


@pytest.mark.parametrize("name,which,M", gemm_cases())
def test_gemm_matches_float64(lib, name, which, M):
    call = next(c for c in gemm_calls(name) if c.name == which)
    outs = run_gemm_case(lib, call, M, seed=zlib.crc32(f"{name}/{which}/{M}".encode()) & 0xFFFF)
    pair = "pair" if uses_cta_pair(call.N, call.K) else f"BN={pick_bn(call.N)}"
    for family, label, st in outs:
        verdict(family, f"{name} {which} M={M} N={call.N} K={call.K} ({pair})", (label, st))


def test_gemm_plain_epilogue_tails_on_the_pair_kernel(lib):
    """The unfused forward's in_proj (plain epilogue) through the pair kernel at the four tail classes."""
    base = next(c for c in gemm_calls("PlantCaduceus_l32") if c.name == "in_proj")
    call = Call("linear", "in_proj", N=base.N, K=base.K, lda=base.lda, ldw=base.ldw, ldc=base.ldc)
    assert uses_cta_pair(call.N, call.K)
    for tail in (1, 127, 128, 129):
        M = 3 * 256 + tail
        (family, label, st), = run_gemm_case(lib, call, M, seed=tail)
        verdict(family, f"l32 in_proj plain M={M}", (label, st))


# ---- forward_calls against values worked out by hand ------------------------------------------------------------------
PARTS = {"PlantCaduceus_l20": 3, "PlantCaduceus_l24": 2, "PlantCaduceus_l28": 3, "PlantCaduceus_l32": 4,
         "PlantCAD2-Small-l24-d0768": 3, "PlantCAD2-Medium-l48-d1024": 4, "PlantCAD2-Large-l48-d1536": 6}


def test_forward_calls_match_hand_derived_shapes():
    """Needs no device: the shapes forward_calls derives from each preset against values worked out by hand."""
    assert set(ALL_PRESETS) == set(PRESETS)
    RP = {"PlantCaduceus_l20": 64, "PlantCaduceus_l24": 64, "PlantCaduceus_l28": 80, "PlantCaduceus_l32": 96}
    DIP = {"PlantCAD2-Small-l24-d0768": 3224, "PlantCAD2-Medium-l48-d1024": 4256, "PlantCAD2-Large-l48-d1536": 6320}
    for name in ALL_PRESETS:
        cfg = preset(name)
        calls = {c.name: c for c in forward_calls(cfg, 256, 512)}
        d, E = cfg.d_model, cfg.d_inner
        for c in calls.values():
            if c.op.startswith("linear"):
                assert c.M == T_PROD
                assert c.lda % 8 == 0 and c.ldw % 8 == 0 and c.ldc % 8 == 0, c
                assert c.lda >= c.K and c.ldw >= c.K and c.ldc >= c.N, c
        assert calls["out_proj"].parts == calls["in_proj"].parts == PARTS[name] == -(-d // pick_bn(d))
        assert (calls["out_proj"].N, calls["out_proj"].K) == (d, E)
        if name in RP:
            R = -(-d // 16)
            assert calls["x_proj"].N == calls["x_proj"].ldc == calls["dt_proj"].lda == calls["scan"].ld_in == RP[name]
            assert calls["dt_proj"].K == calls["scan"].off == R
            assert calls["in_proj"].N == calls["in_proj"].ldc == 2 * E
            assert calls["conv"].E == E and calls["conv"].ld_in == calls["scan"].ld_z == 2 * E
        else:
            dipp = -(-DIP[name] // 8) * 8
            assert calls["in_proj"].N == DIP[name] and calls["in_proj"].ldc == dipp
            assert calls["in_proj"].N % pick_bn(calls["in_proj"].N) != 0   # a partial column tile
            assert calls["conv"].E == E + 128 and calls["conv"].ld_in == dipp
            assert calls["scan"].H == E // 64 and calls["scan"].ld_z == calls["gnorm"].ld_z == dipp
        # the fp32 forward runs the norm kernel and plain GEMMs
        ops32 = [c.op for c in forward_calls(cfg, 2, 64, dtype=F32)]
        assert "linear_residual" not in ops32 and "linear_rowscale" not in ops32 and ops32.count("add_rmsnorm") == 2
    assert uses_cta_pair(4096, 1024) and uses_cta_pair(1024, 2048) and not uses_cta_pair(96, 2048)


def test_sumsq_parts_match_the_library(lib):
    for name in ALL_PRESETS:
        cfg = preset(name)
        d, E = cfg.d_model, cfg.d_inner
        assert lib.pcad_op_sumsq_parts(d) == PARTS[name]
        for N in (d, E, 2 * E, 64, 80, 96, 3224, 4256, 6320):
            assert sumsq_parts(N) == lib.pcad_op_sumsq_parts(N)


# ---- add_rmsnorm -------------------------------------------------------------------------------------------------------
NORM_MODES = [(F32, F32), (BF16, F32), (BF16, BF16)]


def run_norm(lib, rows, d, dtype, res_dtype, seed, with_res=True):
    g = gen(seed)
    td, tr = TD[dtype], TD[res_dtype]
    x = randn(g, rows, d, dtype=td)
    x.mul_(torch.exp(randn(g, rows, 1)).to(td))   # rows of different scale: a wrong row scale shows
    r = randn(g, rows, d, dtype=tr, scale=2.0) if with_res else None
    w = randn(g, d, scale=0.3, shift=1.0)
    y = Guarded(rows, d, td)
    ro = Guarded(rows, d, tr)
    eps = 1e-5
    ok(lib, lib.pcad_op_add_rmsnorm(vp(x), vp(r) if with_res else None, vp(w), y.ptr, ro.ptr, rows, d, eps, dtype, res_dtype, stream()))
    torch.cuda.synchronize()
    assert_guards("add_rmsnorm", y=y, res_out=ro)
    return x, r, w, eps, y, ro


def norm_stats(got_y, got_r, x, r, w, eps, dtype, res_dtype):
    sy, sr = Stats(), Stats()
    rows, d = x.shape
    for r0 in range(0, rows, 16384):
        r1 = min(rows, r0 + 16384)
        s = x[r0:r1].double() + (r[r0:r1].double() if r is not None else 0.0)
        rstd = torch.rsqrt(s.pow(2).mean(-1, keepdim=True) + eps)
        ref = s * rstd * w.double()
        # statistics in fp32 over d terms: 2^-24 d relative on rstd
        sy.add(got_y[r0:r1], ref, ref.abs(), U_OUT[dtype], U32 * d, row0=r0)
        if got_r is not None:
            sr.add(got_r[r0:r1], s, s.abs(), U_OUT[res_dtype], U32, row0=r0)
    return sy, sr


@pytest.mark.parametrize("dtype,res_dtype", NORM_MODES, ids=["f32-f32", "bf16-f32res", "bf16-bf16res"])
@pytest.mark.parametrize("d", [768, 1536, 2048])
def test_add_rmsnorm_matches_float64(lib, d, dtype, res_dtype):
    family = "norm_f32" if dtype == F32 else "norm_bf16"
    # production rows, then every partly empty last block of 8 rows
    for rows in [T_PROD] + [8 * 37 + t for t in range(1, 8)]:
        x, r, w, eps, y, ro = run_norm(lib, rows, d, dtype, res_dtype, seed=d + rows)
        sy, sr = norm_stats(y.t, ro.t, x, r, w, eps, dtype, res_dtype)
        verdict(family, f"d={d} rows={rows} {TD[dtype]}/{TD[res_dtype]} res", ("y", sy), ("res_out", sr))
        del x, r, y, ro
    # first layer: no residual in
    x, _, w, eps, y, ro = run_norm(lib, 8 * 37 + 5, d, dtype, res_dtype, seed=d, with_res=False)
    sy, sr = norm_stats(y.t, ro.t, x, None, w, eps, dtype, res_dtype)
    verdict(family, f"d={d} rows=301 {TD[dtype]}/{TD[res_dtype]} no res", ("y", sy), ("res_out", sr))


# ---- conv + SiLU -------------------------------------------------------------------------------------------------------
def conv_reference(x, wf, bf_, wr, br_, S, L, E):
    """x: [S*L, E] (float64) -> (ref_f, mag_f, ref_r, mag_r), pre-activation magnitude |b| + sum |w| |x|."""
    xs = x.view(S, L, E)
    xp = F.pad(xs, (0, 0, 3, 3))
    af = bf_.double().expand(S, L, E).clone()
    ar = br_.double().expand(S, L, E).clone()
    mf = bf_.double().abs().expand(S, L, E).clone()
    mr = br_.double().abs().expand(S, L, E).clone()
    for k in range(4):
        xf = xp[:, k:k + L]             # x[t - 3 + k]
        xr = xp[:, 6 - k:6 - k + L]     # x[t + 3 - k]
        af += wf[:, k].double() * xf
        ar += wr[:, k].double() * xr
        mf += wf[:, k].double().abs() * xf.abs()
        mr += wr[:, k].double().abs() * xr.abs()
    return (silu64(af).view(S * L, E), mf.view(S * L, E), silu64(ar).view(S * L, E), mr.view(S * L, E))


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("E", [1664, 2048, 3200, 4096])
def test_conv_silu_matches_float64(lib, E, dtype):
    family = "conv_f32" if dtype == F32 else "conv_bf16"
    td = TD[dtype]
    for L in (512, 8192, CONV_TT - 1, CONV_TT + 1):
        S = max(2, 8192 // L)
        g = gen(E * 31 + L)
        ldx = E + 136                               # x inside a wider row (Mamba-2: x|B|C of in_proj's output)
        xz = randn(g, S * L, ldx, dtype=td)
        xz[:, E:] = 1e4                             # a conv that read past its E channels would show
        wf, wr = randn(g, E, 4, scale=0.5), randn(g, E, 4, scale=0.5)
        bf_, br_ = randn(g, E), randn(g, E)
        of, orv = Guarded(S * L, E, td), Guarded(S * L, E, td)
        ok(lib, lib.pcad_op_conv_silu(vp(xz), ldx, vp(wf), vp(bf_), vp(wr), vp(br_), of.ptr, orv.ptr, S, L, E, dtype, stream()))
        torch.cuda.synchronize()
        assert_guards("conv", out_f=of, out_r=orv)
        ref_f, mag_f, ref_r, mag_r = conv_reference(xz[:, :E].double(), wf, bf_, wr, br_, S, L, E)
        u_acc = 4 * U32   # four fp32 products summed; SiLU's slope is at most 1.1
        sf = Stats().add(of.t, ref_f, mag_f, U_OUT[dtype], u_acc)
        sr = Stats().add(orv.t, ref_r, mag_r, U_OUT[dtype], u_acc)
        verdict(family, f"E={E} S={S} L={L}", ("out_f", sf), ("out_r", sr))
        del xz, of, orv, ref_f, mag_f, ref_r, mag_r


# ---- Mamba-1 bidirectional scan ----------------------------------------------------------------------------------------
NS = 16   # d_state


@dataclass
class ScanInputs:
    S: int
    L: int
    E: int
    R: int
    RP: int
    dtype: int
    u: list
    dl: list
    bc: list
    xz: torch.Tensor
    A: list
    D: list
    bias: list


def scan_inputs(S, L, E, R, dtype, seed):
    """Inputs drawn like a checkpoint's: A = -(1..16) (S4D-real), D ~ 1, dt_bias = inverse softplus of log-uniform dt."""
    g = gen(seed)
    td = TD[dtype]
    RP = -(-(R + 2 * NS) // 16) * 16
    u = [randn(g, S * L, E, dtype=td) for _ in range(2)]
    dl = [randn(g, S * L, E, dtype=td, scale=0.5) for _ in range(2)]
    bc = [randn(g, S * L, RP, dtype=td) for _ in range(2)]
    xz = randn(g, S * L, 2 * E, dtype=td)
    A = [(-torch.arange(1, NS + 1, device=DEV, dtype=torch.float32).expand(E, NS) * torch.exp(randn(g, E, 1, scale=0.1))).contiguous()
         for _ in range(2)]
    D = [randn(g, E, scale=0.1, shift=1.0) for _ in range(2)]
    bias = [checkpoint_dt_bias(g, E) for _ in range(2)]
    return ScanInputs(S, L, E, R, RP, dtype, u, dl, bc, xz, A, D, bias)


def biscan_reference(si, seqs):
    """float64 bidirectional scan of the sequences `seqs`: (ref, mag) [len(seqs) * L, E]; mag runs the same recurrence on
    |u|, |B|, |C|, |D| with the same decays."""
    S, L, E, R, RP = si.S, si.L, si.E, si.R, si.RP
    sel = torch.tensor(seqs, device=DEV)
    ns = len(seqs)
    outs = []
    for k in range(2):
        uu = si.u[k].view(S, L, E)[sel].double()
        dd = softplus64(si.dl[k].view(S, L, E)[sel].double() + si.bias[k].double())
        bc = si.bc[k].view(S, L, RP)[sel].double()
        Bm, Cm = bc[..., R:R + NS], bc[..., R + NS:R + 2 * NS]
        A = si.A[k].double()
        Dk = si.D[k].double()
        h = torch.zeros(2, ns, E, NS, dtype=torch.float64, device=DEV)
        y = torch.empty(2, ns, L, E, dtype=torch.float64, device=DEV)
        steps = range(L) if k == 0 else range(L - 1, -1, -1)
        for t in steps:
            dA = torch.exp(dd[:, t, :, None] * A)                                       # [ns, E, N]
            du = torch.stack((dd[:, t] * uu[:, t], dd[:, t] * uu[:, t].abs()))          # [2, ns, E]
            Bt = torch.stack((Bm[:, t], Bm[:, t].abs()))[:, :, None, :]                 # [2, ns, 1, N]
            Ct = torch.stack((Cm[:, t], Cm[:, t].abs()))[:, :, None, :]
            h = dA * h + du[..., None] * Bt
            y[:, :, t] = (h * Ct).sum(-1) + torch.stack((Dk * uu[:, t], Dk.abs() * uu[:, t].abs()))
        outs.append(y)
    gz = silu64(si.xz.view(S, L, 2 * E)[sel][..., E:].double())
    ref = (outs[0][0] + outs[1][0]) * gz
    mag = (outs[0][1] + outs[1][1]) * gz.abs()
    return ref.reshape(ns * L, E), mag.reshape(ns * L, E)


def scan_units(dtype):
    """bf16: one rounding of y, plus one of the direction's partial parked in y (<= 2^-8 mag); fp32: 2^-24 per term of
    one step's 2N-term sums."""
    return (U_OUT[BF16], 2.0 ** -8) if dtype == BF16 else (U32, 2 * NS * U32)


def scan_args(si, y):
    """The 20 data arguments every pcad_op_biscan* entry point starts with."""
    E = si.E
    return (vp(si.u[0]), vp(si.dl[0]), vp(si.bc[0]), vp(si.u[1]), vp(si.dl[1]), vp(si.bc[1]), si.RP, si.R, vp(si.xz, E), 2 * E,
            vp(si.A[0]), vp(si.D[0]), vp(si.bias[0]), vp(si.A[1]), vp(si.D[1]), vp(si.bias[1]), y.ptr, si.S, si.L, E)


def run_biscan(lib, si, segments=0):
    S, L, E = si.S, si.L, si.E
    td = TD[si.dtype]
    y = Guarded(S * L, E, td)
    args = scan_args(si, y)
    if segments:
        state = Guarded(S * segments * 2 * E, NS, torch.float32)
        sumd = Guarded(S * segments * 2, E, torch.float32)
        ok(lib, lib.pcad_op_biscan_segmented(*args, segments, state.ptr, sumd.ptr, si.dtype, stream()))
        torch.cuda.synchronize()
        assert_guards("biscan_segmented", y=y, seg_state=state, seg_sumd=sumd)
    else:
        ok(lib, lib.pcad_op_biscan(*args, si.dtype, stream()))
        torch.cuda.synchronize()
        assert_guards("biscan", y=y)
    return y


def sample_sequences(S, seed, n_random=6):
    g = torch.Generator().manual_seed(seed)
    mid = (torch.randperm(S - 2, generator=g)[:n_random] + 1).tolist() if S > 2 else []
    return sorted(set([0, S - 1] + mid))


def scan_stats(y, si, seqs):
    ref, mag = biscan_reference(si, seqs)
    got = y.t.view(si.S, si.L, si.E)[torch.tensor(seqs, device=DEV)].reshape(-1, si.E)
    u_out, u_acc = scan_units(si.dtype)
    return Stats().add(got, ref, mag, u_out, u_acc), ref, mag


@pytest.mark.parametrize("dtype,S", [(BF16, 512), (F32, 64)], ids=["bf16-S512", "f32-S64"])
@pytest.mark.parametrize("E,R", [(2048, 64), (768, 24)], ids=["l32", "l20"])
def test_biscan_matches_float64(lib, dtype, S, E, R):
    """The sequential scan at the scoring batch (S = 512 strands of 512 bp: blockIdx.y up to 511, every channel block); the
    reference covers the first, the last and six random sequences, all channels.  pcad_op_biscan runs the kScanPlain mode
    (B|C converted in the kernel); the mode the bf16 forward runs at T >= 65536 (kScanBcF32: B|C as fp32 rows from
    bc_to_f32_kernel) is checked on the same inputs by test_biscan_bc_rows_matches_plain_and_float64."""
    si = scan_inputs(S, 512, E, R, dtype, seed=E + S)
    y = run_biscan(lib, si)
    seqs = sample_sequences(S, seed=E)
    st, _, _ = scan_stats(y, si, seqs)
    verdict("scan_f32" if dtype == F32 else "scan_bf16", f"S={S} L=512 E={E} R={R} seqs {seqs}", ("y", st))


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("P", [2, 8, 32])
def test_biscan_segmented_matches_float64(lib, P, dtype):
    S, L, E, R = 2, 4096, 512, 32
    si = scan_inputs(S, L, E, R, dtype, seed=100 + P)
    y = run_biscan(lib, si, segments=P)
    st, _, _ = scan_stats(y, si, list(range(S)))
    verdict("segscan_f32" if dtype == F32 else "segscan_bf16", f"P={P} S={S} L={L} E={E}", ("y", st))


# ---- the scan as the forward runs it: fp32 B|C rows, time-parallel segments, early stop (pcad_op_biscan_ex) --------------
SEG_STATE_BYTES = 16 << 20   # kSegStateBytes (csrc/pcad.cu)


def scan_segments(E, S, L, num_sms):
    """Segments per sequence of the forward's Mamba-1 scan (a copy of scan_segments in csrc/pcad.cu, 64-channel CTAs, 4
    resident per SM)."""
    P = 1
    ctas, slots = -(-E // 64) * S, 4 * num_sms
    while (P < 32 and ctas * P * 2 <= slots and L % (P * 2) == 0 and L // (P * 2) >= 512
           and S * P * 2 * 2 * E * NS * 4 <= SEG_STATE_BYTES):
        P *= 2
    return P


def forward_lrun(L, p, P=1):
    """Steps per direction of the score-only last layer's scan at scored position p (a copy of the line in run_mixer_m1,
    csrc/pcad.cu); 0: the whole sequence.  Rows [L - Lrun, Lrun) then hold final values."""
    pruned = p >= 0 and P == 1 and L >= 8
    return (p if p > L - 1 - p else L - 1 - p) + 1 if pruned else 0


def num_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def run_biscan_ex(lib, si, segments=0, bc_rows=False, Lrun=0):
    """pcad_op_biscan_ex with every buffer it writes (y, the fp32 B|C rows, the segment state) Guarded: (rc, {name: buf})."""
    S, L, E = si.S, si.L, si.E
    bufs = {"y": Guarded(S * L, E, TD[si.dtype])}
    if segments > 1:
        bufs["seg_state"] = Guarded(S * segments * 2 * E, NS, torch.float32)
        bufs["seg_sumd"] = Guarded(S * segments * 2, E, torch.float32)
    if bc_rows:
        bufs["bc_rows"] = Guarded(2 * S * L, 2 * NS, torch.float32)

    def ptr(k):
        return bufs[k].ptr if k in bufs else None
    rc = lib.pcad_op_biscan_ex(*scan_args(si, bufs["y"]), segments, ptr("seg_state"), ptr("seg_sumd"), ptr("bc_rows"), Lrun,
                               si.dtype, stream())
    torch.cuda.synchronize()
    return rc, bufs


def run_biscan_ex_ok(lib, si, **kw):
    rc, bufs = run_biscan_ex(lib, si, **kw)
    ok(lib, rc)
    assert_guards(f"biscan_ex {kw}", **bufs)
    return bufs


def untouched(g):
    return bool((g.raw.view(torch.int16) == SENTINEL).all())


def bc_rows_stats(rows, si):
    """The fp32 B|C scratch: [B ln 2 | C] of both directions.  Bit-exact against the same fp32 product in torch, and within
    one rounding of the product plus one of ln 2 (2^-24 |ref| each) of float64 on the bf16 inputs."""
    S, L, R = si.S, si.L, si.R
    got = rows.t.view(2, S * L, 2 * NS)
    st = Stats()
    for k in range(2):
        bc = si.bc[k][:, R:R + 2 * NS].float()
        want32 = torch.cat((bc[:, :NS] * torch.tensor(math.log(2.0), dtype=torch.float32, device=DEV), bc[:, NS:]), dim=1)
        assert torch.equal(got[k], want32), f"B|C rows, direction {k}: not the fp32 product"
        ref = bc.double() * torch.tensor([math.log(2.0)] * NS + [1.0] * NS, dtype=torch.float64, device=DEV)
        st.add(got[k], ref, ref.abs(), U32, U32)
    return st


@pytest.mark.parametrize("E,R", [(2048, 64), (768, 24)], ids=["l32", "l20"])
def test_biscan_bc_rows_matches_plain_and_float64(lib, E, R):
    """The scan the bf16 forward runs at T >= 65536 (every scan of bench.py): B|C as fp32 rows written by bc_to_f32_kernel and
    read by TMA (kScanBcF32: its own stage layout, double-buffered ys, one barrier per chunk), at the scoring batch, on the
    inputs of test_biscan_matches_float64.  Same arithmetic in the same order as kScanPlain: bit-identical output."""
    S, L = 512, 512
    si = scan_inputs(S, L, E, R, BF16, seed=E + S)
    plain = run_biscan(lib, si)
    bufs = run_biscan_ex_ok(lib, si, bc_rows=True)
    y = bufs["y"]
    assert torch.equal(y.t, plain.t), "fp32 B|C rows mode differs from the plain mode"
    del plain
    seqs = sample_sequences(S, seed=E)
    st, _, _ = scan_stats(y, si, seqs)
    verdict("scan_bf16", f"bc_rows S={S} L={L} E={E} R={R} seqs {seqs}", ("y", st))
    verdict("bc_rows", f"S={S} L={L} R={R} both directions", ("bc_rows", bc_rows_stats(bufs["bc_rows"], si)))


def test_biscan_time_parallel_bc_rows_matches_float64(lib):
    """Low-batch long context as the forward runs it: B = 1, L = 32768 windows of PlantCaduceus_l20 (S = 2, E = 768,
    T = 65536: fp32 B|C rows), cut into the number of segments the forward picks on this device (16 on a 148-SM B200)."""
    S, L, E, R = 2, 32768, 768, 24
    P = scan_segments(E, S, L, num_sms())
    assert P > 1 and forward_lrun(L, L // 2, P) == 0
    si = scan_inputs(S, L, E, R, BF16, seed=321)
    plain = run_biscan(lib, si, segments=P)
    y = run_biscan_ex_ok(lib, si, segments=P, bc_rows=True)["y"]
    assert torch.equal(y.t, plain.t), "time-parallel scan: fp32 B|C rows mode differs from the plain mode"
    del plain
    t0 = time.time()
    st, _, _ = scan_stats(y, si, list(range(S)))
    verdict("segscan_bf16", f"bc_rows P={P} S={S} L={L} E={E} (float64 reference {time.time() - t0:.1f} s)", ("y", st))


SCAN_MODES = [(BF16, False), (BF16, True), (F32, False)]
SCAN_MODE_IDS = ["bf16", "bf16-bc_rows", "f32"]


def check_early_stop(lib, si, full, ref, mag, seqs, p, bc_rows, label):
    """One early-stopped scan against the full-length run of the same mode (bit-identical on the rows that hold final values)
    and against float64 there."""
    S, L, E = si.S, si.L, si.E
    Lrun = forward_lrun(L, p)
    assert Lrun > 0
    y = run_biscan_ex_ok(lib, si, bc_rows=bc_rows, Lrun=Lrun)["y"]
    lo, hi = L - Lrun, Lrun
    got = y.t.view(S, L, E)[:, lo:hi]
    assert torch.equal(got, full.t.view(S, L, E)[:, lo:hi]), f"{label} p={p} Lrun={Lrun}: rows [{lo}, {hi}) differ from the full run"
    sel = torch.tensor(seqs, device=DEV)
    u_out, u_acc = scan_units(si.dtype)
    st = Stats().add(got[sel].reshape(-1, E), ref.view(len(seqs), L, E)[:, lo:hi].reshape(-1, E),
                     mag.view(len(seqs), L, E)[:, lo:hi].reshape(-1, E), u_out, u_acc)
    verdict("scan_f32" if si.dtype == F32 else "scan_bf16", f"{label} p={p} Lrun={Lrun} rows [{lo}, {hi})", ("y", st))


@pytest.mark.parametrize("dtype,bc_rows", SCAN_MODES, ids=SCAN_MODE_IDS)
def test_biscan_early_stop_at_the_scoring_batch(lib, dtype, bc_rows):
    """The score-only last layer (pcad_score_masked_at, the score-window calls, bench.py's scoring workload): each direction
    stops after max(p, L-1-p) + 1 steps.  l32 widths at the scoring batch, p = 255 (the benchmark's), 256, 100, and 0 (a full
    run).  bf16 with fp32 B|C rows is exactly the benchmark's last layer."""
    S, L, E, R = 512, 512, 2048, 64
    si = scan_inputs(S, L, E, R, dtype, seed=77 + dtype)
    full = run_biscan_ex_ok(lib, si, bc_rows=bc_rows)["y"]
    seqs = sample_sequences(S, seed=78)
    st, ref, mag = scan_stats(full, si, seqs)
    label = f"early stop {SCAN_MODE_IDS[SCAN_MODES.index((dtype, bc_rows))]} S={S} L={L} E={E}"
    verdict("scan_f32" if dtype == F32 else "scan_bf16", f"{label} full", ("y", st))
    for p in (255, 256, 100, 0):
        check_early_stop(lib, si, full, ref, mag, seqs, p, bc_rows, label)


RAGGED_STOPS = [(301, 150), (301, 7), (33, 16), (8, 3), (17, 8)]


@pytest.mark.parametrize("dtype,bc_rows", SCAN_MODES, ids=SCAN_MODE_IDS)
def test_biscan_early_stop_ragged(lib, dtype, bc_rows):
    """Early stop where the last chunk is partial (nsteps < 16) and the epilogue's has_final / late_chunk paths change:
    (301, 150) leaves one valid row, (8, 3) is the shortest window the forward prunes (one chunk)."""
    S, E, R = 6, 512, 32
    for L, p in RAGGED_STOPS:
        si = scan_inputs(S, L, E, R, dtype, seed=L * 1000 + p)
        full = run_biscan_ex_ok(lib, si, bc_rows=bc_rows)["y"]
        seqs = list(range(S))
        ref, mag = biscan_reference(si, seqs)
        label = f"early stop {SCAN_MODE_IDS[SCAN_MODES.index((dtype, bc_rows))]} S={S} L={L} E={E}"
        check_early_stop(lib, si, full, ref, mag, seqs, p, bc_rows, label)


def test_biscan_ex_rejects_bad_arguments(lib):
    """Combinations pcad_op_biscan_ex refuses: an error code and not one byte of any buffer written."""
    S, L, E, R = 4, 64, 512, 32
    sis = {dt: scan_inputs(S, L, E, R, dt, seed=9) for dt in (BF16, F32)}
    bad = [(F32, 0, True, 0, "fp32 B|C rows"), (F32, 0, True, L, "fp32 B|C rows"),
           (BF16, 2, False, L - 8, "early stop + time-parallel"), (BF16, 2, True, L // 2, "early stop + time-parallel"),
           (BF16, 0, False, -1, "Lrun < 0"), (BF16, 0, True, L + 1, "Lrun > L"),
           (BF16, 0, False, L // 2 - 1, "Lrun < (L+1)/2"), (F32, 0, False, 1, "Lrun < (L+1)/2")]
    for dtype, segments, bc_rows, Lrun, why in bad:
        rc, bufs = run_biscan_ex(lib, sis[dtype], segments=segments, bc_rows=bc_rows, Lrun=Lrun)
        assert rc != 0, f"{why}: accepted (dtype {dtype}, segments {segments}, bc_rows {bc_rows}, Lrun {Lrun})"
        assert lib.pcad_last_error(None), why
        assert all(untouched(b) for b in bufs.values()), f"{why}: rejected, but a buffer was written"
    # the boundaries themselves are accepted: Lrun = (L+1)/2 (odd L), and Lrun = L with time-parallel segments
    si = scan_inputs(S, 63, E, R, BF16, seed=10)
    run_biscan_ex_ok(lib, si, bc_rows=True, Lrun=32)
    run_biscan_ex_ok(lib, sis[BF16], segments=2, bc_rows=True, Lrun=L)
    print(f"[bounds] biscan_ex: {len(bad)} argument combinations rejected with nothing written; boundaries accepted")


def test_scan_mode_choices_match_hand_derived_values():
    """Needs no device: the Python copies of the forward's scan_segments and Lrun against values worked out by hand."""
    # l20 (E = 768): B = 1, L = 32768 -> 24 CTAs per segment, 24 * 16 = 384 <= 592 slots, 24 * 32 > 592 -> P = 16
    assert scan_segments(768, 2, 32768, 148) == 16
    assert scan_segments(768, 4, 16384, 148) == 8
    assert scan_segments(768, 2, 8192, 148) == 16       # segments of 512 steps, the shortest allowed
    assert scan_segments(768, 2, 1000, 148) == 1        # 500-step segments: too short
    assert scan_segments(768, 2, 2050, 148) == 2        # L / 4 is not an integer
    assert scan_segments(2048, 512, 512, 148) == 1      # bench.py snp: the grid already fills the GPU
    assert scan_segments(2048, 32, 8192, 148) == 1      # bench.py long (B = 16): 1024 CTAs
    assert scan_segments(2048, 2, 65536, 148) == 8
    assert scan_segments(2048, 2, 65536, 8) == 1
    # Lrun = max(p, L-1-p) + 1; valid rows [L - Lrun, Lrun)
    want = {(512, 255): 257, (512, 256): 257, (512, 100): 412, (512, 0): 512, (512, 511): 512,
            (301, 150): 151, (301, 7): 294, (33, 16): 17, (8, 3): 5, (8, 4): 5, (17, 8): 9}
    for (L, p), lrun in want.items():
        assert forward_lrun(L, p) == lrun, (L, p)
        assert (L + 1) // 2 <= lrun <= L
        assert L - lrun <= p < lrun                    # the scored row is a valid row
    assert (301 - forward_lrun(301, 150), forward_lrun(301, 150)) == (150, 151)   # exactly one valid row
    assert forward_lrun(7, 3) == 0                     # windows shorter than 8 are not pruned
    assert forward_lrun(512, 255, P=2) == 0            # nor is a time-parallel scan
    assert forward_lrun(512, -1) == 0


def unit_scan_inputs(S, L, E, dtype, R=8):
    """u = 1 (forward only; the reverse direction's u = 0 contributes nothing), B = C = 1, D = 0, z fixed."""
    td = TD[dtype]
    RP = -(-(R + 2 * NS) // 16) * 16
    u = [torch.ones(S * L, E, dtype=td, device=DEV), torch.zeros(S * L, E, dtype=td, device=DEV)]
    dl = [torch.zeros(S * L, E, dtype=td, device=DEV) for _ in range(2)]
    bc = [torch.zeros(S * L, RP, dtype=td, device=DEV) for _ in range(2)]
    for t in bc:
        t[:, R:R + 2 * NS] = 1.0
    xz = torch.full((S * L, 2 * E), 3.0, dtype=td, device=DEV)
    A = [-torch.ones(E, NS, device=DEV) for _ in range(2)]
    D = [torch.zeros(E, device=DEV) for _ in range(2)]
    bias = [torch.zeros(E, device=DEV) for _ in range(2)]
    return ScanInputs(S, L, E, R, RP, dtype, u, dl, bc, xz, A, D, bias)


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
def test_scan_softplus_sweep(lib, dtype):
    """L = 1: y = 16 softplus(delta + bias) SiLU(3).  The argument sweeps [-40, 40], denser around 0 and around the identity
    threshold 20: delta carries an integer (exact in bf16), the per-channel bias a fraction."""
    S, E = 32, 2048
    si = unit_scan_inputs(S, 1, E, dtype)
    g = gen(7)
    frac = (torch.arange(E, device=DEV, dtype=torch.float64) / E)
    n = S * E
    target = torch.cat([rand(g, n // 2, lo=-40, hi=40), torch.randn(n // 4, generator=g, device=DEV, dtype=torch.float64) * 2,
                        20 + torch.randn(n - n // 2 - n // 4, generator=g, device=DEV, dtype=torch.float64) * 0.5])
    target = target[torch.randperm(n, generator=g, device=DEV)].view(S, E).clamp(-40, 40)
    si.bias[0] = frac.float()
    si.dl[0] = torch.round(target - frac).to(TD[dtype])
    y = run_biscan(lib, si)
    arg = si.dl[0].double() + si.bias[0].double()
    assert float(arg.min()) < -39 and float(arg.max()) > 39 and float(((arg - 20).abs() < 0.5).double().mean()) > 0.1
    ref = 16 * softplus64(arg) * silu64(torch.tensor(3.0, dtype=torch.float64, device=DEV))
    st = Stats().add(y.t, ref, ref.abs(), U_OUT[dtype], 0.0)
    verdict("softplus_f32" if dtype == F32 else "softplus_bf16", f"{n} points in [-40, 40]", ("y", st))


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
def test_scan_decay_sweep(lib, dtype):
    """L = 2, input at t = 0 only: y[1] = 16 delta exp(delta A) SiLU(3) with delta = 22 + s (softplus's identity branch,
    s = 0..7 per sequence) and A per channel, so delta A covers [-119, 0], fp32 underflow included."""
    S, E = 8, 2048
    si = unit_scan_inputs(S, 2, E, dtype)
    a = -torch.linspace(0, 90.0 / 22.0, E, device=DEV, dtype=torch.float64)
    si.A[0] = a.float()[:, None].expand(E, NS).contiguous()
    si.bias[0] = torch.full((E,), 22.0, device=DEV)
    si.dl[0] = torch.arange(S, device=DEV, dtype=torch.float32).repeat_interleave(2)[:, None].expand(S * 2, E).to(TD[dtype]).contiguous()
    si.u[0].view(S, 2, E)[:, 1] = 0
    y = run_biscan(lib, si)
    delta = si.dl[0].double().view(S, 2, E) + 22.0
    dA = delta[:, 1] * si.A[0][:, 0].double()
    g3 = float(silu64(torch.tensor(3.0, dtype=torch.float64)))
    ref = torch.stack((16 * delta[:, 0] * g3, 16 * delta[:, 0] * torch.exp(dA) * g3), dim=1).view(S * 2, E)
    pre = (16 * delta[:, 0] * g3)[:, None, :].expand(S, 2, E).reshape(S * 2, E)
    # the exponent d A is formed in fp32 (2^-24 |dA| absolute -> relative on exp); below 2^-126 results flush to zero
    rel = torch.stack((torch.zeros_like(dA), dA.abs()), dim=1).view(S * 2, E)
    st = Stats().add(y.t, ref, ref.abs() * (1 + rel), U_OUT[dtype], U32, floor=2.0 ** -125 * pre)
    assert float(dA.min()) < -118 and float(dA.max()) == 0.0
    verdict("decay_f32" if dtype == F32 else "decay_bf16", f"{S * E} points, dA in [{float(dA.min()):.0f}, 0]", ("y", st))


# ---- Mamba-2: SSD scan and gated norm ----------------------------------------------------------------------------------
P_HD, N_SSD = 64, 64


def ssd_reference(xbc, dt_raw, A, D, bias, S, L, H):
    """float64 sequential SSD of both directions (reverse direction on its own conv output, same dt row): [(ref, mag)]."""
    E = H * P_HD
    outs = []
    for k in range(2):
        X = xbc[k]
        x = X[:, :E].double().view(S, L, H, P_HD)
        Bm = X[:, E:E + N_SSD].double().view(S, L, N_SSD)
        Cm = X[:, E + N_SSD:E + 2 * N_SSD].double().view(S, L, N_SSD)
        dt = softplus64(dt_raw[:, :H].double().view(S, L, H) + bias[k].double())
        Ak, Dk = A[k].double(), D[k].double()
        h = torch.zeros(2, S, H, P_HD, N_SSD, dtype=torch.float64, device=DEV)
        y = torch.empty(2, S, L, H, P_HD, dtype=torch.float64, device=DEV)
        steps = range(L) if k == 0 else range(L - 1, -1, -1)
        for t in steps:
            dA = torch.exp(dt[:, t] * Ak)[:, :, None, None]                             # [S, H, 1, 1]
            xt = torch.stack((x[:, t], x[:, t].abs()))                                  # [2, S, H, P]
            Bt = torch.stack((Bm[:, t], Bm[:, t].abs()))[:, :, None, None, :]           # [2, S, 1, 1, N]
            Ct = torch.stack((Cm[:, t], Cm[:, t].abs()))[:, :, None, None, :]
            h = dA * h + (dt[:, t, :, None] * xt)[..., None] * Bt
            y[:, :, t] = (h * Ct).sum(-1) + xt * torch.stack((Dk, Dk.abs()))[:, None, :, None]
        outs.append((y[0].reshape(S * L, E), y[1].reshape(S * L, E)))
    return outs


@pytest.mark.parametrize("H", [24, 32, 48])
def test_ssd_scan_matches_float64(lib, H):
    """tcgen05 (chunked) and sequential SSD kernels at L = 8192 against float64.  xbc and dt sit in wider rows whose pad
    columns hold 1e4; dt_bias = 25 on one head makes its state forget within a step."""
    S, L = 4, 8192
    E = H * P_HD
    CD = E + 2 * N_SSD
    ld_x = CD + 64
    DIPP = -(-(E + CD + H) // 8) * 8
    g = gen(H)
    xbc = []
    for _ in range(2):
        t = randn(g, S * L, ld_x, dtype=torch.bfloat16)
        t[:, E:CD] = (t[:, E:CD].float() / N_SSD ** 0.5).to(torch.bfloat16)
        t[:, CD:] = 1e4
        xbc.append(t)
    xz = randn(g, S * L, DIPP, dtype=torch.bfloat16, scale=0.5)    # in_proj's output row: z | x | B | C | dt
    dt_off = E + CD
    A = [-torch.exp(rand(g, H, lo=0.0, hi=math.log(16.0))).float() for _ in range(2)]
    D = [randn(g, H, scale=0.1, shift=1.0) for _ in range(2)]
    bias = [checkpoint_dt_bias(g, H) for _ in range(2)]
    bias[0][0] = 25.0
    dt_view = xz[:, dt_off:dt_off + H]
    want = ssd_reference(xbc, dt_view, A, D, bias, S, L, H)
    for label, dtype, impl in (("tcgen05", BF16, 0), ("sequential", BF16, 1), ("sequential", F32, 1)):
        td = TD[dtype]
        xin = [t.to(td) for t in xbc] if dtype == F32 else xbc
        xzin = xz.to(td) if dtype == F32 else xz
        yf, yr = Guarded(S * L, E, td), Guarded(S * L, E, td)
        ok(lib, lib.pcad_op_ssd_scan(vp(xin[0]), vp(xin[1]), ld_x, vp(xzin, dt_off), DIPP, vp(A[0]), vp(D[0]), vp(bias[0]),
                                     vp(A[1]), vp(D[1]), vp(bias[1]), yf.ptr, yr.ptr, S, L, H, dtype, impl, stream()))
        torch.cuda.synchronize()
        assert_guards(f"ssd {label}", y_f=yf, y_r=yr)
        if dtype == BF16:
            u_out, u_acc = U_OUT[BF16], 2.0 ** -8     # tcgen05: intra-chunk weights and carried states pass through bf16
        else:
            u_out, u_acc = U32, N_SSD * U32
        # the head with dt_bias = 25 forgets within a step: where its x is zero the exact output is a carried state of order
        # 1e-68, below the smallest normal number 2^-126, and comes back as zero
        sts = [(f"y_{'fr'[k]}", Stats().add(got.t, want[k][0], want[k][1], u_out, u_acc, floor=2.0 ** -126))
               for k, got in enumerate((yf, yr))]
        family = "ssd_tc" if impl == 0 else ("ssd_seq_f32" if dtype == F32 else "ssd_seq_bf16")
        verdict(family, f"H={H} S={S} L={L} {label} {td}", *sts)
        del yf, yr, xin, xzin


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("E", [2048, 3072])
def test_gated_norm_sum_matches_float64(lib, E, dtype):
    """out = RMSNorm(y_f SiLU(z)) w_f + RMSNorm(y_r SiLU(z)) w_r with z the first E columns of in_proj's row (ldz = DIPP)."""
    td = TD[dtype]
    H = E // 64
    DIPP = -(-(2 * E + 128 + H) // 8) * 8
    rows = M_RAGGED
    g = gen(E)
    yf = randn(g, rows, E, dtype=td)
    yr = randn(g, rows, E, dtype=td, scale=3.0)
    yf.mul_(torch.exp(randn(g, rows, 1)).to(td))
    z = randn(g, rows, DIPP, dtype=td)
    wf, wr = randn(g, E, scale=0.3, shift=1.0), randn(g, E, scale=0.3, shift=1.0)
    out = Guarded(rows, E, td)
    eps = 1e-5
    ok(lib, lib.pcad_op_gated_norm_sum(vp(yf), vp(yr), vp(z), DIPP, vp(wf), vp(wr), out.ptr, rows, E, C.c_float(eps), dtype, stream()))
    torch.cuda.synchronize()
    assert_guards("gated_norm_sum", out=out)
    gz = silu64(z[:, :E].double())

    def gn(y, w):
        v = y.double() * gz
        rstd = torch.rsqrt(v.pow(2).mean(-1, keepdim=True) + eps)
        return v * rstd * w.double(), y.double().abs() * rstd * w.double().abs()
    (a, ua), (b, ub) = gn(yf, wf), gn(yr, wr)
    ref, mag = a + b, a.abs() + b.abs()
    # bf16: each direction's normed output is rounded to bf16 before the sum, as in the reference; fp32: row statistics
    u_acc = U_OUT[BF16] if dtype == BF16 else U32 * 64
    floor = 0.0
    if dtype == BF16:
        # the bf16 kernel keeps SiLU(z) as fp16 between its two passes: 2^-11 relative, but below 2^-14 fp16 is subnormal
        # and the gate carries up to 2^-25 absolute error, i.e. 2^-25 |y| rstd |w| per direction
        floor = 2.0 ** -25 * (ua + ub)
    st = Stats().add(out.t, ref, mag, U_OUT[dtype], u_acc, floor=floor)
    verdict("gnorm_f32" if dtype == F32 else "gnorm_bf16", f"rows={rows} E={E} ldz={DIPP}", ("out", st))


# ---- embedding, final norm, RC LM head and hidden taps (a model without layers) -----------------------------------------
EMB_KEY = "caduceus.backbone.embeddings.word_embeddings.embedding.weight"
HEAD_KEY = "lm_head.lm_head.weight"
NORM_KEY = "caduceus.backbone.norm_f.weight"
HEAD_ROWS = 8192   # rows per float64 chunk


def bf16_exact(t):
    return t.to(torch.bfloat16).float()


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("B,L", [(256, 512), (16, 8192)], ids=["snp", "long"])
@pytest.mark.parametrize("name", LARGEST)
def test_embedding_norm_and_rc_head_match_float64(cuda_device, name, B, L, dtype):
    """embed -> final norm -> RC LM head at the benchmark shapes, through the model with n_layer = 0, so every output is the
    engine's: hidden_states[-1] = [RMSNorm(emb[id]) w | flip_channels(RMSNorm(emb[comp[id]]) w)] against float64 (the RC half
    carries the complement map, the sequence flip and the channel flip), the logits against float64 of the RC head applied to
    the engine's own hidden output, and every scoring / tap entry point against the matching slice, bit for bit.  Weights are
    bf16-representable, so both dtypes see the same numbers; the ids cover all eight (PAD, mask, N, a, c, g, t, 7)."""
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    from plantcaduceus_b200.tokenizer import CharDNATokenizer
    import dataclasses
    import numpy as np
    cfg = dataclasses.replace(preset(name), n_layer=0)
    d, V = cfg.d_model, cfg.vocab_size
    g = torch.Generator().manual_seed(d + L + dtype)
    sd = {EMB_KEY: bf16_exact(torch.randn(V, d, generator=g) * torch.exp(torch.randn(V, 1, generator=g))),
          HEAD_KEY: bf16_exact(torch.randn(V, d, generator=g) * d ** -0.5),
          NORM_KEY: bf16_exact(torch.randn(d, generator=g) * 0.3 + 1.0)}
    model = CaduceusForMaskedLM.from_pretrained(sd, config=cfg, torch_dtype=TD[dtype]).to(cuda_device)
    tok = CharDNATokenizer()
    acgt = [tok.get_vocab()[c] for c in "acgt"]
    # ASCII windows with upper- and lower-case bases and N, masked at token_idx as the score-window calls mask them; then
    # PAD and id 7 (which no byte maps to) at a few other positions.  Without a layer every position's outputs depend on its
    # own id only, so the score-window calls still see the same inputs at token_idx.
    token_idx = L // 2 - 1
    ascii_ = torch.tensor(list(b"ACGTNacgtn"), dtype=torch.uint8)[torch.randint(0, 10, (B, L), generator=g)]
    lut = torch.as_tensor(np.asarray(tok.lut, dtype=np.uint8))
    ids = lut[ascii_.long()].clone()
    ids[:, token_idx] = tok.mask_token_id
    ids.view(-1)[torch.randperm(B * L, generator=g)[:B * L // 16]] = torch.tensor([0, 7], dtype=torch.uint8).repeat(B * L // 32)
    ids[:, token_idx] = tok.mask_token_id
    assert set(ids.unique().tolist()) == set(range(V))
    ids_dev = ids.to(cuda_device)
    out = model(input_ids=ids_dev.long(), output_hidden_states=True)
    logits, hid = out.logits, out.hidden_states[-1]
    assert logits.shape == (B, L, V) and hid.shape == (B, L, 2 * d)
    # float64 reference rows, one per id: RMSNorm(emb[v]) w, and the RC half flip_channels(RMSNorm(emb[comp[v]]) w)
    comp = torch.tensor([cfg.complement_map.get(i, i) for i in range(V)], device=DEV)
    emb = sd[EMB_KEY].double().to(DEV)
    normed = emb * torch.rsqrt(emb.pow(2).mean(-1, keepdim=True) + cfg.norm_epsilon) * sd[NORM_KEY].double().to(DEV)
    table = torch.cat((normed, normed[comp].flip(-1)), dim=1)                        # [V, 2d]
    W = sd[HEAD_KEY].double().to(DEV)
    Wc = W[comp]
    ids_flat, hid_flat, lg_flat = ids_dev.view(-1).long(), hid.view(B * L, 2 * d), logits.view(B * L, V)
    sh, sl = Stats(), Stats()
    for r0 in range(0, B * L, HEAD_ROWS):
        r1 = min(B * L, r0 + HEAD_ROWS)
        ref = table[ids_flat[r0:r1]]
        sh.add(hid_flat[r0:r1], ref, ref.abs(), U_OUT[dtype], U32 * d, row0=r0)
        hf, hr = hid_flat[r0:r1, :d].double(), hid_flat[r0:r1, d:].flip(-1).double()
        ref = hf @ W.t() + hr @ Wc.t()
        mag = hf.abs() @ W.abs().t() + hr.abs() @ Wc.abs().t()
        sl.add(lg_flat[r0:r1], ref, mag, U32, U32 * 2 * d, row0=r0)
        del ref, mag, hf, hr
    case = f"{name} n_layer=0 B={B} L={L} {TD[dtype]}"
    verdict("norm_f32" if dtype == F32 else "norm_bf16", case, ("hidden", sh))
    verdict("head", case, ("logits", sl))
    # the entry points against slices of the full outputs
    b_idx = torch.arange(B, device=DEV)[:, None]
    pos = torch.randint(0, L, (B, 5), generator=g).to(DEV, torch.int32)
    pos[:, 0], pos[:, 1], pos[:, 2] = 0, L - 1, token_idx
    acgt_dev = torch.tensor(acgt, device=DEV)
    want4 = logits[:, token_idx][:, acgt_dev]
    checks = {
        "hidden_at": (model.hidden_at(ids_dev, pos), hid[b_idx, pos.long()]),
        "score_masked": (model.score_masked(ids_dev, pos), logits[b_idx, pos.long()][..., acgt_dev]),
        "score_masked_at": (model.score_masked(ids_dev, token_idx)[:, 0], want4),
        "score_windows_host": (model.score_windows_host(ascii_.numpy(), token_idx).to(DEV), want4),
        "score_windows_device": (model.score_windows_device(ascii_.to(cuda_device), token_idx), want4),
    }
    torch.cuda.synchronize()
    bad = [k for k, (got, want) in checks.items() if not torch.equal(got, want)]
    print(f"[bounds] {'entry points':14s} {case}: {', '.join(checks)} bit-identical to the full outputs: {not bad}")
    assert not bad, f"{case}: {bad} differ from the matching slice of the full forward"


# ---- the checkers can fail ---------------------------------------------------------------------------------------------
def test_checkers_reject_wrong_outputs(lib):
    """Each checker above, fed a copy of a real kernel output with one deliberate error, rejects it.  CPU-side edits of
    tensors only: nothing is provoked on the GPU."""
    # GEMM: the last K block's contribution removed from one 128-row tile
    call = next(c for c in gemm_calls("PlantCaduceus_l32") if c.name == "in_proj")
    call = Call("linear", "in_proj", N=call.N, K=call.K, lda=call.lda, ldw=call.ldw, ldc=call.ldc)
    M = M_RAGGED
    g = gen(1)
    A, W = make_gemm_operands(g, call, M)
    out = Guarded(M, call.N, torch.bfloat16, ld=call.ldc + PAD)
    ok(lib, lib.pcad_op_linear(vp(A), vp(W), out.ptr, M, call.N, call.K, call.lda, call.ldw, out.ld, BF16, stream()))
    torch.cuda.synchronize()
    st, _ = gemm_reference_stats(out.t, A, W, call.K)
    assert not rejects("gemm", st), st.ratio
    bad = out.t.clone()
    r0, k0 = 128 * 17, call.K - 64
    last = A[r0:r0 + 128, k0:call.K].double() @ W[:, k0:call.K].double().t()
    bad[r0:r0 + 128] = (bad[r0:r0 + 128].double() - last).to(torch.bfloat16)
    st_bad, _ = gemm_reference_stats(bad, A, W, call.K)
    print(f"[bounds] self-check gemm: dropped K block -> max err/unit {st_bad.ratio:.4g} (k = {K['gemm']})")
    assert rejects("gemm", st_bad)
    # guard band: one sentinel byte changed, before the output, after it, and in a pad column
    assert out.intact()
    for where in (out.start - 1, out.start + out.nbytes + 5, out.start + call.N * 2):
        saved = out.raw[where].clone()
        out.raw[where] ^= 1
        assert not out.intact(), where
        out.raw[where] = saved
    assert out.intact()
    del A, W, out, bad
    # norm: one row scaled by (1 + 2^-7)
    x, r, w, eps, y, ro = run_norm(lib, 4093, 768, BF16, BF16, seed=3)
    sy, _ = norm_stats(y.t, None, x, r, w, eps, BF16, BF16)
    assert not rejects("norm_bf16", sy), sy.ratio
    bad = y.t.clone()
    bad[1234] = (bad[1234].double() * (1 + 2.0 ** -7)).to(torch.bfloat16)
    sb, _ = norm_stats(bad, None, x, r, w, eps, BF16, BF16)
    print(f"[bounds] self-check norm: one row x (1 + 2^-7) -> max err/unit {sb.ratio:.4g} (k = {K['norm_bf16']})")
    assert rejects("norm_bf16", sb)
    # scan: 2^-5 D u SiLU(z) added on one channel
    si = scan_inputs(8, 512, 768, 24, BF16, seed=5)
    yb = run_biscan(lib, si)
    seqs = list(range(8))
    st, ref, mag = scan_stats(yb, si, seqs)
    assert not rejects("scan_bf16", st), st.ratio
    ch = 300
    bad = yb.t.view(8, 512, 768).double().clone()
    extra = 2.0 ** -5 * si.D[0][ch].double() * si.u[0].view(8, 512, 768)[:, :, ch].double() * silu64(si.xz.view(8, 512, 1536)[:, :, 768 + ch].double())
    bad[:, :, ch] += extra
    u_out, u_acc = scan_units(BF16)
    sb = Stats().add(bad.to(torch.bfloat16).view(-1, 768), ref, mag, u_out, u_acc)
    print(f"[bounds] self-check scan: 2^-5 D u SiLU(z) on one channel -> max err/unit {sb.ratio:.4g} (k = {K['scan_bf16']})")
    assert rejects("scan_bf16", sb)
    # early stop one step short of the forward's Lrun at p = 255: a legal call whose valid rows [256, 256) are empty; row 255
    # keeps the forward direction's parked partial.  The checker must pass row 255 at Lrun and reject it at Lrun - 1.
    p = 255
    Lrun = forward_lrun(512, p)
    ref255, mag255 = (t.view(8, 512, 768)[:, p] for t in (ref, mag))
    for lr, wrong in ((Lrun, False), (Lrun - 1, True)):
        y = run_biscan_ex_ok(lib, si, Lrun=lr)["y"]
        st = Stats().add(y.t.view(8, 512, 768)[:, p], ref255, mag255, u_out, u_acc)
        print(f"[bounds] self-check early stop: row {p} at Lrun = {lr} (valid rows [{512 - lr}, {lr})) -> max err/unit {st.ratio:.4g}")
        assert rejects("scan_bf16", st) == wrong, lr
