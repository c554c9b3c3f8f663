"""Pins the oracle's selective scan (and, through it, libpcad's) to the reference's own kernel family.

The reference's scan arithmetic lives in ``mamba-ssm==2.2.2``'s ``selective_scan_cuda`` (SURVEY.md §8c), which is
not importable here.  vLLM ships a port of that very CUDA kernel (``csrc/mamba/mamba_ssm/selective_scan_fwd.cu``,
"adapted from state-spaces/mamba", exposed as ``torch.ops._C.selective_scan_fwd``): same recurrence, same
``delta_softplus`` / ``delta_bias`` / ``D`` / ``z`` semantics.  It is LIBRARY code used here as a checker only: it never
runs on the product path.  Two checks on the GPU box:

* ``oracle.selective_scan_ref`` (the CPU restatement every other parity test leans on) == the mamba_ssm-derived kernel;
* ``pcad_op_biscan`` (fp32 parity mode) == forward kernel call + flipped reverse kernel call, with no oracle in between.

Skipped (not failed) when vLLM's compiled op is missing or refuses the batch-mode call on this build.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import caduceus_oracle as O

pytestmark = pytest.mark.gpu

F32 = 1


def _vllm_scan():
    try:
        from vllm.model_executor.layers.mamba.ops.mamba_ssm import selective_scan_fn
    except Exception as e:  # pragma: no cover - depends on the image
        pytest.skip(f"vLLM selective_scan_fn not importable: {type(e).__name__}: {e}")
    return selective_scan_fn


def _run_vllm(fn, u, delta, A, B, Cm, D, z, bias):
    """u, delta, z: [b, E, L]; B, Cm: [b, N, L] (fp32 CUDA).  Returns gated y [b, E, L]; tries batch mode, then varlen."""
    b, E, L = u.shape
    N = A.shape[1]
    errs = []
    try:
        state = torch.zeros(b, E, N, device=u.device, dtype=u.dtype)
        zz = z.clone().contiguous()
        out = fn(u.clone().contiguous(), state, delta.clone().contiguous(), A, B.contiguous(), Cm.contiguous(), D, zz,
                 bias, delta_softplus=True)
        torch.cuda.synchronize()
        return out
    except Exception as e:
        errs.append(f"batch mode: {type(e).__name__}: {e}")
    try:
        flat = lambda t: t.permute(1, 0, 2).reshape(t.shape[1], b * L).contiguous()   # [b, X, L] -> [X, b*L]
        state = torch.zeros(b, E, N, device=u.device, dtype=u.dtype)
        qsl = torch.arange(0, (b + 1) * L, L, device=u.device, dtype=torch.int32)
        out = fn(flat(u), state, flat(delta), A, flat(B), flat(Cm), D, flat(z), bias, delta_softplus=True,
                 query_start_loc=qsl, cache_indices=torch.arange(b, device=u.device, dtype=torch.int32),
                 has_initial_state=torch.zeros(b, device=u.device, dtype=torch.bool))
        torch.cuda.synchronize()
        return out.reshape(E, b, L).permute(1, 0, 2)
    except Exception as e:
        errs.append(f"varlen mode: {type(e).__name__}: {e}")
    pytest.skip("vLLM selective_scan_fwd refused both call forms: " + " | ".join(errs))


def _inputs(b, E, L, N, seed):
    g = torch.Generator().manual_seed(seed)
    mk = lambda *s: torch.randn(*s, generator=g)
    u, delta, z = mk(b, E, L), mk(b, E, L) * 0.5, mk(b, E, L)
    B, Cm = mk(b, N, L), mk(b, N, L)
    A = -(torch.rand(E, N, generator=g) * 4 + 0.1)
    D = mk(E)
    bias = mk(E) - 3
    bias[0] = 30.0   # exercises the softplus threshold (identity above 20)
    return u, delta, z, B, Cm, A, D, bias


@pytest.mark.parametrize("b,E,L", [(2, 256, 512), (1, 128, 70), (3, 384, 33)])
def test_oracle_scan_matches_mamba_ssm_kernel_port(cuda_device, b, E, L):
    fn = _vllm_scan()
    N = 16
    u, delta, z, B, Cm, A, D, bias = _inputs(b, E, L, N, 7 + L)
    want = O.selective_scan_ref(u, delta, A, B, Cm, D, z, bias)
    dev = lambda t: t.to(cuda_device).contiguous()
    got = _run_vllm(fn, dev(u), dev(delta), dev(A), dev(B), dev(Cm), dev(D), dev(z), dev(bias)).cpu().float()
    scale = want.abs().max().item()
    # fp32 both sides; the CUDA kernel uses exp2f / fast intrinsics and a blocked scan order: 1e-4 relative (north star)
    assert (got - want).abs().max().item() <= 1e-4 * scale + 1e-5


@pytest.mark.parametrize("S,L,E,R", [(2, 512, 256, 24), (1, 70, 128, 8)])
def test_biscan_matches_mamba_ssm_kernel_port(cuda_device, S, L, E, R):
    """pcad_op_biscan (fp32) against two calls of the mamba_ssm-derived kernel: (y_f + flip(y_r)) * SiLU(z) is linear in
    the un-gated outputs, so gating each direction with the same z (the reverse one flipped) and adding is identical."""
    fn = _vllm_scan()
    from plantcaduceus_b200 import _lib
    lib = _lib.load()
    N = 16
    RP = (R + 2 * N + 15) // 16 * 16
    g = torch.Generator().manual_seed(S * 100 + L)
    mk = lambda *s: torch.randn(*s, generator=g)
    u = [mk(S * L, E) for _ in range(2)]
    dl = [mk(S * L, E) * 0.5 for _ in range(2)]
    bc = [mk(S * L, RP) for _ in range(2)]
    xz = mk(S * L, 2 * E)
    A = [-(torch.rand(E, N, generator=g) * 4 + 0.1) for _ in range(2)]
    D = [mk(E) for _ in range(2)]
    bias = [mk(E) - 3 for _ in range(2)]
    dev = lambda t: t.to(cuda_device).contiguous()
    u_d, dl_d, bc_d, xz_d = [dev(t) for t in u], [dev(t) for t in dl], [dev(t) for t in bc], dev(xz)
    A_d, D_d, b_d = [dev(t) for t in A], [dev(t) for t in D], [dev(t) for t in bias]
    y = torch.full((S * L, E), float("nan"), device=cuda_device)
    ptr = lambda t: C.c_void_p(t.data_ptr())
    z_ptr = C.c_void_p(xz_d.data_ptr() + E * 4)
    rc = lib.pcad_op_biscan(ptr(u_d[0]), ptr(dl_d[0]), ptr(bc_d[0]), ptr(u_d[1]), ptr(dl_d[1]), ptr(bc_d[1]), RP, R, z_ptr,
                            2 * E, ptr(A_d[0]), ptr(D_d[0]), ptr(b_d[0]), ptr(A_d[1]), ptr(D_d[1]), ptr(b_d[1]), ptr(y),
                            S, L, E, F32, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.pcad_last_error(None)
    torch.cuda.synchronize()

    to_bel = lambda t, w: t.reshape(S, L, w).transpose(1, 2).contiguous()   # [S*L, w] -> [S, w, L]
    z = to_bel(xz_d[:, E:], E)
    total = None
    for k in range(2):
        uu, dd = to_bel(u_d[k], E), to_bel(dl_d[k], E)
        Bm, Cm = to_bel(bc_d[k][:, R:R + N], N), to_bel(bc_d[k][:, R + N:R + 2 * N], N)
        zz = z
        if k == 1:
            uu, dd, Bm, Cm, zz = uu.flip(-1), dd.flip(-1), Bm.flip(-1), Cm.flip(-1), z.flip(-1)
        yk = _run_vllm(fn, uu, dd, A_d[k], Bm, Cm, D_d[k], zz, b_d[k]).float()
        if k == 1:
            yk = yk.flip(-1)
        total = yk if total is None else total + yk
    want = total.transpose(1, 2).reshape(S * L, E)
    assert not torch.isnan(y).any()
    scale = want.abs().max().item()
    assert (y - want).abs().max().item() <= 1e-4 * scale + 1e-5


# ---- fused add + RMSNorm against vLLM's CUDA kernel (library code, checker only) ---------------------------------------
# (The conv is NOT pinned to vLLM: its causal_conv1d_fn is a Triton re-implementation with a continuous-batching calling
# convention, not a port of the causal-conv1d CUDA kernel, and called standalone on the GPU box -- with or without a
# hand-built program table -- it leaves most of its output unwritten (zeros / NaN; tried in rounds 2a and 2b, three
# call forms).  The conv is pinned instead, together with the whole mixer, by transformers' MambaMixer / Mamba2Mixer in
# tests/test_oracle.py, and the engine's kernel by F.conv1d in tests/test_ops_gpu.py::test_conv_silu_both_directions.)
@pytest.mark.parametrize("rows,d", [(300, 384), (64, 1024)])
def test_add_rmsnorm_matches_vllm_fused_add_rms_norm(cuda_device, rows, d):
    """pcad_op_add_rmsnorm (fp32) == torch.ops._C.fused_add_rms_norm (in place: residual <- x + residual,
    x <- RMSNorm(residual) * w), and the oracle's rms_norm_add == both."""
    try:
        import vllm._custom_ops as vops  # noqa: F401
        op = torch.ops._C.fused_add_rms_norm
    except Exception as e:  # pragma: no cover
        pytest.skip(f"vLLM fused_add_rms_norm not available: {type(e).__name__}: {e}")
    from plantcaduceus_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(rows + d)
    x = torch.randn(rows, d, generator=g).to(cuda_device)
    res = torch.randn(rows, d, generator=g).to(cuda_device)
    w = (1 + 0.5 * torch.randn(d, generator=g)).to(cuda_device)
    y = torch.empty_like(x)
    res_out = torch.empty_like(x)
    ptr = lambda t: C.c_void_p(t.data_ptr())
    rc = lib.pcad_op_add_rmsnorm(ptr(x), ptr(res), ptr(w), ptr(y), ptr(res_out), rows, d, C.c_float(1e-5), F32, F32,
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.pcad_last_error(None)
    xi, ri = x.clone(), res.clone()
    try:
        op(xi, ri, w, 1e-5)
        torch.cuda.synchronize()
    except Exception as e:
        pytest.skip(f"fused_add_rms_norm refused the call: {type(e).__name__}: {e}")
    assert (res_out - ri).abs().max().item() <= 1e-6
    assert (y - xi).abs().max().item() <= 1e-5 * max(1.0, xi.abs().max().item())
    oy, ores = O.rms_norm_add(x.cpu(), res.cpu(), w.cpu(), 1e-5, True)
    assert (oy - xi.cpu()).abs().max().item() <= 1e-5 * max(1.0, xi.abs().max().item())
    assert (ores - ri.cpu()).abs().max().item() <= 1e-6


def test_probe_reference_dependencies(cuda_device):
    """Reports whether the reference's own arithmetic packages are importable next to the GPU (SURVEY.md App. A open items
    4, 5, 8 can only be settled against them).  When they are, diff the oracle's mixer against mamba_ssm's Mamba.forward."""
    found = {}
    for mod in ("mamba_ssm", "causal_conv1d"):
        try:
            m = __import__(mod)
            found[mod] = getattr(m, "__version__", "present")
        except Exception as e:
            found[mod] = f"absent ({type(e).__name__})"
    print(found)
    if not all(isinstance(v, str) and not v.startswith("absent") for v in found.values()):
        pytest.skip(f"reference dependencies not importable here: {found}")
    from mamba_ssm.modules.mamba_simple import Mamba
    d = 128
    m = Mamba(d_model=d, d_state=16, d_conv=4, expand=2).to(cuda_device).float()
    p = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    u = torch.randn(2, 64, d)
    want = m(u.to(cuda_device)).cpu()
    got = O.mamba_mixer(u, p)
    assert (got - want).abs().max().item() <= 1e-4 * want.abs().max().item()
