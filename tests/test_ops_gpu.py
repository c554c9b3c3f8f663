"""Per-operator parity of libpcad's sm_100a kernels (through the C ABI) against plain torch / the oracle."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import caduceus_oracle as O

pytestmark = pytest.mark.gpu

BF16, F32 = 0, 1


@pytest.fixture(scope="module")
def lib(cuda_device):
    from plantcaduceus_b200 import _lib
    return _lib.load()


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def check(lib, rc):
    assert rc == 0, lib.pcad_last_error(None)


@pytest.mark.parametrize("M,N,K", [
    (128, 256, 64), (256, 256, 128), (1024, 1536, 384), (2048, 4096, 1024), (1024, 1024, 2048),
    (1000, 96, 2048), (1024, 64, 768), (520, 80, 1536), (1024, 2048, 64), (1024, 768, 24), (77, 384, 768),
    (128, 8, 64), (4096, 3072, 768),
    # CTA-pair (cta_group::2) kernel: N % 256 == 0 and K >= 256, with M tails on either CTA of the last pair
    (256, 256, 256), (257, 512, 256), (383, 256, 320), (129, 1024, 1024), (5000, 2048, 512),
])
def test_linear_bf16_tcgen05(lib, cuda_device, M, N, K):
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, generator=g).to(cuda_device, torch.bfloat16)
    W = (torch.randn(N, K, generator=g) / K ** 0.5).to(cuda_device, torch.bfloat16)
    Cout = torch.full((M, N), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    check(lib, lib.pcad_op_linear(ptr(A), ptr(W), ptr(Cout), M, N, K, K, K, N, BF16, stream()))
    torch.cuda.synchronize()
    want = A.float() @ W.float().t()
    err = (Cout.float() - want).abs().max().item()
    # fp32 accumulation, one bf16 rounding of the result: |err| <= 2^-9 * |want| + accumulation noise
    tol = 2 ** -8 * want.abs().max().item() + 1e-3
    assert err <= tol, (err, tol)


@pytest.mark.parametrize("M,N,K", [(512, 1024, 2048), (300, 384, 768), (128, 128, 64), (77, 256, 256)])
def test_linear_residual_and_rowscale_epilogues(lib, cuda_device, M, N, K):
    """out_proj with the residual add + row sum of squares, and in_proj with the RMSNorm row scale, == the separate
    add+RMSNorm followed by the GEMM (up to where the bf16 roundings sit)."""
    g = torch.Generator().manual_seed(M * 3 + N)
    A = torch.randn(M, K, generator=g).to(cuda_device, torch.bfloat16)
    W = (torch.randn(N, K, generator=g) / K ** 0.5).to(cuda_device, torch.bfloat16)
    resid = torch.randn(M, N, generator=g).to(cuda_device, torch.bfloat16)
    resid_io = resid.clone()
    parts = lib.pcad_op_sumsq_parts(N)
    sumsq = torch.full((M, parts), float("nan"), device=cuda_device)
    check(lib, lib.pcad_op_linear_residual(ptr(A), ptr(W), ptr(resid_io), ptr(resid_io), ptr(sumsq), M, N, K, K, K, N, BF16, stream()))
    torch.cuda.synchronize()
    want = A.float() @ W.float().t() + resid.float()
    assert (resid_io.float() - want).abs().max().item() <= 2 ** -8 * want.abs().max().item() + 1e-3
    want_ss = want.pow(2).sum(-1)
    assert torch.allclose(sumsq.sum(-1), want_ss, rtol=1e-4, atol=1e-3)
    # row scale: C = (X Wn^T) * rsqrt(mean(X^2) + eps), sums of squares taken from above
    d = N
    X = resid_io                                   # [M, d] plays the residual stream
    w_norm = (1 + 0.1 * torch.randn(d, generator=g)).to(cuda_device)
    W2 = (torch.randn(2 * d, d, generator=g) / d ** 0.5).to(cuda_device, torch.bfloat16)
    W2s = (W2.float() * w_norm[None, :]).to(torch.bfloat16)
    out = torch.full((M, 2 * d), float("nan"), device=cuda_device, dtype=torch.bfloat16)
    eps = 1e-5
    check(lib, lib.pcad_op_linear_rowscale(ptr(X), ptr(W2s), ptr(sumsq), parts, C.c_float(eps), ptr(out), M, 2 * d, d, d, d, 2 * d, BF16, stream()))
    torch.cuda.synchronize()
    normed = (want * torch.rsqrt(want.pow(2).mean(-1, keepdim=True) + eps) * w_norm[None, :])
    ref = normed @ W2.float().t()
    err = (out.float() - ref).abs().max().item()
    assert not torch.isnan(out.float()).any()
    assert err <= 2 ** -6 * ref.abs().max().item() + 2e-3, err


def test_linear_bf16_strided(lib, cuda_device):
    """A taken as the first K columns of a wider matrix (dt_proj reads dt out of [T, R+2N])."""
    M, N, K, lda = 512, 768, 24, 64
    g = torch.Generator().manual_seed(1)
    Abig = torch.randn(M, lda, generator=g).to(cuda_device, torch.bfloat16)
    W = torch.randn(N, K, generator=g).to(cuda_device, torch.bfloat16)
    Cout = torch.empty(M, N, device=cuda_device, dtype=torch.bfloat16)
    check(lib, lib.pcad_op_linear(ptr(Abig), ptr(W), ptr(Cout), M, N, K, lda, K, N, BF16, stream()))
    torch.cuda.synchronize()
    want = Abig[:, :K].float() @ W.float().t()
    assert (Cout.float() - want).abs().max().item() <= 2 ** -8 * want.abs().max().item() + 1e-3


@pytest.mark.parametrize("M,N,K", [(130, 70, 33), (512, 1536, 384), (64, 56, 768)])
def test_linear_f32(lib, cuda_device, M, N, K):
    g = torch.Generator().manual_seed(5)
    A = torch.randn(M, K, generator=g).to(cuda_device)
    W = torch.randn(N, K, generator=g).to(cuda_device)
    Cout = torch.empty(M, N, device=cuda_device)
    check(lib, lib.pcad_op_linear(ptr(A), ptr(W), ptr(Cout), M, N, K, K, K, N, F32, stream()))
    torch.cuda.synchronize()
    want = (A.double() @ W.double().t()).float()
    assert torch.allclose(Cout, want, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("dtype,res_dtype", [(F32, F32), (BF16, F32), (BF16, BF16)])
@pytest.mark.parametrize("d", [384, 1024, 128])
def test_add_rmsnorm(lib, cuda_device, dtype, res_dtype, d):
    rows = 333
    td = torch.float32 if dtype == F32 else torch.bfloat16
    tr = torch.float32 if res_dtype == F32 else torch.bfloat16
    g = torch.Generator().manual_seed(d)
    x = torch.randn(rows, d, generator=g).to(cuda_device, td)
    r = torch.randn(rows, d, generator=g).to(cuda_device, tr)
    w = (1 + 0.1 * torch.randn(d, generator=g)).to(cuda_device)
    y = torch.empty_like(x)
    r_out = torch.empty_like(r)
    check(lib, lib.pcad_op_add_rmsnorm(ptr(x), ptr(r), ptr(w), ptr(y), ptr(r_out), rows, d, 1e-5, dtype, res_dtype, stream()))
    torch.cuda.synchronize()
    want_y, want_r = O.rms_norm_add(x.cpu(), r.cpu(), w.cpu().to(td), 1e-5, res_dtype == F32, prenorm=True)
    assert want_r.dtype == tr
    if dtype == F32:
        assert torch.allclose(y.cpu(), want_y, rtol=1e-5, atol=1e-6)
        assert torch.equal(r_out.cpu(), want_r)
    else:
        assert (y.cpu().float() - want_y.float()).abs().max() <= 2 ** -7 * want_y.float().abs().max()
        assert (r_out.cpu().float() - want_r.float()).abs().max() <= 2 ** -8 * want_r.float().abs().max()
    # first layer: no residual in, prenorm=False: no residual out
    y2 = torch.empty_like(x)
    check(lib, lib.pcad_op_add_rmsnorm(ptr(x), None, ptr(w), ptr(y2), None, rows, d, 1e-5, dtype, res_dtype, stream()))
    torch.cuda.synchronize()
    want2 = O.rms_norm_add(x.cpu(), None, w.cpu().to(td), 1e-5, res_dtype == F32, prenorm=False)
    tol = 1e-5 if dtype == F32 else 2 ** -7 * want2.float().abs().max().item()
    assert (y2.cpu().float() - want2.float()).abs().max() <= tol


@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("S,L,E", [(3, 512, 768), (2, 70, 256), (1, 5, 128), (2, 1, 128)])
def test_conv_silu_both_directions(lib, cuda_device, dtype, S, L, E):
    td = torch.float32 if dtype == F32 else torch.bfloat16
    g = torch.Generator().manual_seed(L)
    xz = torch.randn(S * L, 2 * E, generator=g).to(cuda_device, td)   # conv reads the x half, pitch 2E
    wf, wr = torch.randn(E, 4, generator=g).to(cuda_device), torch.randn(E, 4, generator=g).to(cuda_device)
    bf_, br_ = torch.randn(E, generator=g).to(cuda_device), torch.randn(E, generator=g).to(cuda_device)
    of = torch.empty(S * L, E, device=cuda_device, dtype=td)
    orv = torch.empty_like(of)
    check(lib, lib.pcad_op_conv_silu(ptr(xz), 2 * E, ptr(wf), ptr(bf_), ptr(wr), ptr(br_), ptr(of), ptr(orv), S, L, E, dtype, stream()))
    torch.cuda.synchronize()
    x = xz[:, :E].float().cpu().reshape(S, L, E).transpose(1, 2)      # [S, E, L]

    def ref(xx, w, b):
        return F.silu(F.conv1d(xx, w.cpu()[:, None, :], b.cpu(), padding=3, groups=E)[..., :L])
    want_f = ref(x, wf, bf_).transpose(1, 2).reshape(S * L, E)
    want_r = ref(x.flip(-1), wr, br_).flip(-1).transpose(1, 2).reshape(S * L, E)
    tol = dict(rtol=1e-5, atol=1e-5) if dtype == F32 else dict(rtol=2 ** -7, atol=2e-3)
    assert torch.allclose(of.cpu().float(), want_f, **tol)
    assert torch.allclose(orv.cpu().float(), want_r, **tol)


@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("S,L,E,R", [(2, 512, 256, 24), (3, 64, 128, 8), (2, 37, 128, 8), (1, 1, 128, 8), (2, 16, 128, 64), (1, 33, 384, 24),
                                     (1, 40, 128, 8), (1, 47, 200, 8)])
def test_biscan(lib, cuda_device, dtype, S, L, E, R):
    N = 16
    td = torch.float32 if dtype == F32 else torch.bfloat16
    g = torch.Generator().manual_seed(S * 100 + L)
    RP = (R + 2 * N + 15) // 16 * 16
    mk = lambda *shape: torch.randn(*shape, generator=g)
    u = [mk(S * L, E).to(td) for _ in range(2)]
    dl = [(mk(S * L, E) * 0.5).to(td) for _ in range(2)]
    bc = [mk(S * L, RP).to(td) for _ in range(2)]
    xz = mk(S * L, 2 * E).to(td)
    A = [-(torch.rand(E, N, generator=g) * 4 + 0.1) for _ in range(2)]
    D = [mk(E) for _ in range(2)]
    bias = [mk(E) - 3 for _ in range(2)]
    bias[0][0] = 30.0   # exercises the softplus threshold branch
    dev = lambda t: t.to(cuda_device).contiguous()
    dl_in = dl
    u_d, dl_d, bc_d = [dev(t) for t in u], [dev(t) for t in dl_in], [dev(t) for t in bc]
    xz_d = dev(xz)
    A_d, D_d, b_d = [dev(t) for t in A], [dev(t) for t in D], [dev(t) for t in bias]
    y = torch.full((S * L, E), float("nan"), device=cuda_device, dtype=td)
    z_ptr = C.c_void_p(xz_d.data_ptr() + E * xz_d.element_size())
    check(lib, lib.pcad_op_biscan(ptr(u_d[0]), ptr(dl_d[0]), ptr(bc_d[0]), ptr(u_d[1]), ptr(dl_d[1]), ptr(bc_d[1]),
                                  RP, R, z_ptr, 2 * E, ptr(A_d[0]), ptr(D_d[0]), ptr(b_d[0]),
                                  ptr(A_d[1]), ptr(D_d[1]), ptr(b_d[1]), ptr(y), S, L, E, dtype, stream()))
    torch.cuda.synchronize()

    # oracle: two selective_scan_ref calls (fp32 maths on the same rounded inputs), reverse one flipped
    def to_bel(t, width):   # [S*L, width] -> [S, width, L]
        return t.float().reshape(S, L, width).transpose(1, 2)
    ones = torch.ones(S, E, L)   # z gate applied after the sum below, so pass SiLU(z)=... via explicit gate
    ys = []
    for k in range(2):
        uu, dd = to_bel(u[k], E), to_bel(dl[k], E)
        Bm, Cm = to_bel(bc[k][:, R:R + N], N), to_bel(bc[k][:, R + N:R + 2 * N], N)
        if k == 1:
            uu, dd, Bm, Cm = uu.flip(-1), dd.flip(-1), Bm.flip(-1), Cm.flip(-1)
        # z = large positive => SiLU(z) ~= z; instead compute un-gated by passing z with SiLU(z)=1 is impossible,
        # so call with z=None equivalent: replicate the function body without the gate
        yy = O.selective_scan_ref(uu, dd, A[k], Bm, Cm, D[k], torch.full_like(uu, 1.0), bias[k]) / F.silu(torch.tensor(1.0))
        ys.append(yy.flip(-1) if k == 1 else yy)
    z = to_bel(xz[:, E:], E)
    want = ((ys[0] + ys[1]) * F.silu(z)).transpose(1, 2).reshape(S * L, E)
    got = y.cpu().float()
    assert not torch.isnan(got).any()
    scale = want.abs().max().item()
    if dtype == F32:
        assert (got - want).abs().max().item() <= 2e-5 * scale + 1e-5
    else:
        assert (got - want).abs().max().item() <= 2 ** -6 * scale


@pytest.mark.parametrize("dtype", [F32, BF16])
@pytest.mark.parametrize("S,L,E,R,P", [(1, 512, 128, 8, 4), (2, 1024, 256, 24, 8), (1, 96, 128, 8, 2), (3, 320, 200, 8, 5), (1, 8192, 128, 8, 16)])
def test_biscan_time_parallel_matches_sequential(lib, cuda_device, dtype, S, L, E, R, P):
    """pcad_op_biscan_segmented (P concurrent segments per sequence: zero-state scans -> carry combine -> scans from the carried
    states) against the sequential pcad_op_biscan on the same inputs: the recurrence is linear in the state, so the two differ
    only by fp32 rounding of the carry (fp32: 2e-5 of the output scale; bf16: see below)."""
    N = 16
    td = torch.float32 if dtype == F32 else torch.bfloat16
    g = torch.Generator().manual_seed(S * 100 + L + P)
    RP = (R + 2 * N + 15) // 16 * 16
    mk = lambda *shape: torch.randn(*shape, generator=g)
    dev = lambda t: t.to(cuda_device).contiguous()
    u = [dev(mk(S * L, E).to(td)) for _ in range(2)]
    dl = [dev((mk(S * L, E) * 0.5).to(td)) for _ in range(2)]
    bc = [dev(mk(S * L, RP).to(td)) for _ in range(2)]
    xz = dev(mk(S * L, 2 * E).to(td))
    # slow decays too (|A| dt ~ 1e-3): the carried state matters across every segment
    A = [dev(-(torch.rand(E, N, generator=g) * 4 + 0.01)) for _ in range(2)]
    D = [dev(mk(E)) for _ in range(2)]
    bias = [dev(mk(E) - 4) for _ in range(2)]
    z_ptr = C.c_void_p(xz.data_ptr() + E * xz.element_size())
    y_seq = torch.full((S * L, E), float("nan"), device=cuda_device, dtype=td)
    y_par = torch.full((S * L, E), float("nan"), device=cuda_device, dtype=td)
    check(lib, lib.pcad_op_biscan(ptr(u[0]), ptr(dl[0]), ptr(bc[0]), ptr(u[1]), ptr(dl[1]), ptr(bc[1]), RP, R, z_ptr, 2 * E,
                                  ptr(A[0]), ptr(D[0]), ptr(bias[0]), ptr(A[1]), ptr(D[1]), ptr(bias[1]), ptr(y_seq), S, L, E, dtype, stream()))
    state = torch.full((S * P * 2 * E * 16,), float("nan"), device=cuda_device)
    sumd = torch.full((S * P * 2 * E,), float("nan"), device=cuda_device)
    check(lib, lib.pcad_op_biscan_segmented(ptr(u[0]), ptr(dl[0]), ptr(bc[0]), ptr(u[1]), ptr(dl[1]), ptr(bc[1]), RP, R, z_ptr, 2 * E,
                                            ptr(A[0]), ptr(D[0]), ptr(bias[0]), ptr(A[1]), ptr(D[1]), ptr(bias[1]), ptr(y_par), S, L, E, P,
                                            ptr(state), ptr(sumd), dtype, stream()))
    torch.cuda.synchronize()
    a, b = y_seq.float(), y_par.float()
    assert not torch.isnan(b).any()
    scale = a.abs().max().item()
    if dtype == F32:
        assert (a - b).abs().max().item() <= 2e-5 * scale + 1e-6
    else:
        # bf16: the direction that reaches a position first parks its partial sum in y ROUNDED to bf16; which direction that is
        # depends on where the position lies relative to the middle of the (sub)sequence, so the segmented run rounds a
        # different partial than the sequential one: differences of one bf16 ulp on a sizeable fraction of the outputs
        # (measured: ~17 %), none larger, both equally valid bf16 results.  fp32 above proves the carries themselves exact.
        diff = (a - b).abs()
        assert diff.max().item() <= 2 ** -6 * scale, (diff.max().item(), scale)
        assert diff.mean().item() <= 2 ** -11 * scale, (diff.mean().item(), scale)
    # L not divisible by the segment count is refused
    assert lib.pcad_op_biscan_segmented(ptr(u[0]), ptr(dl[0]), ptr(bc[0]), ptr(u[1]), ptr(dl[1]), ptr(bc[1]), RP, R, z_ptr, 2 * E,
                                        ptr(A[0]), ptr(D[0]), ptr(bias[0]), ptr(A[1]), ptr(D[1]), ptr(bias[1]), ptr(y_par), S, L, E, 7,
                                        ptr(state), ptr(sumd), dtype, stream()) != 0
