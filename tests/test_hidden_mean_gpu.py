"""Mean-pooled hidden states: pcad_op_hidden_mean, pcad_hidden_mean_at_layers and the Python surface over them
(`hidden_mean`, `extract_embeddings(pooling="mean")`).

The pooled mean has one fixed summation order (include/pcad.h): fp32 sums over chunks of PCAD_HIDDEN_MEAN_CHUNK positions
counted from the range's start, each sequential in t, then the chunk partials in chunk order, then one correctly rounded
division.  `mean_np` restates that order with explicit sequential adds (np.cumsum); `mean_emulated` is the same order in
torch, so it runs at production shapes on the device.  Every engine output is compared with them bit for bit.

- Without a device: the emulations against hand-worked sums (rounding ties, cancellation, a range crossing a chunk
  boundary, one-position ranges) and against each other; the range and pooling argument rejection; that the chunk
  partials fit the buffer they borrow; the exports and NULL-handle rejection.
- The operator at the l32 / PlantCAD2-Large widths at B = 256 / L = 512 and B = 16 / L = 8192, and at the l20 width with
  B = 1 / L = 32768, in bf16 and fp32, with full, random, one-position and invalid ranges: bit-identical to the emulation,
  within the a-priori bound of the order against float64, inside guard-banded buffers.
- The engine at every preset in three modes: each entry equals the emulation applied to pcad_forward_taps' entry;
  one-position ranges equal pcad_hidden_at_layers; a window alone equals the same window in a batch; a subset of entries
  equals the same entries of "all"; the launch count shows the early stop.
- The semantics: every pooled entry against the CPU oracle's output_hidden_states averaged in float64."""
import ctypes as C
import os
import re
import time
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from plantcaduceus_b200.configuration import CaduceusConfig, preset
from plantcaduceus_b200.modeling import hidden_mean_ranges
from plantcaduceus_b200.weights import random_init_state_dict
from test_forward_replay_gpu import RAGGED, SNP, LONG, first_difference, hidden_tap, make_ids, two_layers
from test_forward_replay_gpu import budget, lib, switches  # noqa: F401  (fixtures)
from test_kernel_bounds_gpu import ALL_PRESETS, BF16, DEV, F32, LARGEST, TD, Guarded, assert_guards, gen, randn

PCAD_ERR_INVALID = -1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_chunk():
    with open(os.path.join(ROOT, "include", "pcad.h")) as f:
        return int(re.search(r"#define PCAD_HIDDEN_MEAN_CHUNK (\d+)", f.read()).group(1))


P = header_chunk()


# ---- the fixed order, restated -------------------------------------------------------------------------------------------
def mean_np(x, ranges=None, p=None):
    """x float32 [B, L, W], ranges [B, 2] or None -> float32 [B, W], NaN rows for invalid ranges."""
    p = p or P
    B, L, W = x.shape
    out = np.full((B, W), np.nan, dtype=np.float32)
    for b in range(B):
        s, e = (0, L) if ranges is None else (int(ranges[b][0]), int(ranges[b][1]))
        if s < 0 or e > L or s >= e:
            continue
        parts = np.stack([np.cumsum(x[b, t:min(t + p, e)], axis=0, dtype=np.float32)[-1] for t in range(s, e, p)])
        out[b] = np.cumsum(parts, axis=0, dtype=np.float32)[-1] / np.float32(e - s)
    return out


def mean_emulated(x, ranges=None):
    """mean_np's order in torch (elementwise fp32 adds, so exact on any device): x float32 [B, L, W] -> float32 [B, W]."""
    B, L, W = x.shape
    dev = x.device
    if ranges is None:
        s = torch.zeros(B, dtype=torch.long, device=dev)
        e = torch.full((B,), L, dtype=torch.long, device=dev)
    else:
        r = torch.as_tensor(ranges).to(dev, torch.long)
        s, e = r[:, 0], r[:, 1]
    valid = (s >= 0) & (e <= L) & (s < e)
    s, e = torch.where(valid, s, 0), torch.where(valid, e, 1)
    n_chunks = -(-L // P)
    t0 = s[:, None] + torch.arange(n_chunks, device=dev)[None] * P           # [B, n_chunks]
    bi = torch.arange(B, device=dev)[:, None]
    acc = x[bi, t0.clamp(max=L - 1)]                                            # [B, n_chunks, W]
    for i in range(1, P):
        live = t0 + i < e[:, None]
        if not bool(live.any()):
            break
        acc = torch.where(live[..., None], acc + x[bi, (t0 + i).clamp(max=L - 1)], acc)
    nc = (e - s + P - 1) // P
    tot = acc[:, 0]
    for c in range(1, n_chunks):
        tot = torch.where((c < nc)[:, None], tot + acc[:, c], tot)
    out = (tot.double() / (e - s).double()[:, None]).float()   # float64 quotient of two floats, rounded once: correctly rounded
    out[~valid] = float("nan")
    return out


def bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ---- device-free -----------------------------------------------------------------------------------------------------------
def test_chunk_is_stated_in_the_header():
    assert P == 128


def f32(*v):
    return np.array(v, dtype=np.float32)


def test_emulation_matches_hand_worked_sums():
    u = 2.0 ** -24
    # a tie: 1 + 2^-24 rounds to even (1), so the order of the terms decides
    x = f32(1.0, u, u)[None, :, None]
    assert mean_np(x)[0, 0] == np.float32(1.0) / np.float32(3)
    x = f32(u, u, 1.0)[None, :, None]
    assert mean_np(x)[0, 0] == np.float32(1.0 + 2 * u) / np.float32(3)
    # cancellation: 1e8 + 1 == 1e8 in fp32
    assert mean_np(f32(1e8, 1.0, -1e8)[None, :, None])[0, 0] == 0.0
    assert mean_np(f32(1e8, -1e8, 1.0)[None, :, None])[0, 0] == np.float32(1.0) / np.float32(3)
    # a range of 130 positions from s = 5 crosses one chunk boundary: chunk 0 is [5, 133), chunk 1 is [133, 135).  Chunk 0
    # is 2^24 followed by 127 ones, each lost to the tie (2^24 + 1 rounds to 2^24); chunk 1 sums to 2; the total 2^24 + 2 is
    # exact.  Chunks counted from 0 instead ([5, 128) and [128, 135)) would give 2^24 + 7 -> 2^24 + 8.
    L = 200
    x = np.zeros((1, L, 1), dtype=np.float32)
    x[0, 5, 0] = 2.0 ** 24
    x[0, 6:135, 0] = 1.0
    got = mean_np(x, [[5, 135]])[0, 0]
    assert got == np.float32(2.0 ** 24 + 2) / np.float32(130)
    assert got != np.float32(2.0 ** 24 + 8) / np.float32(130)
    assert got != np.float32((2.0 ** 24 + 129) / 130)           # the exact mean: the order is visible
    # one-position ranges return the entry itself, -0.0 included; invalid ranges give NaN and leave other rows alone
    x = np.random.default_rng(0).standard_normal((5, 7, 16)).astype(np.float32)
    x[0, 3, 2] = -0.0
    r = [[3, 4], [0, 1], [6, 7], [2, 2], [-1, 3]]
    got = mean_np(x, r)
    for b in range(3):
        assert (got[b].view(np.int32) == x[b, r[b][0]].view(np.int32)).all()
    assert np.isnan(got[3:]).all()
    for bad in ([[0, 8]], [[5, 4]]):
        assert np.isnan(mean_np(x[:1], bad)).all()


def test_torch_emulation_equals_numpy():
    g = np.random.default_rng(1)
    B, L, W = 9, 3 * P + 17, 24
    x = (g.standard_normal((B, L, W)) * np.exp(g.standard_normal((B, L, 1))) + 0.5).astype(np.float32)
    r = np.array([[0, L], [5, 5 + P], [5, 6 + P], [P - 1, P + 1], [17, L], [3, 4], [L - 1, L], [4, 2], [0, L + 1]])
    for ranges in (None, r):
        want = mean_np(x, ranges)
        got = mean_emulated(torch.from_numpy(x), None if ranges is None else torch.from_numpy(ranges))
        assert bits_equal(got, torch.from_numpy(want)), first_difference(got, torch.from_numpy(want))


def test_ranges_are_checked():
    B, L = 3, 10
    assert torch.equal(hidden_mean_ranges([[0, 10], [2, 3], [9, 10]], B, L), torch.tensor([[0, 10], [2, 3], [9, 10]], dtype=torch.int32))
    assert hidden_mean_ranges(np.array([[0, 1]] * 3, dtype=np.int16), B, L).dtype == torch.int32
    # values outside int32 must not wrap into a valid range: clamped to [-1, L + 1], invalid stays invalid
    r = hidden_mean_ranges(torch.tensor([[2 ** 32 + 1, 2 ** 32 + 3], [-2 ** 40, 5], [0, 2 ** 33]]), B, L)
    assert r.tolist() == [[L + 1, L + 1], [-1, 5], [0, L + 1]]
    for bad in ([[0, 1]] * 2, [[0, 1, 2]] * 3, [0, 1, 2], np.zeros((3, 2), dtype=np.float32), torch.zeros(3, 2, dtype=torch.bool),
                [["a", "b"]] * 3, [[0.5, 1]] * 3, torch.zeros(3, 2, 1, dtype=torch.int32)):
        with pytest.raises(ValueError):
            hidden_mean_ranges(bad, B, L)


def test_extract_embeddings_rejects_bad_pooling():
    from plantcaduceus_b200.embeddings import extract_embeddings
    model = SimpleNamespace(config=SimpleNamespace(n_layer=2, d_model=8))   # rejected before the model is used
    with pytest.raises(ValueError, match="pooling"):
        extract_embeddings(model, None, np.zeros((2, 4), dtype=np.uint8), pooling="max")
    with pytest.raises(ValueError, match="mean"):
        extract_embeddings(model, None, np.zeros((2, 4), dtype=np.uint8), ranges=[[0, 1], [0, 1]])
    with pytest.raises(ValueError, match="ranges"):
        extract_embeddings(model, None, np.zeros((2, 4), dtype=np.uint8), pooling="mean", ranges=[[0, 1]])


@pytest.mark.parametrize("name", ALL_PRESETS)
def test_partials_fit_the_borrowed_buffer(name):
    """The chunk partials (2B ceil(L / P) d floats) go to ws.delta[0], [2BL, E] in the model dtype (E = 2d); no workspace
    is added for them."""
    cfg = preset(name)
    d, E = cfg.d_model, cfg.d_inner
    for B, L in (RAGGED, SNP, LONG, (1, 32768), (1, 1), (3, 1), (2, P + 1)):
        assert 2 * B * -(-L // P) * d * 4 <= 2 * B * L * E * 2, (name, B, L)


def test_exports_and_null_handle():
    from plantcaduceus_b200 import _lib
    lib = _lib.load()
    for name in ("pcad_hidden_mean_at_layers", "pcad_op_hidden_mean"):
        assert name in _lib.EXPORTS and hasattr(lib, name)
    idx = (C.c_int32 * 1)(0)
    p = C.c_void_p(16)
    assert lib.pcad_hidden_mean_at_layers(None, p, None, 1, 1, 1, idx, p, None) == PCAD_ERR_INVALID
    # the operator rejects a bad dtype, null buffers and d not a multiple of 8 before any device work
    assert lib.pcad_op_hidden_mean(p, None, p, p, 1, 1, 8, 2, None) == PCAD_ERR_INVALID
    for rows, scratch, out in ((None, p, p), (p, None, p), (p, p, None)):
        assert lib.pcad_op_hidden_mean(rows, None, scratch, out, 1, 1, 8, BF16, None) == PCAD_ERR_INVALID
    assert lib.pcad_op_hidden_mean(p, None, p, p, 1, 1, 12, BF16, None) == PCAD_ERR_INVALID
    assert lib.pcad_op_hidden_mean(p, None, p, p, -1, 1, 8, BF16, None) == PCAD_ERR_INVALID


# ---- the operator ----------------------------------------------------------------------------------------------------------
def _s():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def range_sets(B, L, seed):
    """{kind: int32 [B, 2] on the device or None}: full (NULL), random, one-position, and valid rows mixed with every kind
    of invalid one."""
    g = torch.Generator().manual_seed(seed)
    s = torch.randint(0, L, (B,), generator=g)
    e = s + 1 + (torch.rand(B, generator=g) * (L - s).double()).long().clamp(max=L - s - 1)
    rnd = torch.stack([s, e], 1)
    one = torch.stack([s, s + 1], 1)
    bad = rnd.clone()
    kinds = torch.tensor([[-1, 1], [0, L + 1], [L // 2, L // 2], [L // 2 + 1, L // 2]])
    for b in range(0, B, 2):
        bad[b] = kinds[(b // 2) % 4]
    return {"full": None, "random": rnd, "one": one, "invalid": bad}


def float64_bound_ratio(got, x, ranges):
    """max over valid elements of |got - mean64| / (((P-1) + (chunks-1) + 1) 2^-24 sum|x| / n)."""
    B, L, _ = x.shape
    worst = 0.0
    for b in range(B):
        s, e = (0, L) if ranges is None else (int(ranges[b, 0]), int(ranges[b, 1]))
        if s < 0 or e > L or s >= e:
            continue
        seg = x[b, s:e].double()
        n = e - s
        ref = seg.sum(0) / n
        bound = ((P - 1) + (-(-n // P) - 1) + 1) * 2.0 ** -24 * seg.abs().sum(0) / n
        err = (got[b].double() - ref).abs()
        assert bool((err <= bound).all()), f"row {b}: err {float(err.max()):.3g} beyond the a-priori bound"
        worst = max(worst, float((err / bound.clamp(min=1e-300)).max()))
    return worst


OP_CASES = ([(name, shape) for name in LARGEST for shape in (SNP, LONG)] + [("PlantCaduceus_l20", (1, 32768))])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("name,shape", OP_CASES, ids=[f"{n}-B{s[0]}-L{s[1]}" for n, s in OP_CASES])
def test_op_hidden_mean_matches_emulation_and_float64(lib, switches, name, shape, dtype):
    d = preset(name).d_model
    B, L = shape
    g = gen(B * 7 + L)
    # rows with a per-row scale and an offset, so the means are not near zero and Σ|x| / n is not the mean's magnitude
    rows = (randn(g, 2 * B * L, d) * torch.exp(randn(g, 2 * B * L, 1)) + randn(g, 1, d)).to(TD[dtype])
    x = hidden_tap(rows.float(), B, L, d)                                   # hidden_states layout, exact in fp32
    n_chunks = -(-L // P)
    out, scratch = Guarded(B, 2 * d, torch.float32), Guarded(B * n_chunks, 2 * d, torch.float32)
    ratios = {}
    for kind, r in range_sets(B, L, seed=L).items():
        rd = r.to(DEV, torch.int32).contiguous() if r is not None else None
        rc = lib.pcad_op_hidden_mean(C.c_void_p(rows.data_ptr()), C.c_void_p(rd.data_ptr()) if rd is not None else None,
                                     scratch.ptr, out.ptr, B, L, d, dtype, _s())
        assert rc == 0, lib.pcad_last_error(None)
        torch.cuda.synchronize()
        assert_guards(f"{name} {kind}", out=out, scratch=scratch)
        want = mean_emulated(x, rd)
        assert bits_equal(out.t, want), f"{name} B={B} L={L} {kind}: {first_difference(out.t, want)}"
        if kind == "invalid":
            bad = torch.tensor([b % 2 == 0 for b in range(B)], device=DEV)
            assert bool(torch.isnan(out.t[bad]).all()) and not bool(torch.isnan(out.t[~bad]).any())
            assert bits_equal(out.t[~bad], mean_emulated(x[~bad], rd[~bad]))
        if kind == "one":
            assert torch.equal(out.t, x[torch.arange(B, device=DEV), rd[:, 0].long()])
        ratios[kind] = float64_bound_ratio(out.t, x, rd)
    print(f"[mean] op {name} d={d} B={B} L={L} {'f32' if dtype == F32 else 'bf16'}: bit-identical to the order; largest "
          f"err / a-priori bound " + ", ".join(f"{k} {v:.3g}" for k, v in ratios.items()))


# ---- the engine ------------------------------------------------------------------------------------------------------------
def pooled_guarded(lib, model, ids_u8, ranges, layers):
    """pcad_hidden_mean_at_layers into a guard-banded buffer: float32 [len(layers), B, 2d]."""
    B, L = ids_u8.shape
    w = 2 * model.config.d_model
    out = Guarded(len(layers) * B, w, torch.float32)
    idx = (C.c_int32 * len(layers))(*layers)
    rc = lib.pcad_hidden_mean_at_layers(model._handle, C.c_void_p(ids_u8.data_ptr()),
                                        C.c_void_p(ranges.data_ptr()) if ranges is not None else None, B, L, len(layers), idx,
                                        out.ptr, _s())
    assert rc == 0, lib.pcad_last_error(model._handle)
    torch.cuda.synchronize()
    assert_guards("pcad_hidden_mean_at_layers", out=out)
    return out.t.view(len(layers), B, w).clone()


def engine_ranges(B, L, seed):
    """Random ranges, some crossing chunk boundaries, some one position long, one invalid."""
    r = range_sets(B, L, seed)["random"].clone()
    r[0] = torch.tensor([0, L])
    if B > 2:
        r[1] = torch.tensor([min(3, L - 1), min(3 + P + 2, L)])
        r[2] = torch.tensor([L - 1, L])
    if B > 3:
        r[3] = torch.tensor([L // 2, L // 2])
    return r.to(DEV, torch.int32)


def case(name, shape, mode):
    kw = {"residual_in_fp32": True} if mode == "bf16-res32" else {}
    dtype = F32 if mode == "f32" else BF16
    return pytest.param(name, kw, dtype, shape, id=f"{name}-B{shape[0]}-L{shape[1]}-{mode}")


MODES3 = ("bf16", "bf16-res32", "f32")
CASES = ([case(n, RAGGED, m) for n in ALL_PRESETS for m in MODES3]
         + [case("PlantCaduceus_l32", SNP, "bf16"), case("PlantCAD2-Large-l48-d1536", LONG, "bf16")])


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw,dtype,shape", CASES)
def test_engine_mean_equals_emulation(lib, switches, name, kw, dtype, shape):
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    cfg = two_layers(name, **kw)
    n = cfg.n_layer
    B, L = shape
    label = f"{name} B={B} L={L} {'f32' if dtype == F32 else ('bf16-res32' if kw else 'bf16')}"
    t0 = time.time()
    model = CaduceusForMaskedLM.from_pretrained(random_init_state_dict(cfg, seed=3), config=cfg, torch_dtype=TD[dtype]).to(DEV)
    ids = make_ids(B, L, seed=B * 7919 + L).to(DEV)
    ids_u8 = ids.to(torch.uint8)
    ws0 = model.workspace_bytes(B, L)
    entries = [h.float() for h in model.forward(ids, hidden_layers="all", compute_logits=False).hidden_states]
    ranges = engine_ranges(B, L, seed=L)
    layers = list(range(n + 1))
    for rng in (None, ranges):
        got = pooled_guarded(lib, model, ids_u8, rng, layers)
        for k in layers:
            want = mean_emulated(entries[k], rng)
            assert bits_equal(got[k], want), f"{label} entry {k} ranges={'full' if rng is None else 'mixed'}: {first_difference(got[k], want)}"
    del entries
    # one-position ranges equal pcad_hidden_at_layers, by value (converted to fp32)
    pos = ranges[:, :1].clamp(0, L - 1)
    one = torch.cat([pos, pos + 1], 1)
    at = model.hidden_at(ids_u8, pos, layers="all")[:, :, 0].float()
    assert torch.equal(model.hidden_mean(ids_u8, one, layers="all"), at), f"{label}: one-position means != hidden_at_layers"
    # a window alone equals the same window in the batch; a subset of entries equals the same entries of "all"
    full = model.hidden_mean(ids_u8, ranges, layers="all")
    for b in sorted({0, B // 2, B - 1}):
        alone = model.hidden_mean(ids_u8[b:b + 1], ranges[b:b + 1], layers="all")
        assert bits_equal(alone[:, 0], full[:, b]), f"{label}: window {b} alone != in the batch"
    sub = model.hidden_mean(ids_u8, ranges, layers=[n, 0])
    assert bits_equal(sub, full[[n, 0]]), f"{label}: [n, 0] != the same entries of 'all'"
    assert bits_equal(model.hidden_mean(ids_u8, ranges), full[n])
    assert bits_equal(model.hidden_mean(ids_u8, ranges, layers=[1]), full[[1]])
    # the forward stops after the deepest entry: a pooled call launches what pcad_hidden_at_layers launches, plus one
    # more kernel per entry (partials, then their sum, against one tap kernel)
    for want_layers in ([0], [1], [n], [0, n]):
        c0 = model.launch_count()
        model.hidden_at(ids_u8, pos, layers=want_layers)
        c1 = model.launch_count()
        model.hidden_mean(ids_u8, ranges, layers=want_layers)
        c2 = model.launch_count()
        assert c2 - c1 == (c1 - c0) + len(want_layers), (label, want_layers, c1 - c0, c2 - c1)
        if want_layers == [0]:
            stop0 = c2 - c1
    assert stop0 < c2 - c1, f"{label}: the pooled call for entry 0 did not stop early"
    assert model.workspace_bytes(B, L) == ws0
    model._release()
    print(f"[mean] engine {label:48s} all {n + 1} entries, full and mixed ranges, bit-identical to the order; "
          f"workspace {ws0 / 2 ** 20:.1f} MiB ({time.time() - t0:.1f} s)")


@pytest.mark.gpu
def test_mean_arguments_are_rejected(lib, switches):
    """A bad tap list and a null output return PCAD_ERR_INVALID, launch nothing and write nothing; Python rejects bad
    ranges before any launch."""
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    cfg = two_layers("PlantCaduceus_l20")
    model = CaduceusForMaskedLM.from_random(cfg, seed=1).to(DEV)
    B, L = 2, 64
    ids = make_ids(B, L, seed=2).to(DEV).to(torch.uint8)
    out = Guarded(3 * B, 2 * cfg.d_model, torch.float32)
    n0 = model.launch_count()
    for layers, null in (([], False), ([0, 1, 2, 2], False), ([0, 3], False), ([-1], False), ([1, 0], False), ([0], True)):
        k = max(len(layers), 1)
        idx = (C.c_int32 * k)(*layers)
        rc = lib.pcad_hidden_mean_at_layers(model._handle, C.c_void_p(ids.data_ptr()), None, B, L, len(layers), idx,
                                            None if null else out.ptr, _s())
        assert rc == PCAD_ERR_INVALID, (layers, null)
    for bad in ([[0, 1]], torch.zeros(B, 2), [[0, 1, 2]] * B):
        with pytest.raises(ValueError):
            model.hidden_mean(ids, bad)
    with pytest.raises(ValueError):
        model.hidden_mean(ids, layers=[3])
    torch.cuda.synchronize()
    assert model.launch_count() == n0
    assert_guards("rejected calls", out=out)
    model._release()


# ---- the semantics: the CPU oracle ------------------------------------------------------------------------------------------
def small_config(mixer):
    if mixer == "mamba1":
        return CaduceusConfig(d_model=256, n_layer=3)
    return CaduceusConfig(d_model=256, n_layer=3, ssm_cfg=dict(layer="Mamba2", d_state=64, d_conv=4, expand=2, headdim=64,
                                                              ngroups=1, conv_bias=True, bias=False))


@pytest.mark.gpu
@pytest.mark.parametrize("mixer", ["mamba1", "mamba2"])
def test_mean_matches_the_oracle(lib, switches, mixer):
    """fp32: every pooled entry within 1e-4 relative (to the entry's largest mean) of O.caduceus_forward's
    output_hidden_states averaged in float64, over whole windows and sub-ranges.  extract_embeddings(pooling="mean")
    returns the strand average of the same vectors."""
    from oracle import caduceus_oracle as O
    from plantcaduceus_b200.embeddings import average_strands, extract_embeddings
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    from plantcaduceus_b200.tokenizer import CharDNATokenizer
    cfg = small_config(mixer)
    B, L = 3, 200
    sd = random_init_state_dict(cfg, seed=5)
    tok = CharDNATokenizer()
    g = torch.Generator().manual_seed(7)
    seqs = ["".join("acgt"[int(t)] for t in torch.randint(0, 4, (L,), generator=g)) for _ in range(B)]
    ids = torch.from_numpy(tok.encode_bytes(tok.windows_to_ascii(seqs, L))).long()
    _, ref = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32, output_hidden_states=True)
    model = CaduceusForMaskedLM.from_pretrained(sd, config=cfg, torch_dtype=torch.float32).to(DEV)
    ranges = torch.tensor([[0, L], [17, 170], [100, 101]], dtype=torch.int32)
    errs = []
    for rng in (None, ranges):
        got = model.hidden_mean(ids.to(DEV, torch.uint8), rng, layers="all").cpu()
        for k, r in enumerate(ref):
            want = torch.stack([r[b, (0 if rng is None else int(rng[b, 0])):(L if rng is None else int(rng[b, 1]))].double().mean(0)
                                for b in range(B)])
            errs.append(float((got[k].double() - want).abs().max() / want.abs().max()))
    print(f"[mean] {mixer} fp32 pooled entries against the oracle, max|diff|/max|ref|: " + " ".join(f"{e:.2g}" for e in errs))
    assert max(errs) <= 1e-4, errs
    emb = extract_embeddings(model, tok, seqs, pooling="mean", ranges=ranges.numpy(), layer=[0, -1], batch_size=2)
    want = model.hidden_mean(ids.to(DEV, torch.uint8), ranges, layers=[0, -1]).cpu().numpy()
    assert emb.shape == (2, B, cfg.d_model) and (emb == average_strands(want)).all()
    one = extract_embeddings(model, tok, seqs, pooling="mean")
    assert (one == average_strands(model.hidden_mean(ids.to(DEV, torch.uint8)).cpu().numpy())).all()
    model._release()
