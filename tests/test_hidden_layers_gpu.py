"""Intermediate hidden states: the reference's full `hidden_states` tuple (n_layer + 1 entries) from pcad_forward_taps,
pcad_hidden_at_layers and the Python surface over them (`forward(hidden_layers=...)`, `hidden_at(layers=...)`,
`extract_embeddings(layer=...)`).

- The kernel: pcad_op_linear_residual_tap (out_proj's residual epilogue that also stores the pre-residual tile) at the
  out_proj shapes of the two largest presets and the benchmark's 262 144 rows: the tap equals pcad_op_linear, and the
  residual stream and its sums of squares equal pcad_op_linear_residual, bit for bit, inside guard-banded buffers.
- The engine: every entry equals the forward replay of tests/test_forward_replay_gpu.py bit for bit, with a recorder that
  taps each out_proj through pcad_op_linear; the logits and the last entry equal pcad_forward's (the taps perturb
  nothing); an entry requested alone (the forward stopping early) equals the same entry of a full-depth call;
  pcad_hidden_at_layers equals the matching slices; and every entry is exactly RC-equivariant.
- The semantics: every entry against the CPU oracle's output_hidden_states at a small shape of both mixers.
- Without a device: the Python index normalisation and rejection, the exports, and NULL-handle rejection."""
import ctypes as C
import time

import numpy as np
import pytest
import torch

from plantcaduceus_b200.configuration import CaduceusConfig, preset
from plantcaduceus_b200.modeling import hidden_layer_indices
from plantcaduceus_b200.weights import random_init_state_dict
from test_forward_replay_gpu import (RAGGED, SNP, Launcher, engine_weights, first_difference, forward_modes, hidden_tap,
                                     make_ids, replay, strand_ids, two_layers)
from test_forward_replay_gpu import budget, lib, switches  # noqa: F401  (fixtures)
from test_kernel_bounds_gpu import ALL_PRESETS, BF16, DEV, F32, LARGEST, T_PROD, TD, Guarded, assert_guards, gen, randn

PCAD_ERR_INVALID = -1
PAD = 16   # pad columns on the kernel test's pitched outputs


# ---- device-free ---------------------------------------------------------------------------------------------------------
def test_hidden_layer_indices():
    assert hidden_layer_indices("all", 32) == list(range(33))
    assert hidden_layer_indices([16, 0, -1], 32) == [16, 0, 32]
    assert hidden_layer_indices(range(3), 2) == [0, 1, 2]
    assert hidden_layer_indices((-33,), 32) == [0]
    assert hidden_layer_indices([3, np.int64(4)], 8) == [3, 4]
    assert hidden_layer_indices("all", 0) == [0]                 # n_layer = 0: the tuple has one entry, the final norm
    assert hidden_layer_indices([-1], 0) == [0]
    for bad in ([0, 0], [32, -1], [1, -32]):                      # duplicates, also after counting from the end
        with pytest.raises(ValueError, match="twice"):
            hidden_layer_indices(bad, 32)
    for bad, n_layer in (([33], 32), ([-34], 32), ([1], 0), ([-2], 0)):
        with pytest.raises(ValueError, match="out of range"):
            hidden_layer_indices(bad, n_layer)
    for bad in ("last", 3, None, [1.0], [True], ["1"], [[1]]):
        with pytest.raises(ValueError):
            hidden_layer_indices(bad, 32)
    with pytest.raises(ValueError, match="no hidden layer"):
        hidden_layer_indices([], 32)


def test_exports_and_null_handle():
    from plantcaduceus_b200 import _lib
    lib = _lib.load()
    for name in ("pcad_forward_taps", "pcad_hidden_at_layers", "pcad_op_linear_residual_tap"):
        assert name in _lib.EXPORTS and hasattr(lib, name)
    idx = (C.c_int32 * 1)(0)
    ptrs = (C.c_void_p * 1)(16)
    assert lib.pcad_forward_taps(None, C.c_void_p(16), 1, 1, None, 1, idx, ptrs, None) == PCAD_ERR_INVALID
    assert lib.pcad_hidden_at_layers(None, C.c_void_p(16), C.c_void_p(16), 1, 1, 1, 1, idx, C.c_void_p(16), None) == PCAD_ERR_INVALID
    # the tap epilogue is bf16 only, and needs its tap buffer: rejected before any device work
    p = C.c_void_p(16)
    assert lib.pcad_op_linear_residual_tap(p, p, p, p, p, p, 128, 128, 128, 128, 128, 128, 128, F32, None) == PCAD_ERR_INVALID
    assert lib.pcad_op_linear_residual_tap(p, p, p, p, p, None, 128, 128, 128, 128, 128, 128, 128, BF16, None) == PCAD_ERR_INVALID


# ---- the kernel ----------------------------------------------------------------------------------------------------------
def _s():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.gpu
@pytest.mark.parametrize("name", LARGEST)
def test_linear_residual_tap_kernel(lib, switches, name):
    """out_proj at T_PROD rows, in place as the forward runs it: tap == pcad_op_linear, resid_out and sumsq_out ==
    pcad_op_linear_residual, bit for bit; no byte outside any output changes."""
    cfg = preset(name)
    M, N, K = T_PROD, cfg.d_model, cfg.d_inner
    g = gen(31)
    A = randn(g, M, K, dtype=torch.bfloat16)
    A.mul_(torch.exp(randn(g, M, 1)).to(torch.bfloat16))
    W = randn(g, N, K, dtype=torch.bfloat16, scale=K ** -0.5)
    r0 = randn(g, M, N, dtype=torch.bfloat16, scale=2.0)
    parts = lib.pcad_op_sumsq_parts(N)
    a, w = C.c_void_p(A.data_ptr()), C.c_void_p(W.data_ptr())

    def ok(rc):
        assert rc == 0, lib.pcad_last_error(None)
    plain = Guarded(M, N, torch.bfloat16, ld=N + PAD)
    ok(lib.pcad_op_linear(a, w, plain.ptr, M, N, K, K, K, plain.ld, BF16, _s()))
    res_ref, ss_ref = Guarded(M, N, torch.bfloat16, ld=N + PAD), Guarded(M, parts, torch.float32)
    res_ref.t.copy_(r0)
    ok(lib.pcad_op_linear_residual(a, w, res_ref.ptr, res_ref.ptr, ss_ref.ptr, M, N, K, K, K, res_ref.ld, BF16, _s()))
    res, ss, tap = Guarded(M, N, torch.bfloat16, ld=N + PAD), Guarded(M, parts, torch.float32), Guarded(M, N, torch.bfloat16, ld=N + 2 * PAD)
    res.t.copy_(r0)
    ok(lib.pcad_op_linear_residual_tap(a, w, res.ptr, res.ptr, ss.ptr, tap.ptr, M, N, K, K, K, res.ld, tap.ld, BF16, _s()))
    # malformed tap arguments are rejected and write nothing
    for ld_tap, ptr in ((N + 4, tap.ptr), (N - 8, tap.ptr), (tap.ld, C.c_void_p(tap.mat.data_ptr() + 8))):
        assert lib.pcad_op_linear_residual_tap(a, w, res.ptr, res.ptr, ss.ptr, ptr, M, N, K, K, K, res.ld, ld_tap, BF16, _s()) == PCAD_ERR_INVALID
    torch.cuda.synchronize()
    assert_guards(f"{name} linear_residual_tap", resid=res, sumsq=ss, tap=tap)
    assert_guards(f"{name} references", C=plain, resid=res_ref, sumsq=ss_ref)
    assert torch.equal(tap.t, plain.t), f"tap != pcad_op_linear: {first_difference(tap.t.float(), plain.t.float())}"
    assert torch.equal(res.t, res_ref.t), f"resid_out != pcad_op_linear_residual: {first_difference(res.t.float(), res_ref.t.float())}"
    assert torch.equal(ss.t, ss_ref.t), f"sumsq_out != pcad_op_linear_residual: {first_difference(ss.t, ss_ref.t)}"
    print(f"[taps] {name} out_proj M={M} N={N} K={K}: tap, resid_out and sumsq_out bit-identical; guards intact")


# ---- the engine ----------------------------------------------------------------------------------------------------------
class TapRecorder(Launcher):
    """The replay's executor that also records hidden_states[li + 1] at every out_proj: pcad_op_linear(y, W_out), the mixer
    output before the residual add, through hidden_tap.  (The last layer's entry is recorded too; it is not a hidden state:
    the tuple's last entry is the final norm.)"""

    def __init__(self, lib, B, L, d):
        super().__init__(lib)
        self.B, self.L, self.d, self.taps = B, L, d, []

    def linear(self, name, A, W, Cm, M, N, K, lda, ldw, ldc, dtype, A_off=0):
        super().linear(name, A, W, Cm, M, N, K, lda, ldw, ldc, dtype, A_off)
        if name == "out_proj":       # non-fused: out_proj writes the mixer output itself
            self.taps.append(hidden_tap(Cm, self.B, self.L, self.d))

    def linear_residual(self, name, A, W, res_in, res_out, ss_out, M, N, K, lda, ldw, ld_res):
        y = torch.empty(M, N, dtype=torch.bfloat16, device=A.device)
        self._ok(self.lib.pcad_op_linear(self._p(A), self._p(W), self._p(y), M, N, K, lda, ldw, N, BF16, self._s()))
        self.taps.append(hidden_tap(y, self.B, self.L, self.d))
        super().linear_residual(name, A, W, res_in, res_out, ss_out, M, N, K, lda, ldw, ld_res)


def replay_taps(lib, cfg, sd, dtype, ids, modes):
    """Every hidden_states entry by the replay: [n_layer + 1] tensors [B, L, 2d]."""
    B, L = ids.shape
    d = cfg.d_model
    w = engine_weights(cfg, sd, dtype, DEV)
    ex = TapRecorder(lib, B, L, d)
    ids_dev = ids.to(DEV)
    comp = torch.tensor([cfg.complement_map[i] for i in range(cfg.vocab_size)], device=DEV)
    emb = hidden_tap(w["emb"][strand_ids(ids_dev, comp)], B, L, d)
    final = hidden_tap(replay(ex, cfg, w, dtype, ids_dev, modes), B, L, d)
    assert len(ex.taps) == cfg.n_layer
    return [emb] + ex.taps[:cfg.n_layer - 1] + [final]


def forward_taps_guarded(lib, model, ids_dev, layers, logits=True):
    """pcad_forward_taps through the C ABI into Guarded buffers; checks the guards.  Returns (taps, logits or None)."""
    B, L = ids_dev.shape
    d, V = model.config.d_model, model.config.vocab_size
    bufs = [Guarded(B * L, 2 * d, model.dtype) for _ in layers]
    lg = Guarded(B * L, V, torch.float32) if logits else None
    idx = (C.c_int32 * len(layers))(*layers)
    ptrs = (C.c_void_p * len(layers))(*[b.mat.data_ptr() for b in bufs])
    rc = lib.pcad_forward_taps(model._handle, C.c_void_p(ids_dev.data_ptr()), B, L, lg.ptr if lg else None, len(layers), idx,
                               ptrs, _s())
    assert rc == 0, lib.pcad_last_error(model._handle)
    torch.cuda.synchronize()
    assert_guards("pcad_forward_taps", **{f"tap{k}": b for k, b in zip(layers, bufs)}, **({"logits": lg} if lg else {}))
    return [b.t.view(B, L, 2 * d).clone() for b in bufs], (lg.t.view(B, L, V).clone() if lg else None)


def engine_taps(lib, cfg, sd, dtype, ids, label):
    """Runs the engine checks that need no replay and returns its full-depth taps."""
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    B, L = ids.shape
    n = cfg.n_layer
    model = CaduceusForMaskedLM.from_pretrained(sd, config=cfg, torch_dtype=TD[dtype]).to(DEV)
    ids_dev = ids.to(DEV)
    base = model(input_ids=ids_dev, output_hidden_states=True)
    taps, logits = forward_taps_guarded(lib, model, ids_dev, list(range(n + 1)))
    assert torch.equal(taps[n], base.hidden_states[-1]), f"{label}: hidden_states[n_layer] != pcad_forward's hidden output"
    assert torch.equal(logits, base.logits), f"{label}: logits with every tap != pcad_forward's"
    del base, logits
    # the forward stopped at the one requested entry (Python surface), against the full-depth call
    for k in range(n + 1):
        out = model.forward(ids_dev, hidden_layers=[k], compute_logits=False)
        assert out.logits is None and len(out.hidden_states) == n + 1
        assert all(h is None for i, h in enumerate(out.hidden_states) if i != k)
        assert torch.equal(out.hidden_states[k], taps[k]), f"{label}: entry {k} alone: {first_difference(out.hidden_states[k], taps[k])}"
    # pcad_hidden_at_layers: the matching slices, in the caller's order
    ids_u8 = ids_dev.to(torch.uint8)
    g = torch.Generator().manual_seed(L)
    pos = torch.stack([torch.randperm(L, generator=g)[:3] for _ in range(B)]).to(DEV, torch.int32)
    b_idx = torch.arange(B, device=DEV)[:, None]
    order = list(range(n, -1, -1))
    at = model.hidden_at(ids_u8, pos, layers=order)
    want = torch.stack([taps[k][b_idx, pos.long()] for k in order])
    assert torch.equal(at, want), f"{label}: hidden_at_layers != slices of pcad_forward_taps: {first_difference(at, want)}"
    assert torch.equal(model.hidden_at(ids_u8, pos, layers=[-1])[0], model.hidden_at(ids_u8, pos))
    # RC equivariance, exact: the RC strand of RC(ids) is ids itself
    comp = torch.tensor([cfg.complement_map[i] for i in range(cfg.vocab_size)], device=DEV)
    rc = model.forward(comp[ids_dev.flip(1)], hidden_layers="all", compute_logits=False).hidden_states
    for k in range(n + 1):
        assert torch.equal(rc[k], taps[k].flip(1, 2)), f"{label}: entry {k} is not RC-equivariant: {first_difference(rc[k], taps[k].flip(1, 2))}"
    del rc
    model._release()
    return taps


def case(name, shape, mode, ssd_seq=False):
    kw = {"residual_in_fp32": True} if mode == "bf16-res32" else {}
    dtype = F32 if mode == "f32" else BF16
    tag = f"{name}-B{shape[0]}-L{shape[1]}-{mode}" + ("-ssdseq" if ssd_seq else "")
    return pytest.param(name, kw, dtype, shape, ssd_seq, id=tag)


MODES3 = ("bf16", "bf16-res32", "f32")
CASES = ([case(n, RAGGED, m) for n in ALL_PRESETS for m in MODES3]
         + [case(n, SNP, m) for n in LARGEST for m in MODES3]
         + [case("PlantCaduceus_l20", (1, 8192), "bf16"), case("PlantCAD2-Small-l24-d0768", RAGGED, "bf16", ssd_seq=True)])


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw,dtype,shape,ssd_seq", CASES)
def test_taps_equal_replay(lib, switches, name, kw, dtype, shape, ssd_seq):
    """Every hidden_states entry of pcad_forward_taps equals the replay's bit for bit; the logits and the last entry equal
    pcad_forward's; each entry alone (early exit) and pcad_hidden_at_layers equal the full-depth call; RC-equivariant."""
    if ssd_seq:
        switches.setenv("PCAD_SSD_SEQ", "1")
    cfg = two_layers(name, **kw)
    B, L = shape
    mode = "f32" if dtype == F32 else ("bf16-res32" if kw else "bf16")
    label = f"{name} B={B} L={L} {mode}"
    sd = random_init_state_dict(cfg, seed=3)
    ids = make_ids(B, L, seed=B * 7919 + L)
    modes = forward_modes(cfg, B, L, dtype, torch.cuda.get_device_properties(0).multi_processor_count, ssd_seq)
    t0 = time.time()
    got = engine_taps(lib, cfg, sd, dtype, ids, label)
    want = replay_taps(lib, cfg, sd, dtype, ids, modes)
    torch.cuda.synchronize()
    for k in range(cfg.n_layer + 1):
        assert torch.equal(got[k], want[k]), f"{label}: hidden_states[{k}] != replay: {first_difference(got[k], want[k])}"
    print(f"[taps] {label:52s} {modes.flags()} all {cfg.n_layer + 1} entries bit-identical to the replay ({time.time() - t0:.1f} s)")


@pytest.mark.gpu
def test_tap_arguments_are_rejected(lib, switches):
    """n_taps outside [1, n_layer + 1], an index outside [0, n_layer], indices not strictly increasing and a null tap
    pointer return PCAD_ERR_INVALID, launch nothing and write nothing."""
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    cfg = two_layers("PlantCaduceus_l20")
    model = CaduceusForMaskedLM.from_random(cfg, seed=1).to(DEV)
    B, L = 2, 64
    ids = make_ids(B, L, seed=2).to(DEV)
    pos = torch.zeros(B, 1, dtype=torch.int32, device=DEV)
    bufs = [Guarded(B * L, 2 * cfg.d_model, torch.bfloat16) for _ in range(4)]
    n0 = model.launch_count()
    for layers, null in (([], False), ([0, 1, 2, 2], False), ([0, 3], False), ([-1], False), ([1, 0], False), ([0, 0], False),
                         ([0, 1], True)):
        k = max(len(layers), 1)
        idx = (C.c_int32 * k)(*layers)
        ptrs = (C.c_void_p * k)(*[None if null and i == 1 else bufs[i].mat.data_ptr() for i in range(k)])
        rc = lib.pcad_forward_taps(model._handle, C.c_void_p(ids.data_ptr()), B, L, None, len(layers), idx, ptrs, _s())
        assert rc == PCAD_ERR_INVALID, (layers, null)
        rc = lib.pcad_hidden_at_layers(model._handle, C.c_void_p(ids.to(torch.uint8).data_ptr()), C.c_void_p(pos.data_ptr()), B, L,
                                       1, len(layers), idx, None if null else bufs[0].ptr, _s())
        assert rc == PCAD_ERR_INVALID, (layers, null)
    torch.cuda.synchronize()
    assert model.launch_count() == n0
    assert_guards("rejected calls", **{f"b{i}": b for i, b in enumerate(bufs)})
    with pytest.raises(ValueError):
        model.forward(ids, hidden_layers=[3])
    with pytest.raises(ValueError):
        model.hidden_at(ids.to(torch.uint8), pos, layers=[0, -3])


# ---- the semantics: the CPU oracle ------------------------------------------------------------------------------------------
def small_config(mixer):
    if mixer == "mamba1":
        return CaduceusConfig(d_model=256, n_layer=3)
    return CaduceusConfig(d_model=256, n_layer=3, ssm_cfg=dict(layer="Mamba2", d_state=64, d_conv=4, expand=2, headdim=64,
                                                              ngroups=1, conv_bias=True, bias=False))


BF16_FLOOR = 2e-2   # bf16 entries: max |diff| / max |ref| against the fp32 oracle, or 1.5 x the bf16 oracle's own, if larger


@pytest.mark.gpu
@pytest.mark.parametrize("mixer", ["mamba1", "mamba2"])
def test_taps_match_the_oracle(lib, switches, mixer):
    """Every entry against O.caduceus_forward(output_hidden_states=True): fp32 within 1e-4 relative (to the entry's largest
    value); bf16 within max(BF16_FLOOR, 1.5 x the bf16 oracle's own distance from the fp32 oracle) -- the reference algorithm
    run in bf16 rounds each direction's out_proj before adding them, the engine rounds once after one out_proj on the
    summed y (INTEGRATION.md section 5), so neither is closer to fp32 by construction.  extract_embeddings(layer=...) returns
    the same entries at tokenIdx."""
    from oracle import caduceus_oracle as O
    from plantcaduceus_b200.embeddings import average_strands, extract_embeddings
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    from plantcaduceus_b200.tokenizer import CharDNATokenizer
    cfg = small_config(mixer)
    B, L = 3, 200
    sd = random_init_state_dict(cfg, seed=5)
    ids = make_ids(B, L, seed=7)
    _, ref = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32, output_hidden_states=True)
    _, ref16 = O.caduceus_forward(sd, cfg, ids, dtype=torch.bfloat16, output_hidden_states=True)
    assert len(ref) == cfg.n_layer + 1

    def rel(a, b):
        return float((a.float() - b.float()).abs().max() / b.float().abs().max())
    for torch_dtype in (torch.float32, torch.bfloat16):
        model = CaduceusForMaskedLM.from_pretrained(sd, config=cfg, torch_dtype=torch_dtype).to(DEV)
        out = model(input_ids=ids.to(DEV), hidden_layers="all")
        assert len(out.hidden_states) == cfg.n_layer + 1
        errs = [rel(h.cpu(), r) for h, r in zip(out.hidden_states, ref)]
        if torch_dtype == torch.float32:
            print(f"[taps] {mixer} fp32 max|diff|/max|ref| per entry: " + " ".join(f"{e:.2g}" for e in errs))
            assert max(errs) <= 1e-4, errs
        else:
            own = [rel(r16, r) for r16, r in zip(ref16, ref)]
            print(f"[taps] {mixer} bf16 engine per entry: " + " ".join(f"{e:.2g}" for e in errs)
                  + " | bf16 oracle: " + " ".join(f"{e:.2g}" for e in own))
            for k, (e, o) in enumerate(zip(errs, own)):
                assert e <= max(BF16_FLOOR, 1.5 * o), f"entry {k}: {e:.3g} (bf16 oracle {o:.3g})"
        # extract_embeddings(layer=...) reads the same entries at tokenIdx
        tok = CharDNATokenizer()
        seqs = ["".join("acgt"[int(t) % 4] for t in row) for row in ids]
        ids_tok = torch.from_numpy(tok.encode_bytes(tok.windows_to_ascii(seqs, L))).long()
        want = model(input_ids=ids_tok.to(DEV), hidden_layers="all").hidden_states
        emb = extract_embeddings(model, tok, seqs, tokenIdx=100, layer=[1, 0, -1], average=False)
        assert emb.shape == (3, B, 2 * cfg.d_model)
        for i, k in enumerate([1, 0, cfg.n_layer]):
            assert torch.equal(torch.from_numpy(emb[i]), want[k][:, 100].float().cpu()), (mixer, torch_dtype, k)
        one = extract_embeddings(model, tok, seqs, tokenIdx=100, layer=2)
        assert one.shape == (B, cfg.d_model) and (one == average_strands(want[2][:, 100].float().cpu().numpy())).all()
        model._release()
