"""The hidden-state entry points as one path: pcad_forward's hidden output and pcad_hidden_at are the tap entry points
pcad_forward_taps / pcad_hidden_at_layers with tap_idx = {n_layer}, so they must launch the same kernels.  Their outputs
are compared bit for bit in test_hidden_layers_gpu.py, test_forward_replay_gpu.py and test_kernel_bounds_gpu.py; this file
checks what those do not:

- Launch counts at every preset with one and two layers, in bf16, bf16 residual_in_fp32 and fp32: each old entry point
  launches what its tap counterpart launches, and the hidden output of pcad_forward costs exactly one kernel.
- n_layer = 0, where hidden_states has one entry, the final norm: every tap entry point emits it once, so it launches what
  pcad_forward(NULL, hidden) launches (the pooled call one more: partials, then their sum), and writes pcad_forward's
  hidden output bit for bit, inside guard-banded buffers.
- The return codes of degenerate calls to all five entry points (B = 0, L = 0, n_pos = 0, null outputs and ids, an
  unfinalised or null handle): none launches a kernel or writes a byte."""
import ctypes as C
import dataclasses

import pytest
import torch

from plantcaduceus_b200.configuration import preset
from test_forward_replay_gpu import RAGGED, make_ids
from test_forward_replay_gpu import budget, lib, switches  # noqa: F401  (fixtures)
from test_kernel_bounds_gpu import ALL_PRESETS, BF16, DEV, F32, SENTINEL, TD, Guarded, assert_guards

PCAD_OK, PCAD_ERR_INVALID, PCAD_ERR_STATE = 0, -1, -3
MODES3 = ("bf16", "bf16-res32", "f32")
N_POS = 3


def make_model(name, mode, n_layer):
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    kw = {"residual_in_fp32": True} if mode == "bf16-res32" else {}
    cfg = dataclasses.replace(preset(name, **kw), n_layer=n_layer)
    return CaduceusForMaskedLM.from_random(cfg, seed=1, torch_dtype=TD[F32 if mode == "f32" else BF16]).to(DEV)


def inputs(B, L, seed):
    """int64 and uint8 ids [B, L] and int32 positions [B, N_POS] (both edges among them) on the device."""
    ids = make_ids(B, L, seed=seed).to(DEV)
    g = torch.Generator().manual_seed(seed)
    pos = torch.stack([torch.randperm(L, generator=g)[:N_POS] for _ in range(B)])
    pos[0, :2] = torch.tensor([0, L - 1])
    return ids, ids.to(torch.uint8), pos.to(DEV, torch.int32)


def _p(t):
    return C.c_void_p(t.data_ptr())


def _s():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def launches(lib, model, call):
    """Kernels launched by call(), which must succeed."""
    n0 = model.launch_count()
    rc = call()
    assert rc == PCAD_OK, lib.pcad_last_error(model._handle)
    return model.launch_count() - n0


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES3)
@pytest.mark.parametrize("n_layer", [1, 2])
@pytest.mark.parametrize("name", ALL_PRESETS)
def test_final_state_entries_launch_as_their_taps(lib, switches, name, n_layer, mode):
    """pcad_forward(logits, hidden) == pcad_forward_taps([n_layer], logits) and pcad_hidden_at ==
    pcad_hidden_at_layers([n_layer]) in launches; the hidden output adds one launch to pcad_forward(logits, NULL)."""
    model = make_model(name, mode, n_layer)
    h, cfg = model._handle, model.config
    B, L = RAGGED
    ids, ids8, pos = inputs(B, L, seed=B * 7919 + L)
    logits = torch.empty(B, L, cfg.vocab_size, dtype=torch.float32, device=DEV)
    hidden = torch.empty(B, L, 2 * cfg.d_model, dtype=model.dtype, device=DEV)
    at = torch.empty(B, N_POS, 2 * cfg.d_model, dtype=model.dtype, device=DEV)
    top = (C.c_int32 * 1)(n_layer)
    n = {
        "forward": launches(lib, model, lambda: lib.pcad_forward(h, _p(ids), B, L, _p(logits), _p(hidden), _s())),
        "forward_taps": launches(lib, model, lambda: lib.pcad_forward_taps(h, _p(ids), B, L, _p(logits), 1, top,
                                                                           (C.c_void_p * 1)(hidden.data_ptr()), _s())),
        "forward_no_hidden": launches(lib, model, lambda: lib.pcad_forward(h, _p(ids), B, L, _p(logits), None, _s())),
        "hidden_at": launches(lib, model, lambda: lib.pcad_hidden_at(h, _p(ids8), _p(pos), B, L, N_POS, _p(at), _s())),
        "hidden_at_layers": launches(lib, model, lambda: lib.pcad_hidden_at_layers(h, _p(ids8), _p(pos), B, L, N_POS, 1, top,
                                                                                   _p(at), _s())),
    }
    torch.cuda.synchronize()
    model._release()
    label = f"{name} n_layer={n_layer} {mode}: {n}"
    assert n["forward"] == n["forward_taps"], label
    assert n["forward"] == n["forward_no_hidden"] + 1, label
    assert n["hidden_at"] == n["hidden_at_layers"], label
    print(f"[entry] {label}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES3)
@pytest.mark.parametrize("name", ALL_PRESETS)
def test_no_layer_entry_is_emitted_once(lib, switches, name, mode):
    """n_layer = 0: hidden_states[0] is the final norm.  Each tap entry point asked for [0] writes pcad_forward's hidden
    output (the positions' slices; a one-position mean is the entry itself in fp32) and launches what pcad_forward(NULL,
    hidden) launches, the pooled call one kernel more."""
    model = make_model(name, mode, 0)
    h, d = model._handle, model.config.d_model
    B, L = RAGGED
    ids, ids8, pos = inputs(B, L, seed=B + L)
    zero = (C.c_int32 * 1)(0)
    one_pos = torch.cat([pos[:, :1], pos[:, :1] + 1], 1)
    ref = Guarded(B * L, 2 * d, model.dtype)
    tap, at, at_old = Guarded(B * L, 2 * d, model.dtype), Guarded(B * N_POS, 2 * d, model.dtype), Guarded(B * N_POS, 2 * d, model.dtype)
    mean = Guarded(B, 2 * d, torch.float32)
    n = {
        "forward(NULL, hidden)": launches(lib, model, lambda: lib.pcad_forward(h, _p(ids), B, L, None, ref.ptr, _s())),
        "forward_taps": launches(lib, model, lambda: lib.pcad_forward_taps(h, _p(ids), B, L, None, 1, zero,
                                                                           (C.c_void_p * 1)(tap.mat.data_ptr()), _s())),
        "hidden_at_layers": launches(lib, model, lambda: lib.pcad_hidden_at_layers(h, _p(ids8), _p(pos), B, L, N_POS, 1, zero,
                                                                                   at.ptr, _s())),
        "hidden_at": launches(lib, model, lambda: lib.pcad_hidden_at(h, _p(ids8), _p(pos), B, L, N_POS, at_old.ptr, _s())),
        "hidden_mean_at_layers": launches(lib, model, lambda: lib.pcad_hidden_mean_at_layers(h, _p(ids8), _p(one_pos), B, L, 1,
                                                                                             zero, mean.ptr, _s())),
    }
    torch.cuda.synchronize()
    assert_guards(f"{name} n_layer=0 {mode}", ref=ref, tap=tap, at=at, at_old=at_old, mean=mean)
    hid = ref.t.view(B, L, 2 * d)
    want_at = hid[torch.arange(B, device=DEV)[:, None], pos.long()].reshape(B * N_POS, 2 * d)
    assert torch.equal(tap.t, ref.t), f"{name} {mode}: pcad_forward_taps([0]) != pcad_forward's hidden output"
    assert torch.equal(at.t, want_at), f"{name} {mode}: pcad_hidden_at_layers([0]) != slices of pcad_forward's hidden output"
    assert torch.equal(at_old.t, want_at), f"{name} {mode}: pcad_hidden_at != slices of pcad_forward's hidden output"
    assert torch.equal(mean.t, hid[torch.arange(B, device=DEV), pos[:, 0].long()].float()), \
        f"{name} {mode}: one-position means != pcad_forward's hidden output"
    model._release()
    base = n["forward(NULL, hidden)"]
    extra = {k: v - base for k, v in n.items()}
    assert extra == {"forward(NULL, hidden)": 0, "forward_taps": 0, "hidden_at_layers": 0, "hidden_at": 0,
                     "hidden_mean_at_layers": 1}, f"{name} n_layer=0 {mode}: launches beyond pcad_forward(NULL, hidden) = {base}: {extra}"
    print(f"[entry] {name} n_layer=0 {mode}: {n}")


def unfinalised_handle(lib, n_layer):
    from plantcaduceus_b200 import _lib
    cfg = _lib.PcadConfig(128, n_layer, 8, 16, 4, 2, 8, 1e-5, 0, BF16)
    for i in range(16):
        cfg.complement_map[i] = i
    h = C.c_void_p()
    assert lib.pcad_create(C.byref(cfg), 0, C.byref(h)) == PCAD_OK, lib.pcad_last_error(None)
    return h


@pytest.mark.gpu
def test_degenerate_calls_return_codes(lib, switches):
    """One table of return codes.  An empty call (B, L or n_pos 0) returns PCAD_OK once the handle is finalised, whatever
    its pointers -- except for the outputs the tap entry points check first: pcad_hidden_at_layers' hidden_dev,
    pcad_forward_taps' tap pointers and pcad_hidden_mean_at_layers' out_dev.  No call launches or writes anything."""
    model = make_model("PlantCaduceus_l20", "bf16", 2)
    h, u, cfg = model._handle, unfinalised_handle(lib, 2), model.config
    B, L = 2, 64
    ids, ids8, pos = inputs(B, L, seed=5)
    ranges = torch.tensor([[0, L]] * B, dtype=torch.int32, device=DEV)
    w = 2 * cfg.d_model
    lg, hid = Guarded(B * L, cfg.vocab_size, torch.float32), Guarded(B * L, w, model.dtype)
    at, mean = Guarded(B * N_POS, w, model.dtype), Guarded(B, w, torch.float32)
    top, bad = (C.c_int32 * 1)(2), (C.c_int32 * 1)(3)
    taps, null_tap = (C.c_void_p * 1)(hid.mat.data_ptr()), (C.c_void_p * 1)(None)
    i64, i8, ps, rg, s = _p(ids), _p(ids8), _p(pos), _p(ranges), _s()
    OK, INV, STATE = PCAD_OK, PCAD_ERR_INVALID, PCAD_ERR_STATE

    def fwd(hh, b, l, ids_=i64, logits=lg.ptr, hidden=hid.ptr):
        return lib.pcad_forward(hh, ids_, b, l, logits, hidden, s)

    def hat(hh, b, l, n_pos, ids_=i8, pos_=ps, hidden=at.ptr):
        return lib.pcad_hidden_at(hh, ids_, pos_, b, l, n_pos, hidden, s)

    def ftaps(hh, b, l, ids_=i64, idx=top, tap_dev=taps):
        return lib.pcad_forward_taps(hh, ids_, b, l, lg.ptr, 1, idx, tap_dev, s)

    def hlayers(hh, b, l, n_pos, ids_=i8, pos_=ps, hidden=at.ptr, idx=top):
        return lib.pcad_hidden_at_layers(hh, ids_, pos_, b, l, n_pos, 1, idx, hidden, s)

    def hmean(hh, b, l, ids_=i8, out=mean.ptr, idx=top):
        return lib.pcad_hidden_mean_at_layers(hh, ids_, rg, b, l, 1, idx, out, s)

    table = [
        ("forward B=0", OK, lambda: fwd(h, 0, L)),
        ("forward L=0", OK, lambda: fwd(h, B, 0)),
        ("forward B=0, null ids and outputs", OK, lambda: fwd(h, 0, L, None, None, None)),
        ("forward null ids", INV, lambda: fwd(h, B, L, None)),
        ("forward B<0", INV, lambda: fwd(h, -1, L)),
        ("forward unfinalised", STATE, lambda: fwd(u, B, L)),
        ("forward unfinalised, B=0", STATE, lambda: fwd(u, 0, L)),
        ("forward null handle", INV, lambda: fwd(None, B, L)),
        ("hidden_at B=0, null hidden", OK, lambda: hat(h, 0, L, N_POS, hidden=None)),
        ("hidden_at L=0", OK, lambda: hat(h, B, 0, N_POS)),
        ("hidden_at n_pos=0, null pos and hidden", OK, lambda: hat(h, B, L, 0, pos_=None, hidden=None)),
        ("hidden_at null hidden", INV, lambda: hat(h, B, L, N_POS, hidden=None)),
        ("hidden_at null pos", INV, lambda: hat(h, B, L, N_POS, pos_=None)),
        ("hidden_at null ids", INV, lambda: hat(h, B, L, N_POS, ids_=None)),
        ("hidden_at n_pos<0", INV, lambda: hat(h, B, L, -1)),
        ("hidden_at unfinalised", STATE, lambda: hat(u, B, L, N_POS)),
        ("hidden_at null handle", INV, lambda: hat(None, B, L, N_POS)),
        ("forward_taps B=0", OK, lambda: ftaps(h, 0, L)),
        ("forward_taps L=0", OK, lambda: ftaps(h, B, 0)),
        ("forward_taps B=0, null ids", OK, lambda: ftaps(h, 0, L, ids_=None)),
        ("forward_taps B=0, null tap_dev", INV, lambda: ftaps(h, 0, L, tap_dev=None)),
        ("forward_taps B=0, null tap pointer", INV, lambda: ftaps(h, 0, L, tap_dev=null_tap)),
        ("forward_taps null ids", INV, lambda: ftaps(h, B, L, ids_=None)),
        ("forward_taps unfinalised", STATE, lambda: ftaps(u, B, L)),
        ("forward_taps unfinalised, index out of range", INV, lambda: ftaps(u, B, L, idx=bad)),
        ("forward_taps null handle", INV, lambda: ftaps(None, B, L)),
        ("hidden_at_layers B=0", OK, lambda: hlayers(h, 0, L, N_POS)),
        ("hidden_at_layers B=0, null hidden", INV, lambda: hlayers(h, 0, L, N_POS, hidden=None)),
        ("hidden_at_layers L=0", OK, lambda: hlayers(h, B, 0, N_POS)),
        ("hidden_at_layers n_pos=0, null pos", OK, lambda: hlayers(h, B, L, 0, pos_=None)),
        ("hidden_at_layers null pos", INV, lambda: hlayers(h, B, L, N_POS, pos_=None)),
        ("hidden_at_layers null ids", INV, lambda: hlayers(h, B, L, N_POS, ids_=None)),
        ("hidden_at_layers n_pos<0", INV, lambda: hlayers(h, B, L, -1)),
        ("hidden_at_layers unfinalised", STATE, lambda: hlayers(u, B, L, N_POS)),
        ("hidden_at_layers unfinalised, index out of range", INV, lambda: hlayers(u, B, L, N_POS, idx=bad)),
        ("hidden_at_layers null handle", INV, lambda: hlayers(None, B, L, N_POS)),
        ("hidden_mean B=0", OK, lambda: hmean(h, 0, L)),
        ("hidden_mean L=0", OK, lambda: hmean(h, B, 0)),
        ("hidden_mean B=0, null ids", OK, lambda: hmean(h, 0, L, ids_=None)),
        ("hidden_mean B=0, null out", INV, lambda: hmean(h, 0, L, out=None)),
        ("hidden_mean null ids", INV, lambda: hmean(h, B, L, ids_=None)),
        ("hidden_mean unfinalised", STATE, lambda: hmean(u, B, L)),
        ("hidden_mean unfinalised, index out of range", INV, lambda: hmean(u, B, L, idx=bad)),
        ("hidden_mean null handle", INV, lambda: hmean(None, B, L)),
    ]
    n0 = model.launch_count()
    got = {label: call() for label, _, call in table}
    torch.cuda.synchronize()
    launched = model.launch_count() - n0, lib.pcad_launch_count(u)
    lib.pcad_destroy(u)
    wrong = {label: (got[label], want) for label, want, _ in table if got[label] != want}
    assert not wrong, f"return codes (got, want): {wrong}"
    assert launched == (0, 0), f"degenerate calls launched kernels: {launched}"
    for name, g in (("logits", lg), ("hidden", hid), ("at", at), ("mean", mean)):
        assert bool((g.raw.view(torch.int16) == SENTINEL).all()), f"a degenerate call wrote into {name}"
    model._release()
