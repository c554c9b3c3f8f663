"""End-to-end parity of the B200 engine (through the drop-in HF-style object -> C ABI) against the CPU oracle.

Tolerances are BASELINE.json's: fp32 logits within 1e-4 relative; bf16 logits within 2e-2 absolute;
ref/alt LLR Spearman >= 0.999; tokenisation / RC indexing bit-exact.

bf16 bar, as tested (`assert_bf16_parity`): the engine's bf16 logits are compared with the fp32 oracle.
  * at the scored positions (the masked index, a/c/g/t columns -- the only values the reference's
    scorer reads, zero_shot_score.py:117-118) max |err| <= 2e-2;
  * over ALL positions, max |err| <= max(2e-2, the bf16 ORACLE's own max |err| against the fp32 oracle):
    at 20+ layers a pure-bf16 run of the reference algorithm is itself 3-5e-2 away from fp32 on logits
    of magnitude ~8 (measured: l20, 0.043), so 2e-2 over every position is not a bar the reference meets;
    the engine must be at least as close to fp32 as the reference's bf16 arithmetic is;
  * mean |err| <= 1e-2."""
import numpy as np
import pytest
import torch

from oracle import caduceus_oracle as O
from plantcaduceus_b200 import CaduceusConfig, CharDNATokenizer, preset, random_init_state_dict

pytestmark = pytest.mark.gpu


def make_ids(B, L, seed, mask_at=None):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(3, 7, (B, L), generator=g)
    if mask_at is not None:
        ids[:, mask_at] = 1
    if L > 3:
        ids[0, 1] = 2   # an N
    return ids


def rel_err(got, want):
    return ((got - want).abs().max() / want.abs().max()).item()


def assert_bf16_parity(got, want_fp32, want_bf16, scored=None):
    err = (got - want_fp32).abs()
    ref_self = (want_bf16 - want_fp32).abs().max().item()
    print(f"bf16 engine vs fp32 oracle: max {err.max().item():.4g} mean {err.mean().item():.4g}; "
          f"bf16 oracle vs fp32 oracle: max {ref_self:.4g}")
    assert err.max().item() <= max(2e-2, ref_self)
    assert err.mean().item() <= 1e-2
    if scored is not None:
        assert err[scored].max().item() <= 2e-2


def spearman(a, b):
    ra = np.argsort(np.argsort(a)).astype(np.float64)
    rb = np.argsort(np.argsort(b)).astype(np.float64)
    return float(np.corrcoef(ra, rb)[0, 1])


@pytest.fixture(scope="module")
def Model(cuda_device):
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    return CaduceusForMaskedLM


SMALL = [dict(d_model=128, n_layer=2), dict(d_model=256, n_layer=3, residual_in_fp32=True)]


@pytest.mark.parametrize("kw", SMALL)
@pytest.mark.parametrize("B,L", [(3, 64), (1, 37), (2, 512), (1, 1)])
def test_fp32_logits_and_hidden_match_oracle(Model, cuda_device, kw, B, L):
    cfg = CaduceusConfig(**kw)
    sd = random_init_state_dict(cfg, seed=1)
    ids = make_ids(B, L, seed=B * 1000 + L, mask_at=L // 2)
    want_logits, want_hs = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32, output_hidden_states=True)
    model = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.float32).to(cuda_device)
    out = model(input_ids=ids.to(cuda_device), output_hidden_states=True)
    assert out.logits.dtype == torch.float32 and out.logits.shape == (B, L, 8)
    assert out.hidden_states[-1].shape == (B, L, 2 * cfg.d_model)
    assert rel_err(out.logits.cpu(), want_logits) <= 1e-4
    assert rel_err(out.hidden_states[-1].cpu(), want_hs[-1]) <= 1e-4


@pytest.mark.parametrize("kw", SMALL)
def test_bf16_logits_match_oracle(Model, cuda_device, kw):
    cfg = CaduceusConfig(**kw)
    sd = random_init_state_dict(cfg, seed=2)
    ids = make_ids(4, 128, seed=9, mask_at=64)
    want, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32)
    want_bf16, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.bfloat16)
    model = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
    got = model(input_ids=ids.to(cuda_device)).logits.cpu()
    assert_bf16_parity(got, want, want_bf16, scored=(slice(None), 64, slice(3, 7)))


def test_l20_fp32_and_bf16_real_shape(Model, cuda_device):
    """BASELINE.json config 1 shape: PlantCaduceus_l20 (d 384, 20 layers), 512-bp windows, masked at 255."""
    cfg = preset("PlantCaduceus_l20")
    sd = random_init_state_dict(cfg, seed=0)
    ids = make_ids(2, 512, seed=4, mask_at=255)
    want, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32)
    m32 = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.float32).to(cuda_device)
    got32 = m32(input_ids=ids.to(cuda_device)).logits.cpu()
    assert rel_err(got32, want) <= 1e-4
    del m32
    m16 = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
    got16 = m16(input_ids=ids.to(cuda_device)).logits.cpu()
    want16, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.bfloat16)
    assert_bf16_parity(got16, want, want16, scored=(slice(None), 255, slice(3, 7)))


@pytest.mark.parametrize("name", ["PlantCaduceus_l24", "PlantCaduceus_l28", "PlantCaduceus_l32"])
def test_published_widths_two_layers(Model, cuda_device, name):
    """The other published sizes (d 512 / 768 / 1024; x_proj widths 64 / 80 / 96; dt_rank 32 / 48 / 64) at 2 layers so the
    oracle finishes: every GEMM tile configuration and the real channel counts, fp32 and bf16, residual_in_fp32 on and off."""
    for res32 in (False, True):
        cfg = preset(name, n_layer=2, residual_in_fp32=res32)
        sd = random_init_state_dict(cfg, seed=5)
        ids = make_ids(2, 512, seed=7, mask_at=255)
        want, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32)
        m32 = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.float32).to(cuda_device)
        assert rel_err(m32(input_ids=ids.to(cuda_device)).logits.cpu(), want) <= 1e-4
        del m32
        m16 = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
        got16 = m16(input_ids=ids.to(cuda_device)).logits.cpu()
        want16, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.bfloat16)
        assert_bf16_parity(got16, want, want16, scored=(slice(None), 255, slice(3, 7)))
        del m16


def test_bf16_fused_norm_matches_unfused(Model, cuda_device, monkeypatch):
    """The bf16 forward folds add+RMSNorm into the out_proj / in_proj epilogues; PCAD_NO_FUSED_NORM=1 runs the
    separate norm kernel instead.  Both must sit at the same distance from the fp32 oracle."""
    cfg = CaduceusConfig(d_model=256, n_layer=4)
    sd = random_init_state_dict(cfg, seed=8)
    ids = make_ids(3, 200, seed=2, mask_at=100)
    want, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32)
    fused = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
    a = fused(input_ids=ids.to(cuda_device)).logits.cpu()
    monkeypatch.setenv("PCAD_NO_FUSED_NORM", "1")
    unfused = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
    b = unfused(input_ids=ids.to(cuda_device)).logits.cpu()
    assert fused.launch_count() < unfused.launch_count()
    ea, eb = (a - want).abs().max().item(), (b - want).abs().max().item()
    print(f"fused {ea:.4g}  unfused {eb:.4g}")
    assert ea <= max(2e-2, 1.5 * eb)
    assert (a - b).abs().max().item() <= 2e-2


@pytest.mark.parametrize("B,L,mask_at", [(3, 200, 100), (2, 37, 5), (1, 512, 255), (2, 16, 15), (1, 1024, 1000), (96, 512, 255),
                                         (40, 528, 100)])
def test_scan_fp32_bc_rows_mode_is_bit_identical(Model, cuda_device, monkeypatch, B, L, mask_at):
    """The forward converts B|C to fp32 rows once per layer (bc_to_f32_kernel) and runs the scan in its one-barrier mode
    (scan.cuh kScanBcF32); PCAD_SCAN_BC_F32=0 keeps the in-kernel conversion.  Same arithmetic in the same order: the logits,
    the hidden states and the score-only entry point (pruned last layer) must be bit-identical, ragged lengths included."""
    cfg = CaduceusConfig(d_model=256, n_layer=3)
    sd = random_init_state_dict(cfg, seed=7)
    ids = make_ids(B, L, seed=3, mask_at=mask_at)
    outs = []
    for flag in ("1", "0"):
        monkeypatch.setenv("PCAD_SCAN_BC_F32", flag)
        m = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
        o = m(input_ids=ids.to(cuda_device), output_hidden_states=True)
        sc = m.score_masked(ids.to(cuda_device), mask_at)
        outs.append((o.logits.cpu(), o.hidden_states[-1].cpu(), sc.cpu(), m.launch_count()))
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][1], outs[1][1])
    assert torch.equal(outs[0][2], outs[1][2])
    assert not torch.isnan(outs[0][0]).any()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_engine_rc_equivariance(Model, cuda_device, dtype):
    """Size-independent property (SURVEY.md 8c (1)): logits(RC(ids)) == logits(ids).flip(L)[..., comp]."""
    cfg = CaduceusConfig(d_model=256, n_layer=4)
    sd = random_init_state_dict(cfg, seed=3)
    ids = make_ids(3, 96, seed=5, mask_at=40)
    comp = torch.tensor([cfg.complement_map[i] for i in range(8)])
    model = Model.from_pretrained(sd, config=cfg, torch_dtype=dtype).to(cuda_device)
    a = model(input_ids=ids.to(cuda_device), output_hidden_states=True)
    b = model(input_ids=O.reverse_complement_ids(ids, cfg).to(cuda_device), output_hidden_states=True)
    # both strands run the same kernels on the same numbers, so equivariance is exact up to the order of
    # the two-term sum in the head (commutative) -- require tight agreement
    tol = 1e-5 if dtype == torch.float32 else 1e-5
    assert (b.logits.cpu() - a.logits.cpu().flip(1)[..., comp]).abs().max().item() <= tol
    assert torch.equal(b.hidden_states[-1].cpu(), a.hidden_states[-1].cpu().flip(1, 2))


def test_score_paths_agree_and_llr_spearman(Model, cuda_device):
    cfg = CaduceusConfig(d_model=256, n_layer=4)
    sd = random_init_state_dict(cfg, seed=6)
    tok = CharDNATokenizer()
    rng = np.random.default_rng(0)
    B, L, idx = 48, 512, 255
    ascii_np = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=(B, L))
    ascii_np[3, 10] = ord("N")
    ascii_np[5, 100] = ord("a")   # lower case folds
    seqs = [bytes(r).decode() for r in ascii_np]
    # reference-style host path (zero_shot_score.py:49-62): per-sequence encode_plus + mask
    ids = torch.cat([tok.encode_plus(s, return_tensors="pt")["input_ids"] for s in seqs])
    ids[:, idx] = tok.mask_token_id
    want, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32)
    acgt = [tok.get_vocab()[c] for c in "acgt"]
    want4 = want[:, idx, acgt]

    model = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
    full = model(input_ids=ids.to(cuda_device)).logits[:, idx, acgt].cpu()
    masked = model.score_masked(ids.to(torch.uint8).to(cuda_device), torch.full((B, 1), idx, dtype=torch.int32)).cpu()[:, 0]
    host = model.score_windows_host(torch.from_numpy(ascii_np).pin_memory(), idx).clone()
    assert torch.equal(full, masked)
    assert torch.equal(full, host)
    assert (full - want4).abs().max().item() <= 2e-2
    # LLR for every (ref, alt) pair with ref = the window's own base
    refs = ["ACGT".index(chr(c).upper()) for c in ascii_np[:, idx]]
    llr_got, llr_want = [], []
    for i, r in enumerate(refs):
        for a in range(4):
            if a != r:
                llr_got.append(float(full[i, a] - full[i, r]))
                llr_want.append(float(want4[i, a] - want4[i, r]))
    assert spearman(np.array(llr_got), np.array(llr_want)) >= 0.999
    # multi-mask gather (zero-shot-eval.py:129-140)
    pos = torch.tensor([[0, 255, 511]] * B, dtype=torch.int32)
    multi = model.score_masked(ids.to(torch.uint8).to(cuda_device), pos).cpu()
    full_all = model(input_ids=ids.to(cuda_device)).logits.cpu()
    assert torch.equal(multi, full_all[:, [0, 255, 511]][:, :, acgt])


def test_device_tokenizer_bit_exact(Model, cuda_device):
    cfg = CaduceusConfig(d_model=128, n_layer=1)
    model = Model.from_random(cfg, seed=0).to(cuda_device)
    tok = CharDNATokenizer()
    all_bytes = torch.arange(256, dtype=torch.uint8).repeat(5)
    got = model.tokenize_device(all_bytes.to(cuda_device)).cpu().numpy()
    assert np.array_equal(got, tok.encode_bytes(all_bytes.numpy()))


def test_errors_are_reported_not_fatal(Model, cuda_device):
    from plantcaduceus_b200._lib import PcadError
    with pytest.raises(ValueError):
        Model.from_random(CaduceusConfig(d_model=128, n_layer=1, rcps=False))
    cfg = CaduceusConfig(d_model=128, n_layer=1)
    sd = random_init_state_dict(cfg, seed=0)
    sd2 = {k: v for k, v in sd.items() if "layers.0.norm" not in k}
    with pytest.raises(PcadError, match="missing weight"):
        Model.from_pretrained(sd2, config=cfg).to(cuda_device)
    m = Model.from_pretrained(sd, config=cfg)
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(input_ids=torch.zeros(1, 8, dtype=torch.long))
    m.to(cuda_device)
    out = m(input_ids=torch.zeros(0, 8, dtype=torch.long, device=cuda_device))
    assert out.logits.shape == (0, 8, 8)


def test_full_size_l32_properties(Model, cuda_device):
    """BASELINE.json configs[1] at full model size (PlantCaduceus_l32, 32 layers, bf16, 512-bp windows), where the CPU
    oracle is too slow to be the checker: size-independent properties instead.
      * RC equivariance: the hidden states of RC(ids) are the flipped hidden states of ids, bit for bit (both strands run
        the same kernels on the same numbers), and the logits agree to fp32 summation order;
      * batch independence: a window scores the same alone, inside a batch, and through every entry point;
      * determinism: two runs are bit-identical."""
    cfg = preset("PlantCaduceus_l32")
    sd = random_init_state_dict(cfg, seed=0)
    model = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
    B, L, idx = 24, 512, 255
    ids = make_ids(B, L, seed=31, mask_at=idx)
    comp = torch.tensor([cfg.complement_map[i] for i in range(8)])
    a = model(input_ids=ids.to(cuda_device), output_hidden_states=True)
    b = model(input_ids=O.reverse_complement_ids(ids, cfg).to(cuda_device), output_hidden_states=True)
    assert torch.equal(b.hidden_states[-1].cpu(), a.hidden_states[-1].cpu().flip(1, 2))
    assert (b.logits.cpu() - a.logits.cpu().flip(1)[..., comp]).abs().max().item() <= 1e-4
    assert torch.isfinite(a.logits).all()
    # batch independence + entry points
    acgt = [3, 4, 5, 6]
    full = a.logits[:, idx, acgt].cpu()
    alone = model(input_ids=ids[5:6].to(cuda_device)).logits[:, idx, acgt].cpu()
    assert torch.equal(alone[0], full[5])
    masked = model.score_masked(ids.to(torch.uint8), torch.full((B, 1), idx, dtype=torch.int32)).cpu()[:, 0]
    assert torch.equal(masked, full)
    again = model(input_ids=ids.to(cuda_device)).logits.cpu()
    assert torch.equal(again, a.logits.cpu())


def test_two_devices_in_one_process(Model, cuda_device):
    """Distinct handles are independent (include/pcad.h): two engines on two GPUs of one process give the same bits."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cfg = CaduceusConfig(d_model=256, n_layer=3)
    sd = random_init_state_dict(cfg, seed=13)
    ids = make_ids(4, 256, seed=3, mask_at=128)
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        m = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(dev)
        outs.append(m(input_ids=ids.to(dev)).logits.cpu())
    assert torch.equal(outs[0], outs[1])


def test_small_batch_cuda_graph_replay_is_bit_identical(Model, cuda_device, monkeypatch):
    """Small score-only forwards are launch-bound (~8 launches per layer of a few microseconds each); from the third call with
    a shape they are replayed from a CUDA graph captured on the second.  Same bits as eager launches, same launch accounting,
    and a change of shape / tokenizer in between does not replay a stale graph."""
    cfg = CaduceusConfig(d_model=256, n_layer=4)
    sd = random_init_state_dict(cfg, seed=21)
    rng = np.random.default_rng(4)
    batches = [torch.from_numpy(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=(3, 512))).pin_memory() for _ in range(5)]
    other = torch.from_numpy(rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), size=(2, 300))).pin_memory()
    monkeypatch.setenv("PCAD_NO_GRAPH", "1")
    eager = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
    want = [eager.score_windows_host(b, 255).clone() for b in batches]
    want_other = eager.score_windows_host(other, 100).clone()
    n_eager = eager.launch_count()
    monkeypatch.delenv("PCAD_NO_GRAPH")
    graphed = Model.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(cuda_device)
    got = []
    for k, b in enumerate(batches):
        got.append(graphed.score_windows_host(b, 255).clone())
        if k == 2:   # a different shape and position in between: its own (eager) path, the cached graph stays valid
            assert torch.equal(graphed.score_windows_host(other, 100), want_other)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    assert graphed.launch_count() == n_eager
    # device entry point shares the graphs
    dev_out = graphed.score_windows_device(batches[0].to(cuda_device), 255).cpu()
    assert torch.equal(dev_out, want[0])
    # a new tokenizer invalidates the captured launches (mask id / column selection are baked in)
    vocab = {"[PAD]": 0, "[UNK]": 1, "[MASK]": 2, "t": 3, "a": 4, "g": 5, "c": 6}
    tok = CharDNATokenizer(vocab=vocab)
    graphed.set_tokenizer(tok)
    eager.set_tokenizer(tok)
    for _ in range(3):
        assert torch.equal(graphed.score_windows_host(batches[1], 255), eager.score_windows_host(batches[1], 255))


@pytest.mark.parametrize("kw,dtype", [(dict(d_model=256, n_layer=3), torch.bfloat16), (dict(d_model=128, n_layer=1), torch.bfloat16),
                                      (dict(d_model=256, n_layer=2, residual_in_fp32=True), torch.bfloat16),
                                      (dict(d_model=128, n_layer=2), torch.float32),
                                      (dict(d_model=128, n_layer=1), torch.float32),
                                      (dict(d_model=128, n_layer=1, residual_in_fp32=True), torch.bfloat16)])
def test_score_only_last_layer_pruning_is_bit_identical(Model, cuda_device, monkeypatch, kw, dtype):
    """Score-only calls compute the last layer only as far as the head needs it (the scan stops once both directions have reached
    the scored position; out_proj, residual add and final norm run on the 2B rows the head reads).  Same bits as the full
    computation (PCAD_NO_PRUNE=1) and as the logits of the full forward, for positions at the centre, the edges and off-centre,
    even and odd window lengths."""
    cfg = CaduceusConfig(**kw)
    sd = random_init_state_dict(cfg, seed=17)
    rng = np.random.default_rng(6)
    pruned = Model.from_pretrained(sd, config=cfg, torch_dtype=dtype).to(cuda_device)
    monkeypatch.setenv("PCAD_NO_PRUNE", "1")
    full = Model.from_pretrained(sd, config=cfg, torch_dtype=dtype).to(cuda_device)
    tok = CharDNATokenizer()
    for L, idxs in ((512, (255, 0, 511, 100, 300)), (301, (150, 7, 299)), (33, (16, 32))):
        a = torch.from_numpy(rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), size=(5, L))).pin_memory()
        for idx in idxs:
            got = pruned.score_windows_host(a, idx).clone()
            want = full.score_windows_host(a, idx).clone()
            assert torch.equal(got, want), (L, idx)
            ids = torch.from_numpy(tok.encode_bytes(a.numpy()).astype(np.int64))
            ids[:, idx] = tok.mask_token_id
            logits = full(input_ids=ids.to(cuda_device)).logits[:, idx, 3:7].cpu()
            assert torch.equal(got, logits), (L, idx)
            # ids resident on the device + one shared index (pcad_score_masked_at) and per-row positions (pcad_score_masked)
            assert torch.equal(pruned.score_masked(ids.to(torch.uint8), idx).cpu()[:, 0], got)
            assert torch.equal(pruned.score_masked(ids.to(torch.uint8), torch.full((5, 1), idx, dtype=torch.int32)).cpu()[:, 0], got)
    assert pruned.launch_count() != full.launch_count()
