"""Engine state across calls: what a handle does once it carries state from earlier calls.

The parity files check one call on a fresh handle.  A handle also keeps state between calls: the workspace (grown by
reallocation, re-laid out for every call's (B, L)), the CUDA graphs of the score path (one per (B, L, token_idx), captured
on the second call, replayed from the third on an internal stream ordered by events), and the weights and tokenizer tables
that pcad_set_weight / pcad_finalize / pcad_set_tokenizer rewrite in place.  Checked here, every output bit for bit:

A. the graphed score path (pcad_score_windows_host / _dev) at every preset and mode, against pcad_score_masked_at on
   host-tokenised ids on a PCAD_NO_GRAPH handle, whose pcad_forward logits must hold the same bits; pcad_graph_replays
   shows which calls replayed a graph;
B. graph and workspace lifetimes on one handle: a reallocation between capture and replay, shape ping-pong inside one
   allocation, a new token_idx, profiling, a new tokenizer;
C. every entry point interleaved on a side stream with no host synchronisation in between, and two handles on two streams;
D. a live handle reloaded with a second state dict, and a reload while work is still queued on a side stream.

`GraphCache` restates the engine's graph bookkeeping (score_core_graphed and ensure_workspace in csrc/pcad.cu); the GPU
tests check the replay counter against it call by call, and the device-free tests check it, and the mode of every case
(graph or eager, time-parallel segments, fp32 B|C rows, the pruned scan's length), against values worked out by hand.

Run with -s to see the file's wall time and peak device memory."""
import ctypes as C
import time

import numpy as np
import pytest
import torch

from plantcaduceus_b200.tokenizer import CharDNATokenizer
from plantcaduceus_b200.weights import EMB_KEY, HEAD_KEY, random_init_state_dict
from test_forward_replay_gpu import B200_SMS, SWITCHES, first_difference, forward_modes, two_layers
from test_kernel_bounds_gpu import ALL_PRESETS, BF16, DEV, F32, PLANTCAD2, TD

GRAPH_MAX_TOKENS = 65536     # pcad_handle::graph_max_tokens: strand-tokens 2 B L up to which a score call is graphed
ENGINE_ENV = SWITCHES + ("PCAD_NO_GRAPH", "PCAD_GRAPH_MAX_TOKENS")
CALLS = 4                    # calls per shape: eager, capture, then replays
SLEEP_CYCLES = 100_000_000   # torch.cuda._sleep: about 50 ms at the B200's clock, a fixed spin, not a wait


# ---- the graph bookkeeping, restated ------------------------------------------------------------------------------------
class GraphCache:
    """What score_core_graphed and ensure_workspace decide per call.  Every forward entry point first makes the workspace
    fit (B, L): a larger one is a new allocation, and the graphs, whose launches point into the old one, are dropped.  A
    score call (score_windows_host / _dev) with 2 B L <= max_tokens, graphs enabled and profiling off then runs eagerly the
    first time its (B, L, token_idx) is seen, captures and launches the graph the second time, and replays it from then
    on.  set_weight and set_tokenizer drop the graphs."""

    def __init__(self, use_graphs=True, max_tokens=GRAPH_MAX_TOKENS):
        self.use_graphs, self.max_tokens = use_graphs, max_tokens
        self.alloc, self.graphs = 0, {}

    def call(self, need, B=0, L=0, idx=None, profiling=False):
        """need: the call's workspace bytes, None for tokenize / extract_windows (no workspace); idx None: not a score call.
        Returns "eager", "capture" or "replay"."""
        if need is not None and need > self.alloc:
            self.graphs.clear()
            self.alloc = need
        if idx is None or not self.use_graphs or profiling or 2 * B * L > self.max_tokens:
            return "eager"
        state = self.graphs.get((B, L, idx))
        if state is None:
            self.graphs[(B, L, idx)] = "seen"
            return "eager"
        if state == "seen":
            self.graphs[(B, L, idx)] = "exec"
            return "capture"
        return "replay"

    def drop(self):
        self.graphs.clear()


def plan(name, mode, B, L, idx, ssd_seq=False):
    """(graphed, P, fp32 B|C rows, Lrun of the pruned last layer) of a score call, from the replay file's mode helpers."""
    cfg, dtype = config(name, mode)
    m = forward_modes(cfg, B, L, dtype, B200_SMS, ssd_seq)
    return (2 * B * L <= GRAPH_MAX_TOKENS, m.P, m.bc_rows, m.lrun(cfg, L, idx))


def config(name, mode):
    return two_layers(name, **({"residual_in_fp32": True} if mode == "bf16-res32" else {})), F32 if mode == "f32" else BF16


# ---- A: the case table -------------------------------------------------------------------------------------------------
MODES3 = ("bf16", "bf16-res32", "f32")
# (B, L, token_idx): one window; the same batch scored at the centre, both edges (Lrun = L) and off-centre; the largest
# graphed batch at 512 bp (2 B L = 65536) and the smallest one that is not; L < 8, where the last layer is not pruned
SHORT = ((1, 512, 255), (32, 512, 0), (32, 512, 511), (32, 512, 255), (32, 512, 100), (64, 512, 255), (65, 512, 255),
         (5, 7, 3))
LONG1 = (1, 8192, 4095)
LONGEST = (1, 32768, 16383)


def a_case(name, mode, shapes, ssd_seq=False):
    tag = f"{name}-{mode}" + ("-ssdseq" if ssd_seq else "") + ("" if shapes is SHORT else f"-L{shapes[0][1]}")
    return pytest.param(name, mode, shapes, ssd_seq, id=tag)


A_CASES = ([a_case(n, m, SHORT) for n in ALL_PRESETS for m in MODES3]
           + [a_case("PlantCAD2-Small-l24-d0768", "bf16", SHORT, ssd_seq=True)]
           + [a_case(n, m, (LONG1,)) for n in ("PlantCaduceus_l20", "PlantCaduceus_l32") for m in MODES3]
           + [a_case("PlantCaduceus_l20", m, (LONGEST,)) for m in ("bf16", "bf16-res32")]
           + [a_case(n, "bf16", (LONG1,)) for n in PLANTCAD2]
           + [a_case("PlantCAD2-Small-l24-d0768", "bf16", (LONG1,), ssd_seq=True)])


def test_case_table_modes_match_hand_derived_values():
    """Needs no device: every case of A takes the path it is there for, worked out by hand for a 148-SM B200.  The
    PlantCaduceus presets at 512 bp: graphed up to B = 64, one segment, fp32 B|C rows in bf16 from B = 64
    (T = 65536), the last layer's scan max(p, L-1-p) + 1 steps long.  One window of 8192 bp: graphed and time-parallel (l20: 12
    channel blocks per strand, 16 segments; l32: 32 blocks, 8 segments), not pruned.  l20 at 32768 bp: T = 65536, the
    last graphed size, also fp32 B|C rows in bf16.  PlantCAD2 is never pruned or segmented."""
    lrun512 = {0: 512, 511: 512, 255: 257, 100: 412}
    for p in A_CASES:
        name, mode, shapes, ssd_seq = p.values
        m1 = not name.startswith("PlantCAD2")
        for B, L, idx in shapes:
            got = plan(name, mode, B, L, idx, ssd_seq)
            if L == 512:
                want = (B <= 64, 1, m1 and mode != "f32" and B >= 64, lrun512[idx] if m1 else 0)
            elif L == 7:
                want = (True, 1, False, 0)
            elif L == 8192:
                want = (True, {"PlantCaduceus_l20": 16, "PlantCaduceus_l32": 8}.get(name, 1), False, 0)
            else:
                assert (name, L) == ("PlantCaduceus_l20", 32768)
                want = (True, 16, True, 0)
            assert got == want, (p.id, B, L, idx)
    # the boundary: B = 64 is the largest graphed batch at 512 bp and B = 65 the smallest eager one; both are in the table
    assert 2 * 64 * 512 == GRAPH_MAX_TOKENS and 2 * 65 * 512 > GRAPH_MAX_TOKENS
    # every preset and mode at one window and at the 32-window batch
    covered = {(p.values[0], p.values[1]) for p in A_CASES if p.values[2] is SHORT}
    assert covered == {(n, m) for n in ALL_PRESETS for m in MODES3}


def test_graph_cache_script():
    """Needs no device: GraphCache on A's per-shape sequence and on B's and C's scripts, against outcomes worked out by
    hand (workspace bytes stand in as B L: the layout grows with both)."""
    g = GraphCache()
    assert [g.call(512, 1, 512, 255) for _ in range(CALLS)] == ["eager", "capture", "replay", "replay"]
    assert [g.call(65 * 512, 65, 512, 255) for _ in range(3)] == ["eager"] * 3
    assert [GraphCache(max_tokens=0).call(512, 1, 512, 255) for _ in range(3)] == ["eager"] * 3
    assert [GraphCache(use_graphs=False).call(512, 1, 512, 255) for _ in range(3)] == ["eager"] * 3
    g, outcomes = GraphCache(), []
    for B, L, idx, prof in B_SCRIPT:
        if prof == "tokenizer":
            g.drop()
        else:
            outcomes.append(g.call(B * L, B, L, idx, prof))
    assert outcomes == B_OUTCOMES
    g = GraphCache()
    outcomes = [g.call(None if op in ("tokenize", "extract_windows") else args[0] * args[1], args[0], args[1],
                       args[2] if op == "score_windows_dev" else None) for op, *args in C_SCRIPT]
    assert [o for o, (op, *_) in zip(outcomes, C_SCRIPT) if op == "score_windows_dev"] == C_WINDOW_OUTCOMES


# ---- B and C: the scripts ------------------------------------------------------------------------------------------------
# (B, L, token_idx, profiling); (0, 0, 0, "tokenizer") marks set_tokenizer with a permuted vocabulary
PING = ((8, 512, 255, False), (16, 512, 255, False), (8, 512, 255, False), (3, 300, 100, False), (8, 512, 255, False))
B_SCRIPT = (((8, 512, 255, False),) * 3 + ((256, 512, 255, False),) + ((8, 512, 255, False),) * 3 + PING * 2
            + ((8, 512, 100, False),) * 3 + ((8, 512, 255, True),) * 2 + ((8, 512, 255, False),)
            + ((0, 0, 0, "tokenizer"),) + ((8, 512, 255, False),) * 3)
E, Cp, R = "eager", "capture", "replay"
B_OUTCOMES = ([E, Cp, R] + [E]                   # capture at (8, 512); (256, 512) reallocates: graphs dropped
              + [E, Cp, R]                       # the old exec is not replayed
              + [R, E, R, E, R] + [R, Cp, R, Cp, R]   # inside the (256, 512) allocation: every shape keeps its graph
              + [E, Cp, R]                       # a new token_idx is a new graph
              + [E, E, R]                        # profiling runs eagerly; the graph is still there afterwards
              + [E, Cp, R])                      # a new tokenizer drops the graphs

# (op, B, L, extra): extra is token_idx (score_masked_at, score_windows_dev, extract_windows) or positions per window
C_SCRIPT = (("score_windows_dev", 4, 512, 255), ("forward", 2, 300, None), ("score_windows_dev", 4, 512, 255),
            ("score_windows_dev", 4, 512, 255), ("tokenize", 4, 512, None), ("score_masked_at", 3, 512, 255),
            ("extract_windows", 4, 512, 255), ("score_windows_dev", 4, 512, 255), ("hidden_at", 3, 600, 5),
            ("forward", 128, 512, None),          # reallocates after a capture: the graph is dropped
            ("score_windows_dev", 4, 512, 255), ("score_masked", 16, 512, 3), ("score_windows_dev", 4, 512, 255),
            ("score_windows_dev", 80, 512, 255),  # 2 B L = 81920: eager, inside the (128, 512) allocation
            ("score_windows_dev", 4, 512, 255), ("forward", 1, 9, None), ("score_masked_at", 2, 7, 3),
            ("hidden_at", 5, 512, 2), ("score_windows_dev", 4, 512, 255), ("tokenize", 1, 1000, None))
C_WINDOW_OUTCOMES = [E, Cp, R, R, E, Cp, E, R, R]


# ---- helpers -----------------------------------------------------------------------------------------------------------
STATS = {"workspace": 0}


@pytest.fixture(scope="module")
def lib(cuda_device):
    from plantcaduceus_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def budget():
    """Wall time and peak device memory of the file's GPU tests (printed with -s): torch's allocations and the largest
    workspace an engine of the file held."""
    if not torch.cuda.is_available():
        yield
        return
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    torch.cuda.synchronize()
    print(f"\n[state] file: wall {time.time() - t0:.1f} s, peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} "
          f"GiB in torch, largest engine workspace {STATS['workspace'] / 2 ** 30:.2f} GiB")


@pytest.fixture
def env(monkeypatch, budget):
    """No PCAD_* switch set, graphs on: the engine picks its modes from the shape."""
    for k in ENGINE_ENV:
        monkeypatch.delenv(k, raising=False)
    yield monkeypatch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def engine(env, cfg, sd, dtype, graphs=True, **switches):
    """A handle loaded with sd; graphs=False: PCAD_NO_GRAPH=1.  PCAD_* switches hold only while it is created."""
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    set_env = dict(switches, **({} if graphs else {"PCAD_NO_GRAPH": "1"}))
    for k, v in set_env.items():
        env.setenv(k, v)
    try:
        return CaduceusForMaskedLM.from_pretrained(sd, config=cfg, torch_dtype=TD[dtype]).to(DEV)
    finally:
        for k in set_env:
            env.delenv(k)


def replays(lib, model):
    return int(lib.pcad_graph_replays(model._handle))


def windows(B, L, seed):
    """ASCII windows, mostly ACGT, with lower case, N and bytes outside the alphabet (UNK) at about 10 % of positions."""
    g = np.random.default_rng(seed)
    a = g.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=(B, L))
    spots = g.random((B, L)) < 0.1
    a[spots] = g.choice(np.frombuffer(b"acgtNnRYk-.\x00\xff", dtype=np.uint8), size=int(spots.sum()))
    return torch.from_numpy(a)


def host_ids(tok, ascii, idx):
    """The host tokeniser (the tokenizer's LUT) with position idx of every window masked: uint8 [B, L]."""
    ids = torch.from_numpy(tok.lut[ascii.numpy()])
    ids[:, idx] = tok.mask_token_id
    return ids


def acgt_ids(tok):
    v = tok.get_vocab()
    return [v[c] for c in "acgt"]


def permuted_tokenizer():
    return CharDNATokenizer(vocab={"[PAD]": 0, "[UNK]": 1, "[MASK]": 2, "t": 3, "a": 4, "g": 5, "c": 6})


def score_call(model, ascii, idx, k):
    """Call k of a shape: score_windows_host on even k, score_windows_dev on odd k.  Returns host [B, 4]."""
    if k % 2 == 0:
        return model.score_windows_host(ascii.pin_memory(), idx).clone()
    return model.score_windows_device(ascii.to(DEV), idx).cpu()


def reference(eager, tok, ascii, idx):
    """pcad_score_masked_at on host-tokenised, masked ids (PCAD_NO_GRAPH handle): (logits [B, 4], launches)."""
    n0 = eager.launch_count()
    out = eager.score_masked(host_ids(tok, ascii, idx).to(DEV), idx)[:, 0].cpu()
    return out, eager.launch_count() - n0


# ---- A -------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,mode,shapes,ssd_seq", A_CASES)
def test_graphed_score_path_is_bit_identical(lib, env, name, mode, shapes, ssd_seq):
    """At every shape, CALLS score calls with new window contents each, alternating the host and device entries: each is
    bit-identical to pcad_score_masked_at on a PCAD_NO_GRAPH handle with the same weights, whose pcad_forward logits at
    token_idx hold the same bits.  pcad_graph_replays counts every call from the third on where the shape is graphed and
    none where it is not; the launch counts equal the eager handle's."""
    cfg, dtype = config(name, mode)
    sd = random_init_state_dict(cfg, seed=7)
    sw = {"PCAD_SSD_SEQ": "1"} if ssd_seq else {}
    eager = engine(env, cfg, sd, dtype, graphs=False, **sw)
    graph = engine(env, cfg, sd, dtype, **sw)
    tok = CharDNATokenizer()
    cols = acgt_ids(tok)
    for B, L, idx in shapes:
        graphed = plan(name, mode, B, L, idx, ssd_seq)[0]
        STATS["workspace"] = max(STATS["workspace"], graph.workspace_bytes(B, L))
        r0, n0, n_eager = replays(lib, graph), graph.launch_count(), 0
        for k in range(CALLS):
            ascii = windows(B, L, seed=B * 1000003 + L * 1009 + idx * 7 + k)
            got = score_call(graph, ascii, idx, k)
            want, n = reference(eager, tok, ascii, idx)
            n_eager += n
            label = f"{name} {mode} B={B} L={L} idx={idx} call {k + 1}"
            assert torch.equal(got, want), f"{label}: {first_difference(got, want)}"
            assert replays(lib, graph) - r0 == (max(0, k - 1) if graphed else 0), label
            if k == 0:
                ids = host_ids(tok, ascii, idx).to(DEV, torch.int64)
                lg = eager(input_ids=ids).logits[:, idx][:, cols].cpu()
                assert torch.equal(lg, want), f"{label}: pcad_forward's logits: {first_difference(lg, want)}"
                del ids
        assert graph.launch_count() - n0 == n_eager, f"{name} {mode} B={B} L={L} idx={idx}: launch counts"
    eager._release()
    graph._release()


@pytest.mark.gpu
def test_graphs_off_are_never_replayed(lib, env):
    """PCAD_GRAPH_MAX_TOKENS=0 and PCAD_NO_GRAPH=1: the same bits, no replay."""
    cfg, dtype = config("PlantCaduceus_l20", "bf16")
    sd = random_init_state_dict(cfg, seed=3)
    ref = engine(env, cfg, sd, dtype, graphs=False)
    tok = CharDNATokenizer()
    for off in (engine(env, cfg, sd, dtype, PCAD_GRAPH_MAX_TOKENS="0"), engine(env, cfg, sd, dtype, graphs=False)):
        for k in range(CALLS):
            ascii = windows(4, 512, seed=100 + k)
            assert torch.equal(score_call(off, ascii, 255, k), reference(ref, tok, ascii, 255)[0])
        assert replays(lib, off) == 0
        off._release()
    ref._release()


# ---- B -------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_graph_and_workspace_lifetimes(lib, env):
    """B_SCRIPT on one handle: a capture at (8, 512), a reallocation by (256, 512), shape ping-pong inside one allocation, a
    new token_idx, two profiled calls, a permuted vocabulary.  Every call has new contents and equals the eager handle's
    pcad_score_masked_at; the replay counter moves exactly where GraphCache, fed the engine's workspace sizes, says, and
    the launch counts equal the eager handle's."""
    cfg, dtype = config("PlantCaduceus_l20", "bf16")
    sd = random_init_state_dict(cfg, seed=5)
    eager, graph = engine(env, cfg, sd, dtype, graphs=False), engine(env, cfg, sd, dtype)
    tok = CharDNATokenizer()
    cache = GraphCache()
    n0, n_eager = graph.launch_count(), 0
    outcomes = []
    for k, (B, L, idx, prof) in enumerate(B_SCRIPT):
        if prof == "tokenizer":
            tok = permuted_tokenizer()
            graph.set_tokenizer(tok)
            eager.set_tokenizer(tok)
            cache.drop()
            continue
        graph.set_profiling(prof)
        r0 = replays(lib, graph)
        ascii = windows(B, L, seed=1000 + k)
        got = score_call(graph, ascii, idx, k)
        want, n = reference(eager, tok, ascii, idx)
        n_eager += n
        outcomes.append(cache.call(graph.workspace_bytes(B, L), B, L, idx, prof))
        assert torch.equal(got, want), f"call {k} {(B, L, idx)} ({outcomes[-1]}): {first_difference(got, want)}"
        assert replays(lib, graph) - r0 == (outcomes[-1] == "replay"), f"call {k} {(B, L, idx)}: expected {outcomes[-1]}"
    graph.set_profiling(False)
    assert outcomes == B_OUTCOMES
    assert graph.launch_count() - n0 == n_eager
    STATS["workspace"] = max(STATS["workspace"], graph.workspace_bytes(256, 512))
    eager._release()
    graph._release()


# ---- C -------------------------------------------------------------------------------------------------------------------
class Script:
    """C_SCRIPT's inputs and output buffers for one model, made before any call; `run` issues the calls through the C ABI."""

    def __init__(self, cfg, dtype, seed):
        self.cfg, self.dtype = cfg, dtype
        g = torch.Generator().manual_seed(seed)
        self.chrom = windows(1, 5000, seed).reshape(-1).to(DEV)
        self.calls = []
        for k, (op, B, L, x) in enumerate(C_SCRIPT):
            a = {}
            if op in ("score_windows_dev", "tokenize"):
                a["ascii"] = windows(B, L, seed * 1000 + k).to(DEV)
            elif op == "extract_windows":
                a["pos0"] = torch.randint(0, 5000, (B,), generator=g).to(DEV)
            else:
                ids = torch.randint(0, 8, (B, L), generator=g)
                a["ids"] = (ids if op == "forward" else ids.to(torch.uint8)).to(DEV)
            if op in ("score_masked", "hidden_at"):
                a["pos"] = torch.randint(0, L, (B, x), generator=g, dtype=torch.int32).to(DEV)
            d2 = 2 * cfg.d_model
            a["out"] = {"forward": lambda: (torch.full((B, L, 8), float("nan"), device=DEV),
                                            torch.zeros(B, L, d2, dtype=TD[dtype], device=DEV)),
                        "score_masked": lambda: torch.full((B, x, 4), float("nan"), device=DEV),
                        "score_masked_at": lambda: torch.full((B, 4), float("nan"), device=DEV),
                        "hidden_at": lambda: torch.zeros(B, x, d2, dtype=TD[dtype], device=DEV),
                        "score_windows_dev": lambda: torch.full((B, 4), float("nan"), device=DEV),
                        "extract_windows": lambda: torch.zeros(B, L, dtype=torch.uint8, device=DEV),
                        "tokenize": lambda: torch.full((B, L), 255, dtype=torch.uint8, device=DEV)}[op]()
            self.calls.append((op, B, L, x, a))

    def issue(self, lib, h, k, stream):
        op, B, L, x, a = self.calls[k]
        p = lambda t: C.c_void_p(t.data_ptr())
        s = C.c_void_p(stream.cuda_stream)
        if op == "forward":
            rc = lib.pcad_forward(h, p(a["ids"]), B, L, p(a["out"][0]), p(a["out"][1]), s)
        elif op == "score_masked":
            rc = lib.pcad_score_masked(h, p(a["ids"]), p(a["pos"]), B, L, x, p(a["out"]), s)
        elif op == "score_masked_at":
            rc = lib.pcad_score_masked_at(h, p(a["ids"]), x, B, L, p(a["out"]), s)
        elif op == "hidden_at":
            rc = lib.pcad_hidden_at(h, p(a["ids"]), p(a["pos"]), B, L, x, p(a["out"]), s)
        elif op == "score_windows_dev":
            rc = lib.pcad_score_windows_dev(h, p(a["ascii"]), B, L, x, p(a["out"]), s)
        elif op == "extract_windows":
            rc = lib.pcad_extract_windows(h, p(self.chrom), self.chrom.numel(), p(a["pos0"]), B, L, x, p(a["out"]), s)
        else:
            rc = lib.pcad_tokenize(h, p(a["ascii"]), B * L, p(a["out"]), s)
        assert rc == 0, lib.pcad_last_error(h)

    def outputs(self):
        return [a["out"] if isinstance(a["out"], tuple) else (a["out"],) for *_, a in self.calls]


def reference_outputs(lib, env, cfg, sd, dtype, seed):
    """C_SCRIPT on a fresh PCAD_NO_GRAPH handle, synchronising after every call."""
    ref = engine(env, cfg, sd, dtype, graphs=False)
    sc = Script(cfg, dtype, seed)
    torch.cuda.synchronize()
    for k in range(len(C_SCRIPT)):
        sc.issue(lib, ref._handle, k, torch.cuda.current_stream())
        torch.cuda.synchronize()
    ref._release()
    return [tuple(t.cpu() for t in o) for o in sc.outputs()]


def compare_outputs(label, got, want):
    for k, ((op, B, L, x), g, w) in enumerate(zip(C_SCRIPT, got, want)):
        for gt, wt in zip(g, w):
            gt = gt.cpu()
            assert torch.equal(gt, wt), f"{label}: call {k} {op} B={B} L={L}: {first_difference(gt.float(), wt.float())}"


@pytest.mark.gpu
def test_interleaved_entry_points_on_a_side_stream(lib, env):
    """C_SCRIPT -- every entry point, shapes that grow and shrink, a reallocation between a capture and its replay -- on one
    handle and a torch side stream, one synchronisation at the end.  Every output equals the same call on a fresh
    PCAD_NO_GRAPH handle that synchronises after each call, and the replays are where GraphCache puts them."""
    cfg, dtype = config("PlantCaduceus_l32", "bf16")
    sd = random_init_state_dict(cfg, seed=9)
    want = reference_outputs(lib, env, cfg, sd, dtype, seed=9)
    model = engine(env, cfg, sd, dtype)
    sc = Script(cfg, dtype, seed=9)
    STATS["workspace"] = max(STATS["workspace"], model.workspace_bytes(128, 512))
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        for k in range(len(C_SCRIPT)):
            sc.issue(lib, model._handle, k, side)
    side.synchronize()
    compare_outputs("one handle", sc.outputs(), want)
    assert replays(lib, model) == C_WINDOW_OUTCOMES.count("replay")
    model._release()


@pytest.mark.gpu
def test_two_handles_on_two_streams(lib, env):
    """Distinct handles are independent: C_SCRIPT on PlantCaduceus_l32 and on PlantCAD2-Small, one device, each on its own
    side stream, the calls alternating between them with no synchronisation, equal each model's synchronised reference."""
    models = []
    for name, seed in (("PlantCaduceus_l32", 11), ("PlantCAD2-Small-l24-d0768", 12)):
        cfg, dtype = config(name, "bf16")
        sd = random_init_state_dict(cfg, seed=seed)
        models.append((name, reference_outputs(lib, env, cfg, sd, dtype, seed), engine(env, cfg, sd, dtype),
                       Script(cfg, dtype, seed), torch.cuda.Stream()))
    torch.cuda.synchronize()
    for k in range(len(C_SCRIPT)):
        for _, _, m, sc, st in models:
            with torch.cuda.stream(st):
                sc.issue(lib, m._handle, k, st)
    torch.cuda.synchronize()
    for name, want, m, sc, _ in models:
        compare_outputs(name, sc.outputs(), want)
        assert replays(lib, m) == C_WINDOW_OUTCOMES.count("replay")
        m._release()


# ---- D -------------------------------------------------------------------------------------------------------------------
def load_state_dict(lib, h, sd, dtype, finalize=True):
    """pcad_set_weight for every floating tensor of sd, cast to the model dtype as modeling.py does, the embedding first;
    then pcad_finalize."""
    from plantcaduceus_b200 import _lib
    td = TD[dtype]
    for name in sorted(sd, key=lambda n: n != EMB_KEY):
        t = sd[name]
        if not t.is_floating_point():
            continue
        src = t.detach().to(td).contiguous()
        shape = (C.c_int64 * src.dim())(*src.shape)
        _lib.check(lib.pcad_set_weight(h, name.encode(), C.c_void_p(src.data_ptr()), shape, src.dim(),
                                       BF16 if td == torch.bfloat16 else F32), h)
    if finalize:
        _lib.check(lib.pcad_finalize(h), h)


def state_dicts(cfg, tied):
    """Two different random state dicts; tied: without lm_head.lm_head.weight (the head is derived from the embedding)."""
    out = []
    for seed in (21, 22):
        sd = random_init_state_dict(cfg, seed=seed)
        if tied:
            sd.pop(HEAD_KEY)
        else:
            sd[HEAD_KEY] = sd[HEAD_KEY].clone() * 0.5 + 0.01     # an explicit head, not a copy of the embedding
        out.append(sd)
    return out


def outputs(model, ids, ascii):
    """pcad_forward's logits and hidden state, then CALLS score_windows calls (graphed from the third)."""
    o = model(input_ids=ids, output_hidden_states=True)
    res = [o.logits.cpu(), o.hidden_states[-1].cpu()]
    res += [score_call(model, ascii, 255, k) for k in range(CALLS)]
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["bf16", "f32"])
@pytest.mark.parametrize("tied", [True, False], ids=["tied-head", "own-head"])
def test_reloaded_handle_equals_a_fresh_one(lib, env, mode, tied):
    """A handle loaded with state dict 1 and used (graphs captured), then reloaded with all of state dict 2 and finalized
    again, computes what a fresh handle loaded with state dict 2 computes: the logits, the hidden state, the graphed score
    path.  In bf16 the fused-norm in_proj_s is rescaled from the new norm weights; without lm_head.lm_head.weight the head
    follows the new embedding."""
    cfg, dtype = config("PlantCaduceus_l20", mode)
    sd1, sd2 = state_dicts(cfg, tied)
    ids = torch.randint(0, 8, (3, 300), generator=torch.Generator().manual_seed(1)).to(DEV)
    ascii = windows(4, 512, seed=2)
    live = engine(env, cfg, sd1, dtype)
    first = outputs(live, ids, ascii)
    load_state_dict(lib, live._handle, sd2, dtype)
    got = outputs(live, ids, ascii)
    fresh = engine(env, cfg, sd2, dtype)
    want = outputs(fresh, ids, ascii)
    names = ["logits", "hidden"] + [f"score call {k + 1}" for k in range(CALLS)]
    for n, g, w, f in zip(names, got, want, first):
        assert not torch.equal(w, f), f"{n}: state dicts 1 and 2 give the same output"
        assert torch.equal(g, w), f"{n} after the reload: {first_difference(g.float(), w.float())}"
    assert replays(lib, live) == 2 * (CALLS - 2)
    live._release()
    fresh._release()


@pytest.mark.gpu
def test_reload_waits_for_queued_work(lib, env):
    """Work queued on a side stream behind a bounded spin (torch.cuda._sleep, about 50 ms) before a reload completes with
    the weights and tables it was queued with: a forward and a graph replay queued, then set_weight of a whole new state
    dict and finalize without synchronising; then a graph replay queued and set_tokenizer with a permuted vocabulary.  The
    spin makes the order deterministic: the queued work is provably still pending when the reload starts."""
    cfg, dtype = config("PlantCaduceus_l20", "bf16")
    sd1, sd2 = state_dicts(cfg, tied=True)
    ids = torch.randint(0, 8, (3, 300), generator=torch.Generator().manual_seed(3)).to(DEV)
    ascii = windows(4, 512, seed=4).to(DEV)
    ref1, ref2 = engine(env, cfg, sd1, dtype, graphs=False), engine(env, cfg, sd2, dtype, graphs=False)
    want1 = (ref1(input_ids=ids).logits, ref1.score_windows_device(ascii, 255))
    want2 = ref2.score_windows_device(ascii, 255)
    live = engine(env, cfg, sd1, dtype)
    side = torch.cuda.Stream()
    logits = torch.full((3, 300, 8), float("nan"), device=DEV)
    out1, out2 = (torch.full((4, 4), float("nan"), device=DEV) for _ in range(2))
    h, p = live._handle, (lambda t: C.c_void_p(t.data_ptr()))
    s = C.c_void_p(side.cuda_stream)

    def score(out):
        assert lib.pcad_score_windows_dev(h, p(ascii), 4, 512, 255, p(out), s) == 0, lib.pcad_last_error(h)

    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        score(out1), score(out1)                  # the graph is captured: the next call replays it
        side.synchronize()
        torch.cuda._sleep(SLEEP_CYCLES)
        assert lib.pcad_forward(h, p(ids), 3, 300, p(logits), None, s) == 0
        score(out1)
    assert not side.query(), "the spin ended before the reload started"
    load_state_dict(lib, h, sd2, dtype)
    side.synchronize()
    assert torch.equal(logits, want1[0]), f"queued forward: {first_difference(logits.cpu(), want1[0].cpu())}"
    assert torch.equal(out1, want1[1]), f"queued graph replay: {first_difference(out1.cpu(), want1[1].cpu())}"
    with torch.cuda.stream(side):
        score(out2), score(out2)
        side.synchronize()
        torch.cuda._sleep(SLEEP_CYCLES)
        score(out2)
    assert not side.query(), "the spin ended before set_tokenizer started"
    live.set_tokenizer(permuted_tokenizer())
    side.synchronize()
    assert torch.equal(out2, want2), f"replay queued before set_tokenizer: {first_difference(out2.cpu(), want2.cpu())}"
    assert replays(lib, live) == 2
    for m in (live, ref1, ref2):
        m._release()
