#!/usr/bin/env python
"""bench.py -- zero-shot variant-scoring throughput of the B200 engine (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model l32] [--batch 256] [--workload snp]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Default (the driver's line) = BASELINE.json configs[1]: one "step" = one pass of the scoring hot path over one batch of
synthetic 512-bp windows per GPU (PlantCaduceus_l32, bf16, 256 windows, position 255 masked, random-init weights of the
published architecture): tokenise -> mask -> 32-layer RC BiMamba forward -> LM head at the masked position -> 4 logits
(a,c,g,t) per variant.

  value : variants/s, inputs (token ids) already resident in HBM   (pcad_score_masked_at)
  e2e   : variants/s through the reference-facing host call: pinned ASCII windows on the host -> H2D ->
          device tokenise+mask -> forward -> D2H of [B,4] fp32 logits -> sync   (pcad_score_windows_host)
  roofline     : dominant kernel, algorithmic bytes (or FLOPs) / live CUDA-event time
  parity       : the engine's logits on the committed full-depth oracle fixture (tests/golden/fulldepth_<model>.npz) and on the
                 windows the cpu_baseline leg scores live with the fp32 oracle
  cpu_baseline : the CPU oracle (pure-torch restatement of the reference path) timed on this box's host cores on a bounded
                 sample (rank 0, N = 1 only)

Other workloads of BASELINE.json (same JSON contract, `config.workload` names them):
  --workload genome       config 3: variants at uniform positions of a synthetic chromosome resident in HBM; windows are cut
                          on the device (pcad_extract_windows); positions sharded contiguously over the ranks
  --workload mutagenesis  config 4: every position of 512-bp windows masked in turn (3 alt alleles per masked forward)
  --workload long         config 5: L = 8192 windows, final hidden state of every position (embedding extraction);
                          --model cad2-small / cad2-medium / cad2-large run the PlantCAD2 (Mamba-2 / SSD) architecture

Multi-GPU: windows shard over the ranks with no data-path collective; the per-variant scores are gathered ONCE, after the
last step and inside the timed region (the reference-shaped CLI does the same), so ranks are not barriered every step.

--impl reference times the CPU oracle (the reference's own implementation is not installable offline: its arithmetic lives
in mamba-ssm / causal-conv1d / HF-hub remote code; DESIGN.md) with all host threads.

--dump-outputs DIR writes, after the timed steps, what the timed path returned in its last step as DIR/<name>.npy (float32 /
float64; rows of all ranks in rank order, written by rank 0): `logits_acgt` [windows, 4] for the scoring workloads, and for
--workload long a fixed, seeded sample of rows of the final hidden state (`hidden_sample` [n, 2 * d_model] and its row numbers
in each rank's flattened [windows * L] state, `hidden_sample_rows`) bounded by DUMP_SAMPLE_BYTES; with --impl reference, the
CPU oracle's `logits` [windows, L, vocab].  Inputs and weights are seeded, so the same arguments give the same inputs on every
run and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Algorithmic work per 512-bp window (SURVEY.md 8(d), BASELINE.md section 3); bf16 activations.
SCAN_MB_PER_WINDOW = {"l20": 193.3, "l24": 308.3, "l28": 537.7, "l32": 817.9}
GEMM_GFLOP_PER_WINDOW = {"l20": 41.27, "l24": 86.97, "l28": 225.49, "l32": 455.27}
# exponentials in the scan per window (SURVEY.md 8(d): one per state update; l32 2.147 G) -- the pipe that actually binds
SCAN_GEXP_PER_WINDOW = {"l20": 0.503, "l24": 0.805, "l28": 1.409, "l32": 2.147}
MODELS = {"l20": "PlantCaduceus_l20", "l24": "PlantCaduceus_l24", "l28": "PlantCaduceus_l28", "l32": "PlantCaduceus_l32",
          "cad2-small": "PlantCAD2-Small-l24-d0768", "cad2-medium": "PlantCAD2-Medium-l48-d1024",
          "cad2-large": "PlantCAD2-Large-l48-d1536"}
TOKEN_IDX = 255
WINDOW = 512
LONG = 8192
DUMP_SAMPLE_BYTES = 32 << 20      # --dump-outputs: float32 bytes of the hidden-state sample of --workload long, all ranks


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 10; 1 for --impl reference --workload long)")
    ap.add_argument("--warmup", type=int, default=None,
                    help="untimed steps before them (default 3; 0 for --impl reference --workload long)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="l32", choices=sorted(MODELS))
    ap.add_argument("--workload", default="snp", choices=["snp", "genome", "mutagenesis", "long"])
    ap.add_argument("--batch", type=int, default=None, help="windows per GPU per step (default 256; 16 for --workload long)")
    ap.add_argument("--genome-bases", type=int, default=200_000_000, help="--workload genome: length of the synthetic chromosome")
    ap.add_argument("--cpu-sample", type=int, default=2, help="windows in the cpu_baseline sample (0 = skip); ~9 s each on 16 cores")
    ap.add_argument("--no-clocks", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.batch is None:
        args.batch = 16 if args.workload == "long" else 256
    cpu_long = args.impl == "reference" and args.workload == "long"    # one fp32 CPU forward of an 8192-bp window takes minutes
    if args.steps is None:
        args.steps = 1 if cpu_long else 10
    if args.warmup is None:
        args.warmup = 0 if cpu_long else 3
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def write_dump(out_dir: str, arrays: dict):
    """arrays: name -> numpy array (float32 / float64), written as out_dir/<name>.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=float(d["hbm_gbs"]), bf16=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    bf16_burst=float(d["bf16_tflops"]), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16=1400.0, bf16_burst=1590.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
                power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w": statistics.median(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU oracle arm (cpu_baseline and --impl reference)
# ------------------------------------------------------------------------------------------------
def cpu_oracle_rate(model_name: str, n_windows: int, repeats: int = 1, warmup: int = 0, seed: int = 1, length: int = WINDOW,
                    ids=None):
    """Times oracle.caduceus_forward (fp32, all host threads) on `n_windows` windows per step.
    Returns (variants_per_s, ms_per_step, threads, logits of the last step [n, L, 8])."""
    import torch
    from oracle import caduceus_oracle as O
    from plantcaduceus_b200 import preset, random_init_state_dict
    torch.set_num_threads(os.cpu_count() or 1)   # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every core
    cfg = preset(MODELS[model_name])
    sd = random_init_state_dict(cfg, seed=0)
    if ids is None:
        g = torch.Generator().manual_seed(seed)
        ids = torch.randint(3, 7, (n_windows, length), generator=g)
        ids[:, min(TOKEN_IDX, length - 1)] = 1
    logits = None
    with torch.inference_mode():
        for _ in range(warmup):
            O.caduceus_forward(sd, cfg, ids, dtype=torch.float32)
        t0 = time.perf_counter()
        for _ in range(repeats):
            logits, _ = O.caduceus_forward(sd, cfg, ids, dtype=torch.float32)
            O.extract_acgt_probs(logits, min(TOKEN_IDX, length - 1), (3, 4, 5, 6))
        dt = time.perf_counter() - t0
    return len(ids) * repeats / dt, dt / repeats * 1e3, torch.get_num_threads(), logits


def workload_text(args, B, L):
    name = MODELS[args.model]
    if args.workload == "snp":
        return (f"{name} zero-shot SNP scoring: {B} x {L}-bp windows per GPU per step, mask@{TOKEN_IDX}, random-init weights "
                f"(BASELINE.json configs[1])")
    if args.workload == "genome":
        return (f"{name} genome-wide zero-shot SNP scoring: {B} variants per GPU per step at uniform positions of a synthetic "
                f"{args.genome_bases / 1e6:.0f} Mb chromosome resident in HBM, windows cut on the device (BASELINE.json configs[2])")
    if args.workload == "mutagenesis":
        return (f"{name} in-silico saturation mutagenesis: {B} masked positions per GPU per step (every position of {L}-bp windows "
                f"in turn, 3 alt alleles per masked forward) (BASELINE.json configs[3])")
    return (f"{name} long-context embedding extraction: {B} x {L}-bp windows per GPU per step, final hidden state of every "
            f"position (BASELINE.json configs[4])")


def metric_of(args):
    return {"snp": ("variants scored/sec", "variants/s"), "genome": ("variants scored/sec", "variants/s"),
            "mutagenesis": ("variants scored/sec", "variants/s"), "long": ("windows embedded/sec", "windows/s")}[args.workload]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    n = 1  # windows per step: the bounded sample
    L = LONG if args.workload == "long" else WINDOW
    steps, warmup = args.steps, args.warmup
    rate, ms, threads, logits = cpu_oracle_rate(args.model, n, repeats=steps, warmup=warmup, length=L)
    if args.dump_outputs:
        write_dump(args.dump_outputs, {"logits": logits.float().numpy()})
    per_window = 3 if args.workload == "mutagenesis" else 1     # one masked forward serves the position's 3 alt alleles
    rate *= per_window
    metric, unit = metric_of(args)
    line = {
        "impl": "reference", "metric": metric, "value": rate, "unit": unit,
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args, args.batch, L) + f"; CPU oracle, bounded sample of {n} window per step"},
        "cpu_baseline": {"value": rate, "unit": unit, "cores": threads, "kind": "port",
                         "sample": f"{n} window x {steps} steps of {MODELS[args.model]} fp32, L = {L} (oracle/caduceus_oracle.py, "
                                   f"torch {torch.__version__}, {threads} threads of {os.cpu_count()} cpus)"},
        "e2e": {"value": rate, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# parity of the engine on the committed oracle fixture
# ------------------------------------------------------------------------------------------------
def _spearman(a, b):
    import numpy as np
    ra = np.argsort(np.argsort(a)).astype(np.float64)
    rb = np.argsort(np.argsort(b)).astype(np.float64)
    return float(np.corrcoef(ra, rb)[0, 1])


def _llr_pairs(x4):
    import numpy as np
    x = x4.double().numpy()
    return np.array([x[i, a] - x[i, r] for i in range(len(x)) for r in range(4) for a in range(4) if a != r])


def fixture_parity(model, model_name, dev):
    """Engine logits on tests/golden/fulldepth_<model>.npz (oracle fp32 and bf16 logits of 8 windows at full depth, generated by
    tests/golden/make_fulldepth_golden.py from the same seed-0 weights this bench uses)."""
    import numpy as np
    import torch
    p = os.path.join(ROOT, "tests", "golden", f"fulldepth_{model_name}.npz")
    if not os.path.exists(p):
        return None
    z = np.load(p)
    ids = torch.from_numpy(z["ids"])
    want32, want16 = torch.from_numpy(z["logits_f32"]), torch.from_numpy(z["logits_bf16"])
    got = model(input_ids=ids.to(dev)).logits.cpu()
    acgt = [3, 4, 5, 6]
    err = (got - want32).abs()
    lg, lw = _llr_pairs(got[:, TOKEN_IDX, acgt]), _llr_pairs(want32[:, TOKEN_IDX, acgt])
    return {
        "source": f"tests/golden/fulldepth_{model_name}.npz ({len(ids)} windows, full depth, oracle fp32 / bf16)",
        "max_abs_err_scored": err[:, TOKEN_IDX, acgt].max().item(), "max_abs_err_all": err.max().item(),
        "oracle_bf16_self_err": (want16 - want32).abs().max().item(),
        "oracle_bf16_self_err_scored": (want16 - want32).abs()[:, TOKEN_IDX, acgt].max().item(),
        "logit_scale": want32.abs().max().item(), "rel_err_scored": err[:, TOKEN_IDX, acgt].max().item() / want32.abs().max().item(),
        "llr_max_abs_err": float(np.abs(lg - lw).max()), "spearman": _spearman(lg, lw), "n_llr": int(len(lg)),
        "bar": "bf16: 2e-2 absolute at the scored position OR no further from fp32 than the reference algorithm's own bf16 run; "
               "Spearman >= 0.999"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from plantcaduceus_b200 import genome_scan, preset, random_init_state_dict
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = args.workload
    B, K, W = args.batch, args.steps, args.warmup
    L = LONG if wl == "long" else WINDOW

    cfg = preset(MODELS[args.model])
    sd = random_init_state_dict(cfg, seed=0)
    model = CaduceusForMaskedLM.from_pretrained(sd, config=cfg, torch_dtype=torch.bfloat16).to(dev)
    del sd
    tok = model._tokenizer
    acgt_bytes = np.frombuffer(b"ACGT", dtype=np.uint8)

    # synthetic inputs: a different batch per step and per rank (shard = contiguous range of windows / variants)
    rng = np.random.default_rng(1 + rank)
    n_batches = min(K + W, 4)
    results = torch.zeros((K + W, B, 4), dtype=torch.float32, device=dev)     # per-variant scores of every step, gathered once
    host_out = torch.empty((B, 4), dtype=torch.float32).pin_memory()
    h2d = d2h = 0
    if wl in ("snp", "mutagenesis", "long"):
        host_ascii = [torch.from_numpy(rng.choice(acgt_bytes, size=(B, L))).pin_memory() for _ in range(n_batches)]
        lut = torch.from_numpy(tok.lut.astype(np.uint8))
        dev_ids, dev_pos = [], []
        for k, a in enumerate(host_ascii):
            if wl == "mutagenesis":      # rows of one batch = the same window with consecutive positions masked
                a[:] = a[0:1]
                pos_row = (torch.arange(B, dtype=torch.int64) + k * B) % L
            else:
                pos_row = torch.full((B,), TOKEN_IDX, dtype=torch.int64)
            ids = lut[a.long()].to(torch.uint8)
            if wl != "long":
                ids[torch.arange(B), pos_row] = tok.mask_token_id
            dev_ids.append(ids.to(dev))
            dev_pos.append(pos_row.to(torch.int32)[:, None].to(dev))
    if wl == "genome":
        # rank 0 builds the chromosome; the other ranks receive it over NCCL (GPU to GPU), as the CLI's VCF path does
        G = args.genome_bases
        if rank == 0:
            chrom_dev = torch.from_numpy(np.random.default_rng(2).choice(acgt_bytes, size=G)).to(dev)
        else:
            chrom_dev = torch.empty(G, dtype=torch.uint8, device=dev)
        if world > 1:
            dist.broadcast(chrom_dev, src=0)
        host_pos = [torch.from_numpy(rng.integers(0, G, size=B, dtype=np.int64)).pin_memory() for _ in range(n_batches)]
        dev_posn = [p.to(dev) for p in host_pos]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, gather):
        """K steps bracketed by barrier + synchronize on both sides, CUDA events on the launch stream; max over ranks.
        The one collective of the path -- the gather of per-variant scores (SURVEY.md 8e) -- runs once after the last step,
        inside the timed region."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        if world > 1 and gather:
            full = torch.empty((world,) + tuple(results[:steps].shape), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(full, results[:steps].contiguous())
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        timed.per_rank_ms = [ms]
        if world > 1:
            t = torch.tensor([ms], device=dev)
            allt = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allt, t)
            timed.per_rank_ms = [float(x.item()) for x in allt]
            ms = max(timed.per_rank_ms)
        return ms

    if wl == "snp":
        def step_device(i):   # token ids resident in HBM, one scored index (tokenIdx) for every window
            results[i] = model.score_masked(dev_ids[i % n_batches], TOKEN_IDX, check_ids=False)[:, 0]

        def step_host(i):
            model.score_windows_host(host_ascii[i % n_batches], TOKEN_IDX, out=host_out)
            results[i].copy_(host_out, non_blocking=True)
        h2d, d2h = B * L, B * 16
        api = "CaduceusForMaskedLM.score_windows_host -> pcad_score_windows_host"
    elif wl == "mutagenesis":
        host_ids = [t.cpu().pin_memory() for t in dev_ids]
        host_posn = [t.cpu().pin_memory() for t in dev_pos]

        def step_device(i):
            results[i] = model.score_masked(dev_ids[i % n_batches], dev_pos[i % n_batches], check_ids=False)[:, 0]

        def step_host(i):            # host ids + per-row masked positions in, logits out
            k = i % n_batches
            out = model.score_masked(host_ids[k].to(dev, non_blocking=True), host_posn[k].to(dev, non_blocking=True))
            results[i] = out[:, 0]
            host_out.copy_(out[:, 0])
        h2d, d2h = B * L + B * 4, B * 16
        api = "CaduceusForMaskedLM.score_masked (host ids + positions -> device -> host logits)"
    elif wl == "genome":
        def step_device(i):
            genome_scan.score_positions_local(model, chrom_dev, dev_posn[i % n_batches], B, TOKEN_IDX, L, out=results[i])

        def step_host(i):
            pos = host_pos[i % n_batches].to(dev, non_blocking=True)
            genome_scan.score_positions_local(model, chrom_dev, pos, B, TOKEN_IDX, L, out=results[i])
            host_out.copy_(results[i])
        h2d, d2h = B * 8, B * 16
        api = "genome_scan.score_positions_local (host positions -> pcad_extract_windows + pcad_score_windows_dev -> host logits)"
    else:   # long
        hidden_host = torch.empty((B, 2 * cfg.d_model), dtype=torch.bfloat16).pin_memory()
        dev_ids = [t.long() for t in dev_ids]
        host_ids64 = [t.cpu().pin_memory() for t in dev_ids]
        last_hidden = [None]

        def step_device(i):
            last_hidden[0] = model.forward(dev_ids[i % n_batches], output_hidden_states=True, compute_logits=False).hidden_states[-1]

        def step_host(i):
            ids = host_ids64[i % n_batches].to(dev, non_blocking=True)
            out = model.forward(ids, output_hidden_states=True, compute_logits=False)
            hidden_host.copy_(out.hidden_states[-1][:, TOKEN_IDX, :])
        h2d, d2h = B * L * 8, B * 2 * cfg.d_model * 2
        api = "CaduceusForMaskedLM.forward(output_hidden_states=True) from host int64 ids; D2H of the tokenIdx embedding"

    for i in range(W):
        step_device(i)
    sampler = ClockSampler(local)          # every rank samples its own GPU: the slowest rank sets the multi-GPU number
    if not args.no_clocks:
        sampler.start()
    launches0 = model.launch_count()
    ms_total = timed(step_device, K, gather=wl != "long")
    per_rank_ms = list(timed.per_rank_ms)
    if args.dump_outputs:
        # the last timed step's outputs, taken before the e2e and profiling passes below reuse the buffers
        extra = {}
        if wl == "long":
            rows = B * L
            n = min(rows, DUMP_SAMPLE_BYTES // (world * 2 * cfg.d_model * 4))
            sel = np.sort(np.random.default_rng(0).choice(rows, size=n, replace=False))
            dump = {"hidden_sample": last_hidden[0].reshape(rows, -1)[torch.from_numpy(sel).to(dev)].float()}
            extra["hidden_sample_rows"] = sel.astype(np.float64)     # the same rows of every rank's batch
        else:
            dump = {"logits_acgt": results[K - 1].clone()}
        if world > 1:      # rows of every rank, in rank order
            for name, t in dump.items():
                full = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=dev)
                dist.all_gather_into_tensor(full, t.contiguous())
                dump[name] = full.reshape((-1,) + tuple(t.shape[1:]))
        if rank == 0:
            write_dump(args.dump_outputs, {**{name: t.cpu().numpy() for name, t in dump.items()}, **extra})
    launches = model.launch_count() - launches0
    clocks = sampler.stop() if not args.no_clocks else None
    per_rank_mhz = None
    if world > 1 and clocks is not None:
        t = torch.tensor([float(clocks.get("sm_mhz") or 0.0)], device=dev)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank_mhz = [float(x.item()) for x in allt]
    per_item = 3 if wl == "mutagenesis" else 1       # variants per masked forward
    value = world * B * K * per_item / (ms_total * 1e-3)

    for i in range(min(W, 2)):
        step_host(i)
    ms_e2e = timed(step_host, K, gather=wl != "long")
    e2e_value = world * B * K * per_item / (ms_e2e * 1e-3)

    # per-stage breakdown, measured live with CUDA events on the launch stream (pcad_set_profiling)
    prof_steps = min(K, 3)
    model.set_profiling(True)
    for i in range(prof_steps):
        step_device(i)
    torch.cuda.synchronize(dev)
    prof = model.get_profile()
    model.set_profiling(False)
    ws_bytes = model.workspace_bytes(B, L)

    parity = None
    if rank == 0 and world == 1 and wl == "snp":
        parity = fixture_parity(model, args.model, dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    stage_ms = {k: v["ms"] / prof_steps for k, v in prof.items()}
    total_stage_ms = sum(stage_ms.values())
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    tokens = 2.0 * B * L                                  # strand-tokens per step
    metric, unit = metric_of(args)
    line = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {
            "workload": workload_text(args, B, L),
            "windows_per_gpu_per_step": B, "seq_len": L, "sharding": f"windows/{world}" if world > 1 else "single GPU",
            "gather": "one all_gather of every step's scores after the last step, inside the timed region" if world > 1 else None,
            "l2": f"activation working set {ws_bytes / 1e9:.2f} GB per step >> 126 MB L2 (no flush needed)",
        },
        "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / K, "api": api},
        "gpu_launches": int(launches),
    }
    if wl == "long":
        line["bp_per_s"] = value * L
    gemm_ms = stage_ms["in_proj"] + stage_ms["out_proj"] + stage_ms["x_proj"] + stage_ms["dt_proj"]
    if cfg.is_mamba2:
        # PlantCAD2: the projections dominate; report the tensor roofline of the two GEMM stages and the SSD kernel's HBM view
        gemm_flop = 2.0 * cfg.d_model * (cfg.d_in_proj + cfg.d_inner) * tokens * cfg.n_layer
        gemm_tflops = gemm_flop / (gemm_ms * 1e-3) / 1e12
        ssd_ms = prof["scan"]["ms"] / max(1, prof["scan"]["launches"])
        ssd_bytes = 2.0 * (4 * cfg.d_inner + 4 * cfg.d_state) * tokens      # per launch: x + B + C read, y written, both directions, bf16
        line["roofline"] = {
            "kernel": "gemm_bf16_tcgen05_kernel (in_proj + out_proj)", "bound": "tensor", "achieved": gemm_tflops,
            "peak": peaks["bf16"], "unit": "TFLOP/s", "frac": gemm_tflops / peaks["bf16"], "traffic": None,
            "peak_source": peaks["source"], "algorithmic_flop_per_step": gemm_flop}
        line["roofline_ssd"] = {
            "kernel": "ssd_chunk_tc_kernel (chunked SSD on tcgen05, 1 launch per layer, both directions)", "bound": "hbm",
            "achieved": ssd_bytes / (ssd_ms * 1e-3) / 1e9, "peak": peaks["hbm"], "unit": "GB/s",
            "frac": ssd_bytes / (ssd_ms * 1e-3) / 1e9 / peaks["hbm"], "ms_per_launch": ssd_ms,
            "algorithmic_bytes_per_launch": ssd_bytes}
    else:
        scale = (B * L) / float(WINDOW)                   # 512-bp window equivalents per step
        scan_launch_ms = prof["scan"]["ms"] / max(1, prof["scan"]["launches"])
        scan_bytes_per_launch = SCAN_MB_PER_WINDOW[args.model] * 1e6 * scale / cfg.n_layer
        scan_gbs = scan_bytes_per_launch / (scan_launch_ms * 1e-3) / 1e9
        # MUFU view of the same kernel, counting the special-function ops it EXECUTES per (step, channel, direction):
        # 16 ex2 for the decays, 1 ex2 for softplus (its log2(1+e) is an FMA-pipe polynomial) and 1 for the gate (ex2 + rcp
        # per output, shared by the two directions) = 18/16 of the state-update count, against 16 MUFU lanes / clk / SM
        # (measured: tools/ub/fma_pipes.cu) at the observed clock
        mufu_peak = 16.0 * 148 * sm_mhz * 1e6
        mufu_ops = SCAN_GEXP_PER_WINDOW[args.model] * 1e9 * scale / cfg.n_layer * (18.0 / 16.0)
        mufu_rate = mufu_ops / (scan_launch_ms * 1e-3)
        gemm_tflops = GEMM_GFLOP_PER_WINDOW[args.model] * 1e9 * scale / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
        traffic, traffic_note = None, None
        tp = os.path.join(ROOT, "profiles", "scan_traffic.json")
        if os.path.exists(tp) and wl == "snp" and B == 256:
            with open(tp) as f:
                traffic = json.load(f).get(args.model)
            traffic_note = ("STORED figure: dram__bytes_read.sum + dram__bytes_write.sum of one biscan_kernel launch from an "
                            "`ncu --set full` capture of this workload (profiles/scan_traffic.json), not measured in this run")
        line["roofline"] = {
            "kernel": "biscan_kernel (bidirectional selective scan, 1 launch per layer)", "bound": "hbm",
            "achieved": scan_gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": scan_gbs / peaks["hbm"],
            "traffic": traffic, "traffic_note": traffic_note, "peak_source": peaks["source"], "ms_per_launch": scan_launch_ms,
            "algorithmic_bytes_per_launch": scan_bytes_per_launch}
        line["roofline_mufu"] = {
            "kernel": "biscan_kernel", "bound": "mufu (ex2/lg2/rcp special-function pipe: what binds the scan at d_state 16)",
            "achieved": mufu_rate / 1e12, "peak": mufu_peak / 1e12, "unit": "Tops/s", "frac": mufu_rate / mufu_peak,
            "note": "18 executed MUFU ops per 16 state updates (16 decays + softplus ex2 + gate; softplus' log2 is an FMA-pipe polynomial); peak = 16 lanes/clk/SM x 148 SMs x sampled SM clock"}
    line["gemm"] = {"achieved_tflops": gemm_tflops, "peak_tflops": peaks["bf16"],
                    "frac": (gemm_tflops / peaks["bf16"]) if gemm_tflops else None,
                    "note": "minimal algorithmic FLOPs (in/out_proj once per strand) over the summed GEMM-stage time"}
    line["stage_ms_per_step"] = {k: round(v, 3) for k, v in stage_ms.items()}
    line["stage_share"] = {k: round(v / total_stage_ms, 4) for k, v in stage_ms.items()} if total_stage_ms > 0 else None
    if clocks is not None:
        line["clocks"] = clocks
    if world > 1:
        # the timed value is the MAX over ranks: with no data-path collective, what separates N GPUs from N x one GPU is the
        # slowest GPU's power-capped clock, visible here rank by rank
        line["ranks"] = {"ms_per_step": [round(m / K, 2) for m in per_rank_ms], "sm_mhz": per_rank_mhz}
    if world == 1 and args.cpu_sample > 0:
        n = 1 if wl == "long" else args.cpu_sample
        if wl == "snp":
            ids = dev_ids[0][:n].cpu().long()
            rate, ms, threads, want = cpu_oracle_rate(args.model, n, ids=ids)
            got = model(input_ids=ids.to(dev)).logits.cpu()
            err = (got - want).abs()
            if parity is None:
                parity = {}
            parity["live"] = {"windows": n, "max_abs_err_scored": err[:, TOKEN_IDX, 3:7].max().item(),
                              "max_abs_err_all": err.max().item(), "logit_scale": want.abs().max().item(),
                              "source": "this run's cpu_baseline windows: engine bf16 vs oracle fp32"}
        else:
            rate, ms, threads, _ = cpu_oracle_rate(args.model, n, length=L)
        line["cpu_baseline"] = {
            "value": rate * per_item, "unit": unit, "cores": threads, "kind": "port",
            "sample": f"{n} window(s) of the same workload (L = {L}), fp32, oracle/caduceus_oracle.py "
                      f"({threads} torch threads of {os.cpu_count()} cpus), {ms / 1e3:.1f} s"}
    if parity is not None:
        line["parity"] = parity
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict):
    """The one JSON line on the real stdout (everything else -- NCCL banners, library chatter -- goes to stderr)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)          # fd 1 -> stderr for the duration of the run
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
