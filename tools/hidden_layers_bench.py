"""Cost of the intermediate hidden states on one GPU, timed with CUDA events (random weights of the named presets):

- early exit: hidden_at(ids, pos, layers=[k]) against hidden_at(ids, pos) (full depth, final norm) for k in {n/4, n/2, n}, at
  PlantCaduceus_l32 with B = 256, L = 512 and PlantCAD2-Small with B = 16, L = 8192 (one position per window);
- tapping every entry: forward(hidden_layers="all") against forward(output_hidden_states=True) (logits and the final
  entry), both with logits, at PlantCaduceus_l32 with B = 256, L = 512.

Variants of one case are timed in alternating rounds after a warm-up of each; the median of the rounds is reported.
The card's name and power limit are read in the same run.

    python tools/hidden_layers_bench.py [--rounds 5] [--out results/hidden_layers_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def time_rounds(variants, rounds, warmup=2):
    """variants: {name: fn}.  Median milliseconds per call of each, rounds alternating between the variants."""
    import torch
    for fn in variants.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    return {k: statistics.median(v) for k, v in ms.items()}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    if not torch.cuda.is_available():
        print("hidden_layers_bench needs a CUDA device", file=sys.stderr)
        return 1
    dev = torch.device("cuda:0")
    result = {"card": card(), "cases": []}
    print(f"card: {result['card']}")
    g = torch.Generator().manual_seed(0)
    for name, B, L in (("PlantCaduceus_l32", 256, 512), ("PlantCAD2-Small-l24-d0768", 16, 8192)):
        model = CaduceusForMaskedLM.from_random(name, seed=0).to(dev)
        n = model.config.n_layer
        ids = torch.randint(3, 7, (B, L), generator=g).to(dev, torch.uint8)
        pos = torch.full((B, 1), L // 2 - 1, dtype=torch.int32, device=dev)
        variants = {"full": lambda: model.hidden_at(ids, pos)}
        for k in (n // 4, n // 2, n):
            variants[f"k={k}"] = (lambda k=k: model.hidden_at(ids, pos, layers=[k]))
        ms = time_rounds(variants, args.rounds)
        case = {"preset": name, "B": B, "L": L, "n_layer": n, "ms": ms,
                "ratio_to_full": {k: v / ms["full"] for k, v in ms.items() if k != "full"}}
        result["cases"].append(case)
        print(f"{name} B={B} L={L}: hidden_at full depth {ms['full']:.1f} ms; " + "; ".join(
            f"layers=[{k[2:]}] {v:.1f} ms ({v / ms['full']:.3f} of full, k/n = {int(k[2:]) / n:.3f})"
            for k, v in ms.items() if k != "full"))
        if name == "PlantCaduceus_l32":
            ids64 = ids.long()
            variants = {"untapped": lambda: model(input_ids=ids64, output_hidden_states=True),
                        "all": lambda: model(input_ids=ids64, hidden_layers="all")}
            ms = time_rounds(variants, args.rounds)
            extra = ms["all"] - ms["untapped"]
            tap_gb = B * L * 2 * model.config.d_model * 2 / 1e9
            case = {"preset": name, "B": B, "L": L, "ms": ms, "extra_ms_per_intermediate_entry": extra / n,
                    "entry_gb": tap_gb}
            result["cases"].append(case)
            print(f"{name} B={B} L={L}: forward with logits and hidden_states[-1] {ms['untapped']:.1f} ms; with all {n + 1} "
                  f"entries {ms['all']:.1f} ms (+{100 * extra / ms['untapped']:.1f} %, {extra / n:.2f} ms per extra entry of "
                  f"{tap_gb:.2f} GB)")
        model._release()
        del model
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
