"""Cost of the mean-pooled hidden states on one GPU, timed with CUDA events (random weights of the named presets), at
PlantCaduceus_l32 with B = 256, L = 512 and PlantCAD2-Large with B = 16, L = 8192:

- (a) pooling every entry: hidden_mean(layers="all") against hidden_at(ids, pos, layers=[n_layer]) (the same full-depth
  forward, one position of the final entry);
- (b) what a user does without it: forward(hidden_layers="all", compute_logits=False) and a torch mean of every entry,
  against hidden_mean(layers="all"), with the peak device memory of each (torch's allocations, which hold the caller
  buffers, beside the engine's workspace);
- (c) the operator alone (pcad_op_hidden_mean on one entry's rows, bf16), with the GB/s achieved on the bytes it must read.

Variants of one case are timed in alternating rounds after a warm-up of each; the median of the rounds is reported.
The card's name and power limit are read in the same run.

    python tools/hidden_mean_bench.py [--rounds 5] [--out results/hidden_mean_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from hidden_layers_bench import card, time_rounds  # noqa: E402

OP_REPS = 20   # operator launches per timed round


def peak_gb(fn):
    """Peak torch device memory (GB) of one call, from a clean slate."""
    import torch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 1e9


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from plantcaduceus_b200 import _lib
    from plantcaduceus_b200.modeling import CaduceusForMaskedLM
    if not torch.cuda.is_available():
        print("hidden_mean_bench needs a CUDA device", file=sys.stderr)
        return 1
    dev = torch.device("cuda:0")
    lib = _lib.load()
    result = {"card": card(), "cases": []}
    print(f"card: {result['card']}")
    g = torch.Generator().manual_seed(0)
    for name, B, L in (("PlantCaduceus_l32", 256, 512), ("PlantCAD2-Large-l48-d1536", 16, 8192)):
        model = CaduceusForMaskedLM.from_random(name, seed=0).to(dev)
        n, d = model.config.n_layer, model.config.d_model
        ids = torch.randint(3, 7, (B, L), generator=g).to(dev, torch.uint8)
        ids64 = ids.long()
        pos = torch.full((B, 1), L // 2 - 1, dtype=torch.int32, device=dev)
        entry_gb = B * L * 2 * d * 2 / 1e9

        def torch_mean():
            hs = model.forward(ids64, hidden_layers="all", compute_logits=False).hidden_states
            return torch.stack([h.float().mean(1) for h in hs])

        # (a) and (b), alternating in one set of rounds
        ms = time_rounds({"hidden_at_final": lambda: model.hidden_at(ids, pos, layers=[n]),
                          "hidden_mean_all": lambda: model.hidden_mean(ids, layers="all"),
                          "taps_all_torch_mean": torch_mean}, args.rounds)
        peak = {"hidden_mean_all": peak_gb(lambda: model.hidden_mean(ids, layers="all")),
                "taps_all_torch_mean": peak_gb(torch_mean)}
        extra = ms["hidden_mean_all"] - ms["hidden_at_final"]
        case = {"preset": name, "B": B, "L": L, "n_layer": n, "entries": n + 1, "entry_gb": entry_gb, "ms": ms,
                "pooling_all_extra_ms": extra, "pooling_all_extra_fraction": extra / ms["hidden_at_final"],
                "pooling_extra_ms_per_entry": extra / (n + 1), "torch_peak_gb": peak,
                "engine_workspace_gb": model.workspace_bytes(B, L) / 1e9}
        print(f"{name} B={B} L={L}: (a) hidden_at final entry {ms['hidden_at_final']:.1f} ms, hidden_mean all {n + 1} entries "
              f"{ms['hidden_mean_all']:.1f} ms (+{100 * extra / ms['hidden_at_final']:.2f} %, {1e3 * extra / (n + 1):.0f} us "
              f"per entry of {entry_gb:.2f} GB); (b) taps + torch mean {ms['taps_all_torch_mean']:.1f} ms, peak torch memory "
              f"{peak['taps_all_torch_mean']:.2f} GB against {peak['hidden_mean_all']:.3f} GB (engine workspace "
              f"{case['engine_workspace_gb']:.2f} GB in both)")
        model._release()
        del model
        torch.cuda.empty_cache()

        # (c) the operator alone on one entry's rows
        rows = torch.randn(2 * B * L, d, generator=torch.Generator(device=dev).manual_seed(1), device=dev).to(torch.bfloat16)
        n_chunks = -(-L // 128)
        scratch = torch.empty(B * n_chunks * 2 * d, dtype=torch.float32, device=dev)
        out = torch.empty(B, 2 * d, dtype=torch.float32, device=dev)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

        def op():
            for _ in range(OP_REPS):
                rc = lib.pcad_op_hidden_mean(C.c_void_p(rows.data_ptr()), None, C.c_void_p(scratch.data_ptr()),
                                             C.c_void_p(out.data_ptr()), B, L, d, _lib.PCAD_BF16, st)
                assert rc == 0
        op_ms = time_rounds({"op": op}, args.rounds)["op"] / OP_REPS
        read_gb = rows.numel() * 2 / 1e9   # the entry's rows (bf16), each read once; the partials are B ceil(L/128) 2d floats
        case["op"] = {"ms": op_ms, "read_gb": read_gb, "gb_per_s": read_gb / (op_ms / 1e3),
                      "partials_gb": scratch.numel() * 4 / 1e9}
        print(f"{name} B={B} L={L}: (c) pcad_op_hidden_mean bf16 {1e3 * op_ms:.1f} us for {read_gb:.3f} GB of rows: "
              f"{case['op']['gb_per_s']:.0f} GB/s")
        result["cases"].append(case)
        del rows, scratch, out
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
