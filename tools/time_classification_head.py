"""GPU timing of the classification heads (CUDA events).

1. The C2 training step (10 k molecules of ~25 atoms, bf16 BondMessagePassing h = 300 depth 3, mean aggregation, batch norm,
   2-layer FFN of width 300) as ONE CUDA graph, with three heads alternated round by round in rotating order: MSE (1 task),
   BCE (12 tasks) and cross entropy (12 tasks x 3 classes).  Per head: median / min / max ms per step over the rounds.
2. The criterion kernels alone (dmpnn_mse_loss, dmpnn_bce_loss, dmpnn_ce_loss with C = 3, dmpnn_class_probs) at 10 k x 12 and
   10 k x 617 (ToxCast width): median us per launch.  The inputs are written just before timing (as the FFN writes the logits
   in a step), so they are partly L2-resident, as they are in the step.

Prints the card's name and power limit with the numbers and writes everything to <out>/classification_head_timing.json.

    python tools/time_classification_head.py [--rounds 7] [--steps 50] [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402


def device_info() -> dict:
    info = {"torch_device_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip() or q.stderr.strip()
    except Exception as e:  # noqa: BLE001 -- the number is reported without it, and says so
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def events_ms(fn, n: int) -> float:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def make_step(kind: str, bmg, n: int):
    from chemprop_b200.graph import CudaGraphStep
    from chemprop_b200.nn import (BondMessagePassing, EngineBinaryClassificationFFN, EngineMPNN,
                                  EngineMulticlassClassificationFFN, EngineRegressionFFN, MeanAggregation)

    torch.manual_seed(0)                                   # the same encoder weights under every head
    mp = BondMessagePassing(precision="bf16")
    ffn = dict(input_dim=300, hidden_dim=300, n_layers=2)
    gen = torch.Generator().manual_seed(1)
    if kind == "mse_1":
        head, Y = EngineRegressionFFN(n_tasks=1, **ffn), torch.randn(n, 1, generator=gen)
    elif kind == "bce_12":
        head = EngineBinaryClassificationFFN(n_tasks=12, **ffn)
        Y = (torch.rand(n, 12, generator=gen) < 0.3).float()
        Y[torch.rand(n, 12, generator=gen) < 0.2] = float("nan")
    else:
        head = EngineMulticlassClassificationFFN(n_classes=3, n_tasks=12, **ffn)
        Y = torch.randint(0, 3, (n, 12), generator=gen).float()
        Y[torch.rand(n, 12, generator=gen) < 0.2] = float("nan")
    model = EngineMPNN(mp, MeanAggregation(), head, batch_norm=True).cuda().train()
    Y = Y.cuda()
    for p in model.parameters():
        p.grad = torch.zeros_like(p)

    def body(b):
        b._layout = None                                   # the device layout build is part of every step (as in bench.py)
        for p in model.parameters():
            p.grad.zero_()
        loss = model.training_loss(b, Y)
        loss.backward()
        return loss

    step = CudaGraphStep(body)
    return lambda: step(bmg), step


def time_steps(rounds: int, steps: int) -> dict:
    from chemprop_b200.data import BatchMolGraph, make_molecules, tile_packing_order_of

    n = 10_000
    mgs = make_molecules(n, seed=1, mean_atoms=25.0)
    bmg = BatchMolGraph([mgs[i] for i in tile_packing_order_of(mgs)])
    bmg.to("cuda")
    kinds = ["mse_1", "bce_12", "ce_12x3"]
    runs, graphs = {}, {}
    for k in kinds:
        runs[k], graphs[k] = make_step(k, bmg, n)
        for _ in range(5):                                 # capture (2 eager warm-ups + capture) and warm replays
            runs[k]()
    torch.cuda.synchronize()
    ms = {k: [] for k in kinds}
    for r in range(rounds):
        for k in kinds[r % 3:] + kinds[:r % 3]:            # rotating order: no head always runs first
            ms[k].append(events_ms(runs[k], steps))
    out = {"n_mols": n, "atoms": int(bmg.V.shape[0]), "edge_rows": int(bmg.E.shape[0]), "rounds": rounds,
           "steps_per_round": steps}
    for k in kinds:
        assert graphs[k].captures == 1, (k, graphs[k].captures)
        v = ms[k]
        out[k] = {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "per_round_ms": v,
                  "kernels_per_replay": graphs[k].last_launches}
    return out


def time_kernels(reps: int) -> dict:
    from chemprop_b200 import engine

    out = {}
    gen = torch.Generator().manual_seed(2)
    for B, T in ((10_000, 12), (10_000, 617)):
        w, tw = (torch.rand(B, generator=gen) + 0.5).cuda(), (torch.rand(T, generator=gen) + 0.5).cuda()
        loss = torch.empty(1, device="cuda")
        P = torch.randn(B, T, generator=gen).cuda()
        Yr = torch.randn(B, T, generator=gen).cuda()
        Yb = (torch.rand(B, T, generator=gen) < 0.3).float().cuda()
        Z = torch.randn(B, T * 3, generator=gen).cuda()
        Yc = torch.randint(0, 3, (B, T), generator=gen).float().cuda()
        for Y in (Yr, Yb, Yc):
            Y[(torch.rand(B, T, generator=gen) < 0.2).cuda()] = float("nan")
        dP, dZ, Q = torch.empty_like(P), torch.empty_like(Z), torch.empty_like(Z)
        cases = {
            "mse_loss": lambda: engine.mse_loss(P, Yr, w, tw, loss, dP),
            "bce_loss": lambda: engine.bce_loss(P, Yb, w, tw, loss, dP),
            "ce_loss_C3": lambda: engine.ce_loss(Z, Yc, w, tw, loss, dZ, 3),
            "class_probs_C1": lambda: engine.class_probs(P, 1, dP),
            "class_probs_C3": lambda: engine.class_probs(Z, 3, Q),
        }
        res = {}
        for name, fn in cases.items():
            for _ in range(10):
                fn()
            res[name + "_us"] = statistics.median(events_ms(fn, reps) * 1e3 for _ in range(5))
        out[f"{B}x{T}"] = res
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=200, help="launches per kernel timing")
    ap.add_argument("--out", default=None, help="directory for classification_head_timing.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: a timing without the GPU means nothing")
    res = {"device": device_info(), "kernels": time_kernels(args.reps), "step_graph": time_steps(args.rounds, args.steps)}
    print(json.dumps(res["device"]))
    for shape, r in res["kernels"].items():
        print(f"kernels {shape}: " + "  ".join(f"{k}={v:.1f}" for k, v in r.items()))
    s = res["step_graph"]
    for k in ("mse_1", "bce_12", "ce_12x3"):
        print(f"C2 step as one CUDA graph, head {k:8s}: median {s[k]['median_ms']:.3f} ms  (min {s[k]['min_ms']:.3f}, "
              f"max {s[k]['max_ms']:.3f}; {s['rounds']} rounds x {s['steps_per_round']} steps; "
              f"{s[k]['kernels_per_replay']} kernels per replay)")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "classification_head_timing.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
