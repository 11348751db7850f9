"""Training-step time of the eDOS model (H = 256, T = 201, 3 processor layers, 2 transformer layers, bf16x3), eager against
the whole-step CUDA-graph replay (graphed.GraphedStep), for B in {8, 64} crystals and attn_drop in {0, 0.1}.

    python scripts/graph_dropout_time.py [--steps 60] [--warmup 5] [--out FILE]

CUDA events around `--steps` consecutive steps after `--warmup` steps of the same batches (three batches rotated); prints
one JSON line with the GPU's name and power limit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from dostransformer_b200 import ops  # noqa: E402
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer  # noqa: E402
from dostransformer_b200.graphed import GraphedStep  # noqa: E402
from dostransformer_b200.synthetic import make_edos_batch  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (s.strip() for s in r.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_steps(fn, batches, steps, warmup):
    for i in range(warmup):
        fn(batches[i % len(batches)])
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        fn(batches[i % len(batches)])
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("graph_dropout_time.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = DOSTransformer(3, 2, 200, 41, 2, 256, dev, 0.0, n_energies=201, precision="bf16x3").to(dev).train()

    def eager(g):
        model.zero_grad(set_to_none=True)
        dg, _, ds = model(g)
        loss = ops.dos_loss(dg, ds, g.y_ft, mode="edos", beta=1.0)
        loss.backward()
        return loss

    rows = []
    for B in (8, 64):
        gs = [make_edos_batch(B, seed=2000 + i).to(dev) for i in range(3)]
        for p in (0.0, 0.1):
            model.attn_drop = p
            eager_ms = time_steps(eager, gs, args.steps, args.warmup)
            step = GraphedStep(model, "edos")
            graph_ms = time_steps(step, gs, args.steps, args.warmup)
            assert step.replays == args.steps + args.warmup, "a step ran eagerly"
            rows.append({"B": B, "attn_drop": p, "eager_ms": round(eager_ms, 3), "graph_ms": round(graph_ms, 3),
                         "speedup": round(eager_ms / graph_ms, 2), "captures": step.captures,
                         "launches_per_replay": step.launches // max(step.replays, 1)})
    line = {"what": "eDOS train step, eager vs GraphedStep replay", "model": "H=256 T=201 layers=3 t_layers=2 bf16x3",
            "steps": args.steps, "warmup": args.warmup, **gpu_info(), "rows": rows}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
