"""Cost of one structure-gradient training step (loss backpropagated to the parameters and to `pos` / `lattice`) three ways:

* `fresh`: `neighbors.*_graph_batch` from the structures every step (neighbour search with its host read, eager model,
  eager reduction to `pos` / `lattice`);
* `topology`: the topology built once (`neighbors.*_topology`), `topology.batch` every step, eager model;
* `replay`: the same step captured once by `graphed.GraphedStep(..., structure=True)` and replayed.

Cases: eDOS bf16x3 and fp32 at B = 8 and B = 64 (H = 256, T = 201, 3 processor / 2 transformer layers) and the fp64 phonon
model at B = 1 and B = 64 (H = 256, T = 51).

    python scripts/structure_step_time.py [--reps 20] [--rounds 5] [--out-dir profiles]

Structures are seeded random triclinic cells (oracle.neighbors_oracle.random_crystal).  CUDA events around `--reps`
consecutive steps after warm-up; the three variants alternate for `--rounds` rounds and the median per-step time of each is
reported with the GPU's name and power limit, in <out-dir>/structure_step_time.json."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402

from dostransformer_b200 import neighbors, ops  # noqa: E402
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer  # noqa: E402
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon  # noqa: E402
from dostransformer_b200.graphed import GraphedStep  # noqa: E402
from geometry_grad_time import gpu_info, structures  # noqa: E402


def step_ms(step, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        step()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def measure(name, variants, reps, rounds, shape):
    for f in variants.values():          # warm-up (the replay variant captures here)
        f()
        f()
    samples = {k: [] for k in variants}
    for _ in range(rounds):
        for k, f in variants.items():
            samples[k].append(step_ms(f, reps))
    med = {k: statistics.median(v) for k, v in samples.items()}
    return {"case": name, **shape, **{f"{k}_ms": round(v, 3) for k, v in med.items()},
            "replay_speedup_vs_fresh": round(med["fresh"] / med["replay"], 2),
            "replay_speedup_vs_topology": round(med["topology"] / med["replay"], 2),
            "samples_ms": {k: [round(x, 3) for x in v] for k, v in samples.items()}}


def variants(model, mode, lattice, pos, node_ptr, x, per):
    graph_batch = neighbors.phonon_graph_batch if mode == "phonon" else neighbors.edos_graph_batch
    topo = (neighbors.phonon_topology if mode == "phonon" else neighbors.edos_topology)(lattice, pos, node_ptr)
    target = "phdos" if mode == "phonon" else "y_ft"

    def eager(build):
        lat, p = lattice.clone().requires_grad_(), pos.clone().requires_grad_()
        g = build(lat, p)
        model.zero_grad(set_to_none=True)
        dg, _, ds = model(g)
        ops.dos_loss(dg, ds, getattr(g, target), mode=mode).backward()
        return p.grad, lat.grad

    replay = GraphedStep(model, mode, structure=True)
    return topo, {"fresh": lambda: eager(lambda lat, p: graph_batch(lat, p, node_ptr, x, **per)),
                  "topology": lambda: eager(lambda lat, p: topo.batch(lat, p, x, **per)),
                  "replay": lambda: replay(topo, lattice, pos, x, **per)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("structure_step_time.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda")
    rows = []

    for prec in ("bf16x3", "fp32"):
        torch.set_default_dtype(torch.float32)
        torch.manual_seed(0)
        em = DOSTransformer(3, 2, 200, 41, 2, 256, dev, 0.0, n_energies=201, precision=prec).to(dev).train()
        for B in (8, 64):
            lattice, pos, node_ptr, sizes = structures(B, 3 + B, 4, 36, 3.5, 6.5, dev)
            N = int(sizes.sum())
            gen = torch.Generator().manual_seed(4)
            per = {"glob": torch.randn(2 * B, generator=gen).to(dev),
                   "system": torch.randint(0, 7, (B,), generator=gen).to(dev),
                   "y_ft": torch.rand(B * 201, generator=gen).to(dev)}
            feats = torch.randn(N, 200, generator=gen).to(dev)
            topo, var = variants(em, "edos", lattice, pos, node_ptr, feats, per)
            rows.append(measure(f"eDOS {prec} B={B} H=256 T=201", var, args.reps, args.rounds,
                                {"atoms": N, "slots": topo.src.numel()}))
        del em

    torch.set_default_dtype(torch.float64)
    torch.manual_seed(0)
    pm = DOSTransformer_phonon(3, 2, 118, 4, 256, 51, dev).to(dev).train()
    for B in (1, 64):
        lattice, pos, node_ptr, sizes = structures(B, 1 + B, 4, 10, 3.0, 5.5, dev)
        N = int(sizes.sum())
        gen = torch.Generator().manual_seed(2)
        x = torch.zeros(N, 118)
        x[torch.arange(N), torch.randint(0, 118, (N,), generator=gen)] = 1.0 + 200.0 * torch.rand(N, generator=gen)
        per = {"system": torch.randint(0, 7, (B,), generator=gen).to(dev), "phdos": torch.rand(B, 51, generator=gen).to(dev)}
        topo, var = variants(pm, "phonon", lattice, pos, node_ptr, x.to(dev), per)
        rows.append(measure(f"phonon fp64 B={B} H=256 T=51", var, args.reps, args.rounds,
                            {"atoms": N, "edges": topo.src.numel()}))

    line = {"what": "structure-gradient training step (loss -> parameters, pos, lattice): fresh neighbour list every step, "
                    "reused topology, CUDA-graph replay of the reused-topology step", "reps": args.reps,
            "rounds": args.rounds, **gpu_info(), "rows": rows}
    text = json.dumps(line)
    print(text, flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "structure_step_time.json"), "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
