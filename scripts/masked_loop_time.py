"""Cost per step of a phonon structure loop with a held edge set against one with a masked edge set, both as CUDA-graph
replays (`graphed.GraphedStep(..., structure=True)`, training step: loss -> parameters, `pos`, `lattice`), fp64 phonon
model (3 processor / 2 transformer layers, H = 256, T = 51) at B = 1 and B = 64, skin 0.5 A:

* `skin_held`: `neighbors.phonon_topology(..., skin=0.5)`, the edges within r_max at the build held; every 10 steps one
  read of `topology.stale`, and when it is set a rebuild at the current geometry (a new edge count captures a new graph);
* `masked`: `neighbors.phonon_topology(..., skin=0.5, masked=True)`, every candidate within r_max + skin carried with an
  `edge_mask`; every 10 steps one read of `topology.stale` (set only by the completeness test).

Two trajectories, each cycled in order:

* (a) `slow`: 10 geometries about 1e-6 A from the build.  No bond crosses r_max, so neither variant rebuilds: this is the
  price of running the edge MLPs over the candidates instead of the edges.
* (b) `crossing`: a seeded random walk of the atoms (0.02 A steps, each coordinate kept within 0.08 A of the build, so
  the completeness test passes throughout) whose bonds cross r_max: the held variant rebuilds and recaptures, the masked
  one follows the crossings inside its one graph.

    python scripts/masked_loop_time.py [--reps 50] [--rounds 5] [--out-dir profiles]

Structures are seeded random triclinic cells (geometry_grad_time.structures).  CUDA events around `--reps` consecutive
steps (host work inside the window shows up as device idle time); the variants alternate for `--rounds` rounds and the
median per-step time of each is reported, with rebuilds, captures and the GPU's name and power limit, in
<out-dir>/masked_loop_time.json."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402

from dostransformer_b200 import neighbors  # noqa: E402
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon  # noqa: E402
from dostransformer_b200.graphed import GraphedStep  # noqa: E402
from geometry_grad_time import gpu_info, structures  # noqa: E402
from skin_loop_time import CHECK_EVERY, loop_ms  # noqa: E402

SKIN = 0.5


def slow(lattice, pos):
    gen = torch.Generator().manual_seed(7)
    return [(lattice + 1e-6 * torch.randn(lattice.shape, generator=gen, dtype=torch.float64).to(lattice.device),
             pos + 1e-6 * torch.randn(pos.shape, generator=gen, dtype=torch.float64).to(pos.device)) for _ in range(10)]


def crossing(lattice, pos, n=40, step=0.02, bound=0.08):
    gen = torch.Generator().manual_seed(11)
    walk, out = torch.zeros(pos.shape, dtype=torch.float64), []
    for _ in range(n):
        walk = (walk + step * torch.randn(pos.shape, generator=gen, dtype=torch.float64)).clamp(-bound, bound)
        out.append((lattice, pos + walk.to(pos.device)))
    return out


def variants(model, lattice, pos, node_ptr, x, per, geoms):
    held = neighbors.phonon_topology(lattice, pos, node_ptr, skin=SKIN)
    masked = neighbors.phonon_topology(lattice, pos, node_ptr, skin=SKIN, masked=True)
    step_held, step_masked = GraphedStep(model, "phonon", structure=True), GraphedStep(model, "phonon", structure=True)
    counts = {"rebuilds_skin_held": 0, "rebuilds_masked": 0}

    def run_held(i):
        nonlocal held
        lat, p = geoms[i % len(geoms)]
        step_held(held, lat, p, x, **per)
        if i % CHECK_EVERY == CHECK_EVERY - 1 and int(held.stale.item()):
            held = neighbors.phonon_topology(lat, p, node_ptr, skin=SKIN)
            counts["rebuilds_skin_held"] += 1

    def run_masked(i):
        nonlocal masked
        lat, p = geoms[i % len(geoms)]
        step_masked(masked, lat, p, x, **per)
        if i % CHECK_EVERY == CHECK_EVERY - 1 and int(masked.stale.item()):
            masked = neighbors.phonon_topology(lat, p, node_ptr, skin=SKIN, masked=True)
            counts["rebuilds_masked"] += 1

    shape = {"edges_held": held.src.numel(), "candidates_masked": masked.src.numel()}
    shape["candidates_per_edge"] = round(shape["candidates_masked"] / shape["edges_held"], 3)
    return {"skin_held": run_held, "masked": run_masked}, shape, counts, (step_held, step_masked)


def measure(name, var, reps, rounds, shape, counts, steps):
    for f in var.values():               # warm-up: the first captures happen here
        for i in range(CHECK_EVERY):
            f(i)
    samples = {k: [] for k in var}
    for _ in range(rounds):
        for k, f in var.items():
            samples[k].append(loop_ms(f, reps))
    med = {k: statistics.median(v) for k, v in samples.items()}
    return {"case": name, **shape, **{f"{k}_ms": round(v, 3) for k, v in med.items()},
            "masked_over_held": round(med["masked"] / med["skin_held"], 3), **counts,
            "captures_skin_held": steps[0].captures, "captures_masked": steps[1].captures,
            "samples_ms": {k: [round(x, 3) for x in v] for k, v in samples.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("masked_loop_time.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda")
    rows = []
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
        for traj, geoms in (("slow", slow(lattice, pos)), ("crossing", crossing(lattice, pos))):
            var, shape, counts, steps = variants(pm, lattice, pos, node_ptr, x.to(dev), per, geoms)
            rows.append(measure(f"phonon fp64 B={B} H=256 T=51 {traj}", var, args.reps, args.rounds,
                                {"atoms": N, "trajectory": traj, **shape}, counts, steps))
            print(json.dumps(rows[-1]), flush=True)
    line = {"what": "phonon structure loop as CUDA-graph replays, per step: skin topology with held edges (stale read every "
                    "10 steps, rebuild + recapture when set) vs masked topology (stale read every 10 steps)",
            "reps": args.reps, "rounds": args.rounds, "check_every": CHECK_EVERY, "skin": SKIN, **gpu_info(), "rows": rows}
    text = json.dumps(line)
    print(text, flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "masked_loop_time.json"), "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
