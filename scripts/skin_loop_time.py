"""Cost per step of a structure loop that watches its neighbour list, two ways, both as CUDA-graph replays
(`graphed.GraphedStep(..., structure=True)`, training step: loss -> parameters, `pos`, `lattice`):

* `held_matches`: a held topology (`neighbors.*_topology(...)`) and `topology.matches()` every 10 steps (a neighbour search
  on the device, one host read, the comparison);
* `skin_stale`: a skin topology (`skin=`: eDOS re-picks its neighbours inside the replay, both run the topology check)
  and one 4-byte read of `topology.stale` every 10 steps.

Cases: eDOS bf16x3 at B = 8 and B = 64 (H = 256, T = 201, 3 processor / 2 transformer layers, skin 1.0 A) and the fp64
phonon model at B = 1 and B = 64 (H = 256, T = 51, skin 0.5 A).

    python scripts/skin_loop_time.py [--reps 50] [--rounds 5] [--out-dir profiles]

Structures are seeded random triclinic cells (oracle.neighbors_oracle.random_crystal); the loop cycles through 10 seeded
geometries about 1e-6 A away from the build, so that the timed loops measure the checks rather than rebuilds (the
rebuilds each variant did are counted in the output).  CUDA events around `--reps` consecutive
steps (the host work of the checks shows up as device idle time inside the window); the two variants alternate for
`--rounds` rounds and the median per-step time of each is reported with the GPU's name and power limit, in
<out-dir>/skin_loop_time.json."""
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
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer  # noqa: E402
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon  # noqa: E402
from dostransformer_b200.graphed import GraphedStep  # noqa: E402
from geometry_grad_time import gpu_info, structures  # noqa: E402

CHECK_EVERY = 10


def loop_ms(run, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for i in range(reps):
        run(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def variants(model, mode, lattice, pos, node_ptr, x, per, skin):
    build = neighbors.phonon_topology if mode == "phonon" else neighbors.edos_topology
    gen = torch.Generator().manual_seed(7)
    geoms = [(lattice + 1e-6 * torch.randn(lattice.shape, generator=gen, dtype=torch.float64).to(lattice.device),
              pos + 1e-6 * torch.randn(pos.shape, generator=gen, dtype=torch.float64).to(pos.device)) for _ in range(10)]
    held, sk = build(lattice, pos, node_ptr), build(lattice, pos, node_ptr, skin=skin)
    step_held, step_skin = GraphedStep(model, mode, structure=True), GraphedStep(model, mode, structure=True)
    counts = {"rebuilds_held": 0, "rebuilds_skin": 0}

    def run_held(i):
        nonlocal held
        lat, p = geoms[i % len(geoms)]
        step_held(held, lat, p, x, **per)
        if i % CHECK_EVERY == CHECK_EVERY - 1 and not held.matches(lat, p):
            held = build(lat, p, node_ptr)
            counts["rebuilds_held"] += 1

    def run_skin(i):
        nonlocal sk
        lat, p = geoms[i % len(geoms)]
        step_skin(sk, lat, p, x, **per)
        if i % CHECK_EVERY == CHECK_EVERY - 1 and int(sk.stale.item()):
            sk = build(lat, p, node_ptr, skin=skin)
            counts["rebuilds_skin"] += 1

    shape = {"entries_held": held.src.numel(), "candidates_skin": (sk.cand_src if mode == "phonon" else sk.src).numel(),
             "skin": skin}
    return {"held_matches": run_held, "skin_stale": run_skin}, shape, counts


def measure(name, var, reps, rounds, shape, counts):
    for f in var.values():               # warm-up: the captures happen here
        for i in range(CHECK_EVERY):
            f(i)
    samples = {k: [] for k in var}
    for _ in range(rounds):
        for k, f in var.items():
            samples[k].append(loop_ms(f, reps))
    med = {k: statistics.median(v) for k, v in samples.items()}
    return {"case": name, **shape, **{f"{k}_ms": round(v, 3) for k, v in med.items()},
            "skin_speedup": round(med["held_matches"] / med["skin_stale"], 2), **counts,
            "samples_ms": {k: [round(x, 3) for x in v] for k, v in samples.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("skin_loop_time.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda")
    rows = []

    torch.set_default_dtype(torch.float32)
    torch.manual_seed(0)
    em = DOSTransformer(3, 2, 200, 41, 2, 256, dev, 0.0, n_energies=201, precision="bf16x3").to(dev).train()
    for B in (8, 64):
        lattice, pos, node_ptr, sizes = structures(B, 3 + B, 4, 36, 3.5, 6.5, dev)
        N = int(sizes.sum())
        gen = torch.Generator().manual_seed(4)
        per = {"glob": torch.randn(2 * B, generator=gen).to(dev),
               "system": torch.randint(0, 7, (B,), generator=gen).to(dev),
               "y_ft": torch.rand(B * 201, generator=gen).to(dev)}
        feats = torch.randn(N, 200, generator=gen).to(dev)
        var, shape, counts = variants(em, "edos", lattice, pos, node_ptr, feats, per, 1.0)
        rows.append(measure(f"eDOS bf16x3 B={B} H=256 T=201", var, args.reps, args.rounds, {"atoms": N, **shape}, counts))
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
        var, shape, counts = variants(pm, "phonon", lattice, pos, node_ptr, x.to(dev), per, 0.5)
        rows.append(measure(f"phonon fp64 B={B} H=256 T=51", var, args.reps, args.rounds, {"atoms": N, **shape}, counts))

    line = {"what": "structure loop as CUDA-graph replays, per step: held topology + matches() every 10 steps vs skin "
                    "topology + one read of topology.stale every 10 steps", "reps": args.reps, "rounds": args.rounds,
            "check_every": CHECK_EVERY, **gpu_info(), "rows": rows}
    text = json.dumps(line)
    print(text, flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "skin_loop_time.json"), "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
