"""Cost of the geometry gradients: one training step from structures (device graph construction + forward + loss +
backward) with and without `pos` / `lattice` requiring grad, for the fp64 phonon model at B = 64 (H = 256, T = 51, 3
processor layers, 2 transformer layers) and the eDOS model at B = 512 (H = 256, T = 201, bf16x3).

    python scripts/geometry_grad_time.py [--reps 10] [--rounds 5] [--out-dir profiles]

Structures are seeded random triclinic cells (oracle.neighbors_oracle.random_crystal).  CUDA events around `--reps`
consecutive steps after one warm-up step of each kind; the two kinds alternate for `--rounds` rounds and the median
per-step time of each is reported with the GPU's name and power limit, in <out-dir>/geometry_grad_time.json."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from dostransformer_b200 import neighbors, ops  # noqa: E402
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer  # noqa: E402
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon  # noqa: E402
from oracle.neighbors_oracle import random_crystal  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (s.strip() for s in r.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def structures(B, seed, lo, hi, a_lo, a_hi, dev):
    rng = np.random.default_rng(seed)
    sizes = rng.integers(lo, hi + 1, B)
    cells = [random_crystal(rng, int(n), a_lo, a_hi) for n in sizes]
    lattice = torch.tensor(np.stack([c[0] for c in cells]), dtype=torch.float64, device=dev)
    pos = torch.tensor(np.concatenate([c[1] for c in cells]), dtype=torch.float64, device=dev)
    node_ptr = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int64, device=dev)
    return lattice, pos, node_ptr, sizes


def step_ms(step, reps, geo):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        step(geo)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def measure(name, step, reps, rounds, shape):
    step(False)
    step(True)
    off, on = [], []
    for _ in range(rounds):
        off.append(step_ms(step, reps, False))
        on.append(step_ms(step, reps, True))
    off_ms, on_ms = statistics.median(off), statistics.median(on)
    return {"case": name, **shape, "step_ms": round(off_ms, 3), "step_with_geometry_grad_ms": round(on_ms, 3),
            "overhead_ms": round(on_ms - off_ms, 3), "overhead_pct": round(100 * (on_ms - off_ms) / off_ms, 1),
            "off_samples_ms": [round(x, 3) for x in off], "on_samples_ms": [round(x, 3) for x in on]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("geometry_grad_time.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda")
    rows = []

    torch.set_default_dtype(torch.float64)
    torch.manual_seed(0)
    pm = DOSTransformer_phonon(3, 2, 118, 4, 256, 51, dev).to(dev).train()
    lattice, pos, node_ptr, sizes = structures(64, 1, 4, 10, 3.0, 5.5, dev)
    N = int(sizes.sum())
    gen = torch.Generator().manual_seed(2)
    x = torch.zeros(N, 118)
    x[torch.arange(N), torch.randint(0, 118, (N,), generator=gen)] = 1.0 + 200.0 * torch.rand(N, generator=gen)
    x, system = x.to(dev), torch.randint(0, 7, (64,), generator=gen).to(dev)
    ph = torch.rand(64, 51, generator=gen).to(dev)

    def phonon_step(geo):
        lat, p = lattice.clone().requires_grad_(geo), pos.clone().requires_grad_(geo)
        g = neighbors.phonon_graph_batch(lat, p, node_ptr, x, system=system, phdos=ph)
        pm.zero_grad(set_to_none=True)
        dg, _, ds = pm(g)
        ops.dos_loss(dg, ds, g.phdos, mode="phonon").backward()
        return g

    E = phonon_step(False).edge_index.shape[1]
    rows.append(measure("phonon fp64 B=64 H=256 T=51", phonon_step, args.reps, args.rounds, {"atoms": N, "edges": E}))
    del pm

    torch.set_default_dtype(torch.float32)
    torch.manual_seed(0)
    em = DOSTransformer(3, 2, 200, 41, 2, 256, dev, 0.0, n_energies=201, precision="bf16x3").to(dev).train()
    lattice, pos, node_ptr, sizes = structures(512, 3, 4, 36, 3.5, 6.5, dev)
    N = int(sizes.sum())
    gen = torch.Generator().manual_seed(4)
    feats = torch.randn(N, 200, generator=gen).to(dev)
    glob = torch.randn(2 * 512, generator=gen).to(dev)
    esys = torch.randint(0, 7, (512,), generator=gen).to(dev)
    y = torch.rand(512 * 201, generator=gen).to(dev)

    def edos_step(geo):
        lat, p = lattice.clone().requires_grad_(geo), pos.clone().requires_grad_(geo)
        g = neighbors.edos_graph_batch(lat, p, node_ptr, feats, glob=glob, system=esys, y_ft=y)
        em.zero_grad(set_to_none=True)
        dg, _, ds = em(g)
        ops.dos_loss(dg, ds, g.y_ft, mode="edos").backward()
        return g

    E = edos_step(False).edge_index.shape[1]
    rows.append(measure("eDOS bf16x3 B=512 H=256 T=201", edos_step, args.reps, args.rounds, {"atoms": N, "edges": E}))

    line = {"what": "training step from structures (graph construction + forward + loss + backward) without and with "
                    "pos / lattice requiring grad", "reps": args.reps, "rounds": args.rounds, **gpu_info(), "rows": rows}
    text = json.dumps(line)
    print(text, flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "geometry_grad_time.json"), "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
