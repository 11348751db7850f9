"""Cost of attention-map recording (dostransformer_b200.attention_maps): eval forward under no_grad with and without the
recorder, for the eDOS model at B = 512 (H = 256, T = 201, 3 processor layers, 2 transformer layers, bf16x3) and the fp64
phonon model at B = 64 (H = 256, T = 51, 3 processor layers, 2 transformer layers).

    python scripts/attention_maps_time.py [--reps 20] [--rounds 5] [--out profiles/attention_maps_time.json]

CUDA events around `--reps` consecutive forwards of one seeded batch, after one warm-up forward of each kind; the two kinds
alternate for `--rounds` rounds and the median per-forward time of each is reported, with the bytes of maps one recorded
forward returns and the GPU's name and power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import dostransformer_b200 as D  # noqa: E402
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer  # noqa: E402
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon  # noqa: E402
from dostransformer_b200.synthetic import make_edos_batch, make_phonon_batch  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (s.strip() for s in r.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def forward_ms(model, g, reps, record):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            if record:
                with D.attention_maps(model):
                    model(g)
            else:
                model(g)
        b.record()
        torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def measure(name, model, g, reps, rounds):
    with torch.no_grad(), D.attention_maps(model) as rec:
        model(g)                                                   # warm-up of the recording path
    map_bytes = sum(t.numel() * t.element_size() for ts in rec.maps.values() for t in ts)
    forward_ms(model, g, 1, False)
    off, on = [], []
    for _ in range(rounds):
        off.append(forward_ms(model, g, reps, False))
        on.append(forward_ms(model, g, reps, True))
    off_ms, on_ms = statistics.median(off), statistics.median(on)
    return {"case": name, "forward_ms": round(off_ms, 3), "recording_ms": round(on_ms, 3),
            "overhead_ms": round(on_ms - off_ms, 3), "overhead_pct": round(100 * (on_ms - off_ms) / off_ms, 1),
            "map_bytes_per_forward": map_bytes, "off_samples_ms": [round(x, 3) for x in off],
            "on_samples_ms": [round(x, 3) for x in on]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "attention_maps_time.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_maps_time.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda")
    rows = []
    torch.manual_seed(0)
    m = DOSTransformer(3, 2, 200, 41, 2, 256, dev, 0.0, n_energies=201, precision="bf16x3").to(dev).eval()
    rows.append(measure("eDOS B=512 H=256 T=201 bf16x3", m, make_edos_batch(512, seed=2000).to(dev), args.reps, args.rounds))
    del m
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(0)
    m = DOSTransformer_phonon(3, 2, 118, 4, 256, 51, dev).to(dev).eval()
    rows.append(measure("phonon fp64 B=64 H=256 T=51", m, make_phonon_batch(64, seed=2001).to(dev), args.reps, args.rounds))
    line = {"what": "eval forward (no_grad) with and without attention_maps recording", "reps": args.reps,
            "rounds": args.rounds, **gpu_info(), "rows": rows}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
