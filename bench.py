#!/usr/bin/env python
"""bench.py -- train-step crystals/sec (fwd+bwd) of the eDOS DOSTransformer on synthetic crystal graphs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl product|reference]
                    [--workload edos|large|phonon|sweep] [--scaling weak|strong] [--batch B_PER_GPU] [--graph auto|on|off]
                    [--dump-outputs DIR]

Headline (default flags; BASELINE.json configs[1]/[2]): DOSTransformer(3 GNN, 2 transformer layers, hidden 256), eDOS
random-split shape (SURVEY.md 8d config 2: ~20 atoms/crystal log-normal, 12 neighbours, 200-d node features, 41-d edge
features, T = 201), 512 crystals per GPU, data-parallel over crystals with weak scaling.  A step = graph prep + forward +
loss + backward (+ gradient all-reduce when N > 1); no optimizer, no data loading, as the metric is defined (SURVEY.md 8d).

One JSON line is printed by rank 0.  `value` is measured with the batches resident in HBM; `e2e` repeats the same steps
from pinned host batches (H2D inside the timed region, loss read back every step).  Next to the headline the line carries
the other BASELINE configurations as extra keys, each with its own `config.workload` (they never replace the headline):

  strong_scaling   config 3 as written: a GLOBAL batch of 512 crystals through the LPT sharder (64 per GPU at N = 8),
                   whole-step CUDA-graph replay (dostransformer_b200/graphed.py)
  large_cell       config 4: 200-400 atoms, 24 neighbours, 64 crystals per GPU
  sweep            config 5: forward-only prediction sweep, 125 k crystal evaluations per GPU (1 M at N = 8) from crystal
                   ids with on-device batch assembly
  small_batch      (N = 1) the reference's default batch 8 (utils.py:31) train step and batch-size-1 evaluation
                   (main_eDOS.py:55-56), eager and graph replay
  phonon           (N = 1) config 1's model on the GPU: DOSTransformer_phonon, fp64, B = 1 and B = 64
  optimizer_in_loop (N = 1) fwd + bwd + fused AdamW every step (weight operand planes refreshed every step)
  cpu_baseline(s)  (N = 1) the reference's own modules (oracle/_ref) on the host cores: all cores and the reference's
                   torch.set_num_threads(2) (main_eDOS.py:12), eDOS B = 64 / B = 8 and phonon fp64 B = 1

`--dump-outputs DIR` writes what the last timed step of the line's train step returned to its caller - the loss and the
gradient of every parameter - as DIR/<name>.npy, so that two builds run with the same arguments (hence the same seeded
model and batches) can be compared output for output.

`--workload/--scaling/--batch` make one of those the line's own metric instead (same JSON contract).  `--impl reference`
times the reference's CPU implementation (kind "reference" when oracle/_ref or /root/reference is present, else the oracle
port) on the host cores.
"""
from __future__ import annotations

import argparse
import gc
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

import torch  # noqa: E402

PREC_DESC = {"fp32": "fp32 FMA pipe", "bf16x3": "tcgen05 bf16x3 error-compensated operand planes (hi*hi + hi*lo + lo*hi), fp32 accumulate: outputs/loss <= 1e-4, gradients <= 2e-3 rel-L2 vs the fp64 reference",
             "bf16": "tcgen05 bf16 operands, fp32 accumulate (tolerance 5e-2 on gradients)"}
METRIC = "train-step crystals/sec (fwd+bwd)"
UNIT = "crystals/s"
HIDDEN, GNN_LAYERS, T_LAYERS, T = 256, 3, 2, 201
MODEL_DESC = f"eDOS DOSTransformer hidden={HIDDEN} L={GNN_LAYERS} t={T_LAYERS}"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            d = json.load(f)
        return dict(hbm=float(d["hbm_gbs"]), tensor=float(d["bf16_tflops"]), tensor_sustained=float(
            d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms.  The process is started BEFORE the warm-up steps: its
    NVML attach takes 0.1-2 s (longer on an 8-GPU box) and stalls CUDA work on the box while it lasts, which must not land
    inside the timed region; only the samples stamped inside the region (`mark()` .. `stop()`) are reported."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.lines, self.proc, self.t0 = gpu_index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_ready(self, timeout: float = 8.0):
        """Blocks until the first sample has arrived (the NVML attach is over) or the timeout passes."""
        t_end = time.time() + timeout
        while self.proc is not None and not self.lines and time.time() < t_end and self.proc.poll() is None:
            time.sleep(0.02)

    def mark(self):
        """The timed region starts now."""
        self.t0 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time()
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = self.t0 if self.t0 is not None else 0.0
        inside = [ln for ts, ln in self.lines if t0 <= ts <= t1 + 0.12]
        if not inside and self.lines:                    # region shorter than one sampling period: the closest sample
            inside = [min(self.lines, key=lambda x: abs(x[0] - t1))[1]]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_batches(rank: int, nb: int, B: int, workload: str = "edos"):
    from dostransformer_b200.synthetic import make_edos_batch, make_large_cell_batch, make_phonon_batch
    if workload == "large":      # BASELINE configs[3]: 200-400 atoms per crystal, 24 neighbours (not the headline line)
        return [make_large_cell_batch(B, seed=4000 + 1000 * rank + i, T=T) for i in range(nb)]
    if workload == "phonon":     # BASELINE configs[0]'s shape (SURVEY 8d config 1)
        return [make_phonon_batch(B, seed=1000 + 1000 * rank + i) for i in range(nb)]
    return [make_edos_batch(B, seed=2000 + 1000 * rank + i, T=T) for i in range(nb)]


def flops_per_crystal_fwd(n_nodes: float, n_edges: float, nmax: float) -> float:
    """SURVEY.md 8d formula (forward FLOPs per crystal), H=256, L=3, t=2."""
    H, L, t = HIDDEN, GNN_LAYERS, T_LAYERS
    Fa, Fe, Fg = 200, 41, 2
    f = 2 * n_nodes * (Fa * H + H * H) + 2 * n_edges * (Fe * H + H * H) + 2 * (Fg * H + H * H)
    f += L * 2 * n_edges * (3 * H * 2 * H + 2 * H * H) + L * 2 * n_nodes * (2 * H * 2 * H + 2 * H * H)
    f += 3 * t * 4 * T * nmax * H + 2 * t * 4 * T * T * H + 5 * t * 2 * T * (8 * H * H)
    f += 2 * T * (2 * H * H) + 2 * T * (2.5 * H * H) + 4 * T * H + 2 * (2 * H * H)
    return f


# ======================================================================================================== output dump
DUMP_BYTES = 60 << 20        # array data of --dump-outputs; with the .npy headers the directory stays under 64 MB


def step_outputs(model, loss) -> dict:
    """What a caller of the train step receives: the loss and the gradient of every parameter that has one."""
    out = {"loss": loss}
    out.update({f"grad.{k}": p.grad for k, p in model.named_parameters() if p.grad is not None})
    return out


def dump_outputs(out_dir: str, arrays: dict, budget: int = DUMP_BYTES) -> None:
    """Writes every tensor as out_dir/<name>.npy, float64 ones as float64 and all others as float32.  When the set holds
    more than `budget` bytes, every array is cut to the same fraction of its elements (flattened), chosen by a generator
    seeded from nothing but the array's length: two runs with the same arguments write the same elements."""
    import numpy as np
    host = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32) for k, v in arrays.items()}
    total = sum(v.numel() * v.element_size() for v in host.values())
    keep = min(1.0, budget / max(total, 1))
    os.makedirs(out_dir, exist_ok=True)
    for name, v in host.items():
        if keep < 1.0:
            n = v.numel()
            idx = torch.randperm(n, generator=torch.Generator().manual_seed(n))[:max(1, int(n * keep))].sort().values
            v = v.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), v.numpy())


# ======================================================================================================== CPU legs
def cpu_leg(workload: str, B: int, steps: int, warmup: int, threads: int, seed: int):
    """The reference's train step (fwd+bwd) on the host cores: oracle/cpu_reference.py (the reference's own modules when
    oracle/_ref or /root/reference is present, else the oracle port).  Returns a cpu_baseline-style dict."""
    from dostransformer_b200.synthetic import make_edos_batch, make_phonon_batch
    from oracle import cpu_reference
    g = make_edos_batch(B, seed=seed) if workload == "edos" else make_phonon_batch(B, seed=seed)
    r = cpu_reference.throughput(workload, g, steps, warmup, threads)
    what = ("eDOS fp32" if workload == "edos" else "phonon fp64 (main_phDOS.py:15-16)")
    src = ("the reference's own modules (embedder_*/, layers/ staged under oracle/_ref, imported unchanged behind "
           "oracle/shims.py)" if r["kind"] == "reference" else "oracle/dost_oracle.py (torch CPU restatement of the reference)")
    return {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "ms_per_step": r["ms_per_step"],
            "sample": f"{what}, {B} crystal(s)/step of the same generator, median of {steps} fwd+bwd steps after {warmup} "
                      f"warm-up ({r['seconds']:.1f} s of CPU work), {src}; host has {r['host_cores']} cores"}


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    wl = "phonon" if args.workload == "phonon" else "edos"
    sample = 1 if wl == "phonon" else args.cpu_sample
    r = cpu_leg(wl, sample, args.steps, args.warmup, threads, seed=2000 if wl == "edos" else 1000)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32" if wl == "edos" else "f64", "data": "synthetic",
        "config": {"workload": (f"{MODEL_DESC} T={T}, random-split shape; bounded sample of {sample} crystals per step (CPU)"
                                if wl == "edos" else "DOSTransformer_phonon hidden=256 L=3 t=2 T=51 fp64, B=1 (BASELINE "
                                "configs[0], main_phDOS.py defaults)"), "sample_crystals": sample},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ======================================================================================================== kernel rooflines
def time_kernel(fn, iters=10):
    fn()
    torch.cuda.synchronize()
    st = torch.cuda.current_stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(iters):
        fn()
    b.record(st)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e-3


def kernel_rooflines(B: int, pk, precision: str, traffic):
    """Times the dominant kernels alone, on the stream they are launched on, at the shapes AND WITH THE EPILOGUE FEATURES
    the step uses.

    `roofline`: the GEMM kernel of the FFN block (65% of the model's FLOPs): the six GEMMs of one FFN layer execution as
    ops._FFNBlock issues them - fc1 forward (bias + ReLU + bf16 hi/lo plane store), fc2 forward (bias + residual, fp32
    store), fc2 input gradient (relu' mask from the saved plane + plane store + fused bias-gradient column sums), fc1
    input gradient (fp32 store), and the two split-K weight gradients - at M = 2 B T rows (the global and the system
    branch run as one batch).  Algorithmic FLOPs = 2 M N K each.
    `roofline_hbm*`: the CSR segmented reduction that replaces scatter_sum, and the LayerNorm that writes operand planes."""
    from dostransformer_b200 import _lib as L
    from dostransformer_b200 import ops
    dev = torch.device("cuda")
    out = {}
    M, Hh, F = 2 * B * T, HIDDEN, 4 * HIDDEN
    kname = {"fp32": "gemm_kernel<float> (fp32 FMA pipe)",
             "bf16x3": "bf::gemm_bf_kernel<3,256,pairs> (TMA-fed tcgen05 cta_group::2, 3 MMAs per product: tensor-pipe work = 3x "
                       "algorithmic)",
             "bf16": "bf::gemm_bf_kernel<1,256,pairs> (TMA-fed tcgen05 cta_group::2)"}

    def six_gemms(prec):
        per_shape, tot_fl, tot_s = [], 0.0, 0.0
        Pp = L.PRECISIONS[prec]
        if prec == "fp32":
            shapes = [("fc1 fwd", M, F, Hh, L.KC, L.KC, 1), ("fc2 fwd", M, Hh, F, L.KC, L.KC, 1), ("fc2 dA", M, F, Hh, L.KC, L.MC, 1),
                      ("fc1 dA", M, Hh, F, L.KC, L.MC, 1), ("fc2 dW", Hh, F, M, L.MC, L.MC, 0), ("fc1 dW", F, Hh, M, L.MC, L.MC, 0)]
            fns = []
            for name, m, n, k, am, bm, split in shapes:
                a = torch.randn((m, k) if am == L.KC else (k, m), device=dev)
                b = torch.randn((n, k) if bm == L.KC else (k, n), device=dev)
                o = torch.empty(m, n, device=dev)
                sk = ops._pick_split(m, n, k, 4) if split == 0 else 1
                fns.append((name, m, n, k, (lambda a=a, b=b, o=o, m=m, n=n, k=k, am=am, bm=bm, sk=sk: ops.gemm_raw(
                    M=m, N=n, K=k, a=[(a, None)], a_mode=am, b=b, b_mode=bm, out=o, split_k=sk, prec=Pp))))
        else:
            with ops.precision(prec):
                y = torch.randn(M, Hh, device=dev)
                h0p = ops.split_planes(torch.randn(M, Hh, device=dev))
                h1p = ops.empty_planes(M, F, dev, ops._with_lo())
                w1p, w2p = ops.split_planes(torch.randn(F, Hh, device=dev) * 0.05), ops.split_planes(torch.randn(Hh, F, device=dev) * 0.05)
                b1, b2 = torch.randn(F, device=dev), torch.randn(Hh, device=dev)
                dop = ops.split_planes(torch.randn(M, Hh, device=dev))
                dv1p = ops.empty_planes(M, F, dev, ops._with_lo())
                gate = torch.zeros(F // 32, M, dtype=torch.int32, device=dev) if ops.gate_bits_ok(M, F) else None
                o_mh, db1 = torch.empty(M, Hh, device=dev), torch.empty(F, device=dev)
                dw2, dw1 = torch.empty(Hh, F, device=dev), torch.empty(F, Hh, device=dev)
                sk2, sk1 = ops._split_for(Hh, F, M), ops._split_for(F, Hh, M)

            def wrap(fn):
                def run():
                    with ops.precision(prec):
                        fn()
                return run
            fns = [
                ("fc1 fwd (bias+ReLU -> hi/lo planes + gate bits)", M, F, Hh, wrap(lambda: ops.gemm_planes(
                    M=M, N=F, K=Hh, a=[h0p], a_mode=L.KC, b=w1p, b_mode=L.KC, bias=b1, act=L.ACT_RELU, out_planes=h1p, out_gate=gate))),
                ("fc2 fwd (bias+residual -> fp32)", M, Hh, F, wrap(lambda: ops.gemm_planes(
                    M=M, N=Hh, K=F, a=[h1p], a_mode=L.KC, b=w2p, b_mode=L.KC, bias=b2, residual=y, out=o_mh))),
                ("fc2 dA (relu' gate bits, planes out, bias-grad column sums)", M, F, Hh, wrap(lambda: ops.gemm_planes(
                    M=M, N=F, K=Hh, a=[dop], a_mode=L.KC, b=w2p, b_mode=L.MC, dact=h1p if gate is None else None, dact_gate=gate,
                    dact_slope=0.0, out_planes=dv1p, colsum_out=db1))),
                ("fc1 dA (fp32)", M, Hh, F, wrap(lambda: ops.gemm_planes(
                    M=M, N=Hh, K=F, a=[dv1p], a_mode=L.KC, b=w1p, b_mode=L.MC, out=o_mh))),
                ("fc2 dW (split-K)", Hh, F, M, wrap(lambda: ops.gemm_planes(
                    M=Hh, N=F, K=M, a=[dop], a_mode=L.MC, b=h1p, b_mode=L.MC, out=dw2, split_k=sk2))),
                ("fc1 dW (split-K)", F, Hh, M, wrap(lambda: ops.gemm_planes(
                    M=F, N=Hh, K=M, a=[dv1p], a_mode=L.MC, b=h0p, b_mode=L.MC, out=dw1, split_k=sk1))),
            ]
        for name, m, n, k, fn in fns:
            sec = time_kernel(fn)
            fl = 2.0 * m * n * k
            per_shape.append({"gemm": name, "M": m, "N": n, "K": k, "ms": sec * 1e3, "tflops": fl / sec / 1e12})
            tot_fl += fl
            tot_s += sec
        tf = tot_fl / tot_s / 1e12
        mult = 3 if prec == "bf16x3" else 1
        return {"kernel": kname[prec] + ", the six GEMMs of one FFN layer execution with the step's epilogues", "bound": "tensor",
                "achieved": tf, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": tf / pk["tensor"], "traffic": traffic,
                "peak_source": pk["source"] + ", bf16 burst", "algorithmic_flops_per_launch": tot_fl / len(fns),
                "launch_ms": tot_s / len(fns) * 1e3, "tensor_pipe_tflops": tf * mult, "tensor_pipe_frac": tf * mult / pk["tensor"],
                "note": ("launch_ms includes the split-K reduction / column-sum kernels that belong to the GEMM call; bf16x3 "
                         "issues 3 MMAs per algorithmic product, so frac <= 1/3 by construction and tensor_pipe_frac is the "
                         "utilisation of the tensor pipe" if prec == "bf16x3" else ""),
                "per_shape": per_shape}

    out["roofline"] = six_gemms(precision)
    if precision == "bf16x3":
        out["roofline_bf16_mode"] = six_gemms("bf16")     # the same kernel reading only the hi planes (1 MMA per product)
    # scatter_sum as a CSR segmented reduction: [E,256] -> [N,256]
    from dostransformer_b200.synthetic import make_edos_batch
    g = make_edos_batch(B, seed=2000, T=T)
    gr = ops.build_graph(g.edge_index.to(dev), g.batch.to(dev), g.system.to(dev))
    dst = torch.empty(gr.N, HIDDEN, device=dev)
    big = [torch.randn(gr.E, HIDDEN, device=dev) for _ in range(max(1, int(300e6 // (gr.E * HIDDEN * 4))))]
    it = {"i": 0}

    def seg():
        s = big[it["i"] % len(big)]
        it["i"] += 1
        ops.segment_reduce_raw(s, gr.by_dst.rowptr, gr.by_dst.perm, gr.N, out=dst)

    sec = time_kernel(seg, iters=max(10, len(big) * 3))
    nbytes = 4.0 * HIDDEN * (gr.E + gr.N) + 4.0 * gr.E + 4.0 * (gr.N + 1)
    gbs = nbytes / sec / 1e9
    out["roofline_hbm"] = {"kernel": "segment_reduce_vec_kernel<float,2> (scatter_sum [E,256]->[N,256])", "bound": "hbm",
                           "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                           "traffic": ncu_capture("r2_ncu_streaming_segment_reduce") if B == 512 else None,
                           "algorithmic_bytes_per_launch": nbytes, "launch_ms": sec * 1e3, "E": gr.E, "N": gr.N,
                           "note": "inputs rotated over >300 MB so they do not sit in L2"}
    del big
    # LayerNorm of the [2*B*T, 256] token stream writing bf16 hi/lo operand planes: reads 4 B, writes 4 B per element
    xs = [torch.randn(M, HIDDEN, device=dev) for _ in range(3)]
    gam, bet = torch.ones(HIDDEN, device=dev), torch.zeros(HIDDEN, device=dev)
    it2 = {"i": 0}

    def ln():
        it2["i"] += 1
        with ops.precision("bf16x3"):
            ops.ln_fwd_planes(xs[it2["i"] % 3], gam, bet)

    sec = time_kernel(ln, iters=12)
    nbytes = 8.0 * M * HIDDEN + 8.0 * M
    out["roofline_hbm_ln"] = {"kernel": "rbf::ln_fwd_kernel<2> (LayerNorm [2*B*T,256] -> bf16 hi/lo planes)", "bound": "hbm",
                              "achieved": nbytes / sec / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                              "frac": nbytes / sec / 1e9 / pk["hbm"], "traffic": None, "algorithmic_bytes_per_launch": nbytes,
                              "launch_ms": sec * 1e3}
    # fused attention forward (csrc/attn_fused.cu): the T x T energy self attention of the 2 B sequences, and the ragged
    # energy -> atom cross attention of the same batch.  Algorithmic FLOPs: 2 contractions x 2 Lq Lk H per sequence (the
    # cross attention: Lk = the crystal's own atoms + 1 phantom column).
    with ops.precision(precision):
        fused_ok = precision != "fp32" and ops.fused_attention_ok(HIDDEN, T, 0.0)
    if fused_ok:
        S2 = 2 * B
        del xs
        with ops.precision(precision):
            qs = [torch.randn(S2, T, HIDDEN, device=dev) for _ in range(2)]
            ks = [torch.randn(S2, T, HIDDEN, device=dev) for _ in range(2)]
            for t in qs + ks:
                t._dost_planes = ops.split_planes(t.view(S2 * T, HIDDEN))
            it3 = {"i": 0}

            def sa():
                it3["i"] += 1
                with ops.precision(precision), torch.no_grad():
                    ops.self_attention(qs[it3["i"] % 2], ks[it3["i"] % 2], qs[(it3["i"] + 1) % 2])

            sec = time_kernel(sa, iters=10)
            fl = 4.0 * S2 * T * T * HIDDEN
            mult = 3 if precision == "bf16x3" else 1
            out["roofline_attention"] = {
                "kernel": "fa::attn_fwd_kernel (QK^T -> fp32 softmax in TMEM -> PK, one kernel), energy self attention [2B, 201, 256]",
                "bound": "tensor", "achieved": fl / sec / 1e12, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": fl / sec / 1e12 / pk["tensor"],
                "traffic": ncu_capture("r2_ncu_attn_self") if (B == 512 and precision == "bf16x3") else None,
                "traffic_note": "ncu --set full capture (profiles/r2_ncu_attn_self.summary.txt) of this kernel inside a training step, "
                                "where it also writes the bf16 probability planes the backward reads (about 170 MB more than the "
                                "forward-only launch timed here)",
                "algorithmic_flops_per_launch": fl, "launch_ms": sec * 1e3,
                "tensor_pipe_frac": fl * mult / sec / 1e12 / pk["tensor"],
                "hbm_gbytes_per_s": 3.0 * S2 * T * HIDDEN * 4 / sec / 1e9,
                "note": "201 queries / keys occupy 256-wide tiles (62 % of the issued MMA work is algorithmic); q, residual and out "
                        "are the only HBM traffic (no score matrix); the three-kernel formulation it replaces is timed next to it",
            }
            os.environ["DOST_NO_ATTN_FUSED"] = "1"
            L.reload_switches()
            try:
                out["roofline_attention"]["unfused_launch_ms"] = time_kernel(sa, iters=10) * 1e3
            finally:
                os.environ.pop("DOST_NO_ATTN_FUSED", None)
                L.reload_switches()
            kv, ph = torch.randn(gr.N, HIDDEN, device=dev), torch.randn(HIDDEN, device=dev)
            gr2 = ops.build_graph(g.edge_index.to(dev), g.batch.to(dev), g.system.to(dev), nmax_hint=g.max_num_nodes)

            def xa():
                it3["i"] += 1
                with ops.precision(precision), torch.no_grad():
                    ops.cross_attention(qs[it3["i"] % 2], kv, ph, qs[(it3["i"] + 1) % 2], gr2, S2)

            sec = time_kernel(xa, iters=10)
            nk = (torch.bincount(g.batch) + 1).double().sum().item() * 2          # keys (atoms + phantom column) over the 2 B sequences
            out["roofline_attention"]["cross_attention"] = {
                "launch_ms": sec * 1e3, "tflops": 4.0 * T * nk * HIDDEN / sec / 1e12, "mean_keys_per_sequence": nk / S2,
                "note": "ragged keys (mean 25 per crystal) against 128-query tiles: bound by the q / residual / out streams, "
                        + f"{3.0 * S2 * T * HIDDEN * 4 / sec / 1e9:.0f} GB/s of {pk['hbm']:.0f}; includes the key-plane build kernel"}
    return out


def ncu_capture(name: str):
    """dram bytes (read + write) per launch of one named `ncu --set full` capture recorded in profiles/ncu_gemm_traffic.json
    (the summaries themselves are profiles/<name>.summary.txt); None when the capture is not there."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_gemm_traffic.json")) as f:
            return json.load(f).get("captures", {}).get(name)
    except Exception:
        return None


def ncu_traffic(precision: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant GEMM, from the newest committed `ncu --set full`
    summary under profiles/ (written by scripts/ncu_gemm_traffic.sh on this round's build); None when there is none."""
    path = os.path.join(ROOT, "profiles", "ncu_gemm_traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(precision)
    except Exception:
        return None


# ======================================================================================================== GPU legs
def _to_device(g, dev):
    from dostransformer_b200.synthetic import CrystalBatch
    return CrystalBatch(**{k: (getattr(g, k).to(dev, non_blocking=True) if torch.is_tensor(getattr(g, k)) else
                               getattr(g, k)) for k in g.keys()})


class Runner:
    """One configuration's step function: whole-step CUDA-graph replay (graphed.GraphedStep + flat all-reduce) or the eager
    step (`model(batch)` + ops.dos_loss + backward + bucketed GradReducer).  A capture that fails (first call of a new
    batch signature) falls back to the eager step for the rest of the run and says so in `mode`."""

    def __init__(self, model, mode, world, weight, use_graph, reducer=None):
        from dostransformer_b200 import dp, ops
        from dostransformer_b200.graphed import GraphedStep
        self.model, self.mode, self.world, self.weight, self.ops, self.dp = model, mode, world, weight, ops, dp
        self.reducer = reducer
        self.own_reducer = False
        self.graph = GraphedStep(model, mode, loss_weight=weight, world=world) if use_graph else None
        self.tkey = "y_ft" if mode == "edos" else "phdos"
        self.fallback = None
        self.last = None          # the loss of the last step (a graph replay overwrites it with the next one)

    def describe(self):
        if self.graph is not None:
            return "whole-step CUDA-graph replay (graphed.GraphedStep)" + (", flat NCCL all-reduce after the replay" if self.world > 1 else "")
        base = "eager step" + (", bucketed all-reduce overlapped with backward" if self.world > 1 else "")
        return base + (f" (graph capture failed: {self.fallback})" if self.fallback else "")

    def __call__(self, g):
        self.last = self._step(g)
        return self.last

    def _step(self, g):
        if self.graph is not None:
            try:
                return self.graph(g)
            except Exception as ex:  # noqa: BLE001  (a failed capture must not take the measurement down)
                if self.graph.replays > 0:
                    raise
                self.fallback = repr(ex)[:200]
                self.graph = None
                torch.cuda.synchronize()
        if self.reducer is None and self.world > 1:
            self.reducer = self.dp.GradReducer(self.dp.live_named_parameters(self.model))
            self.own_reducer = True
        model = self.model
        model.zero_grad(set_to_none=True)
        dg, _, ds = model(g)
        loss = self.ops.dos_loss(dg, ds, getattr(g, self.tkey), mode=self.mode, beta=1.0)
        if self.weight != 1.0:
            loss = loss * self.weight
        loss.backward()
        if self.reducer is not None:
            self.reducer.finish()
        return loss.detach()

    def close(self):
        if self.reducer is not None and self.own_reducer:
            self.reducer.remove()
        self.reducer = None
        self.graph = None

    def launches(self, L, l0):
        return (self.graph.launches if self.graph is not None else 0) + (L.launch_count() - l0)


def timed_steps(step, batches, steps, warmup, barrier, st, ncu_window=False):
    """W warm-up steps, then K steps bracketed by barrier + synchronize, CUDA events on the launching stream.  Returns
    (seconds, per-step device ms)."""
    for i in range(warmup):
        step(batches[i % len(batches)])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    e0.record(st)
    for i in range(steps):
        if ncu_window and i == 0:       # `ncu --profile-from-start off python bench.py --ncu-window`: the launch list of
            torch.cuda.cudart().cudaProfilerStart()      # exactly one timed step of this very command
        step(batches[i % len(batches)])
        if os.environ.get("DOST_BENCH_SYNC_EACH"):       # (debugging aid)
            torch.cuda.synchronize()
        if ncu_window and i == 0:
            torch.cuda.synchronize()
            torch.cuda.cudart().cudaProfilerStop()
        marks[i].record(st)
    e1.record(st)
    barrier()
    each = [round(a.elapsed_time(b), 3) for a, b in zip([e0] + marks[:-1], marks)]
    return e0.elapsed_time(e1) * 1e-3, each


def max_over_ranks(x: float, world: int, dev):
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def e2e_steps(step, host, dev, steps, warmup, barrier):
    """The same steps from pinned host batches: H2D of the whole batch and a D2H read of the loss inside the timed region."""
    # Input pipeline of a training loop with a pinned-memory loader: the H2D copy of step i + 1 is issued on a copy stream
    # before step i is launched and overlaps its compute (double buffering); every step's copy and its loss read-back are
    # inside the timed region, the first copy included.
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream(dev)

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            b = _to_device(host[i % len(host)], dev)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return b, ev

    # every distinct batch shape once through the same path: graph capture, and the copy stream's allocator pool
    nwarm = max(len(host), min(2, warmup)) + 1
    nxt = prefetch(0)
    for i in range(nwarm):
        cur, ev = nxt
        main.wait_event(ev)
        nxt = prefetch(i + 1)
        step(cur).item()
    del nxt, cur
    # Long-lived objects (model, batches, autograd metadata) leave the cyclic GC's working set: without this a
    # generation-2 collection lands inside the synchronous loop every few steps and stalls one step by 10-70 ms
    # (the device-resident loop hides such pauses behind the launch queue).
    gc.collect()
    gc.freeze()
    gc.disable()          # (and none of the younger generations either: a step allocates ~10^4 short-lived Python objects)
    try:
        barrier()
        per_step = []
        t0 = time.perf_counter()
        nxt = prefetch(0)
        for i in range(steps):
            ts = time.perf_counter()
            cur, ev = nxt
            main.wait_event(ev)
            if i + 1 < steps:
                nxt = prefetch(i + 1)                             # H2D of the NEXT batch from pinned memory, during this step
            loss = step(cur)
            loss.item()                                           # D2H of the step's result (also keeps `cur` alive until done)
            per_step.append((time.perf_counter() - ts) * 1e3)
        barrier()
        return time.perf_counter() - t0, per_step
    finally:
        gc.enable()


def strong_scaling_leg(model, rank, world, dev, steps, warmup, barrier, st, global_batch, use_graph, L):
    """BASELINE config 3 as written: a GLOBAL batch through the LPT sharder, loss weight B_local / B_global, the sharder's
    global padding length; whole-step graph replay + flat all-reduce (or the eager step + bucketed reducer)."""
    from dostransformer_b200 import dp
    from dostransformer_b200.synthetic import make_edos_batch
    NB = 3
    parts, weights, nmaxes = [], None, []
    for i in range(NB):
        g = make_edos_batch(global_batch, seed=2000 + i, T=T)         # the same global batches on every rank
        if world > 1:
            ps, nmax, ws, _ = dp.shard_batch(g, world, T=T, hidden=HIDDEN)
            mine = ps[rank]
            mine.max_num_nodes = int(torch.bincount(mine.batch).max())
            weights = ws
        else:
            mine, nmax, weights = g, g.max_num_nodes, [1.0]
        parts.append(mine.pin_memory())
        nmaxes.append(nmax)
    old_nmax = model.max_num_nodes
    model.max_num_nodes = max(nmaxes)        # the sharder's global padding length (one value for the 3 rotating batches)
    run = Runner(model, "edos", world, weights[rank] if world > 1 else 1.0, use_graph)
    resident = [p.clone().to(dev) for p in parts]
    l0 = L.launch_count()
    sec, each = timed_steps(run, resident, steps, max(warmup, NB), barrier, st)
    launches = run.launches(L, l0)
    sec = max_over_ranks(sec, world, dev)
    e2e_sec, _ = e2e_steps(run, parts, dev, steps, warmup, barrier)
    e2e_sec = max_over_ranks(e2e_sec, world, dev)
    mode_desc = run.describe()
    run.close()
    model.max_num_nodes = old_nmax
    b_local = int(parts[0].system.numel())
    return {"metric": METRIC, "value": global_batch * steps / sec, "unit": UNIT, "scaling": "strong", "n_gpus": world,
            "ms_per_step": sec / steps * 1e3, "ms_each_step_device": each, "steps": steps,
            "e2e": {"value": global_batch * steps / e2e_sec, "unit": UNIT, "ms_per_step": e2e_sec / steps * 1e3,
                    "h2d_bytes_per_step": int(parts[0].nbytes()), "d2h_bytes_per_step": 4},
            "gpu_launches_per_step": launches / max(1, steps + max(warmup, NB)),
            "config": {"workload": f"{MODEL_DESC} T={T}, training step, GLOBAL batch {global_batch} crystals with ragged atom counts, "
                                   f"data-parallel {world}xB200 through the LPT sharder (BASELINE configs[2])",
                       "global_batch": global_batch, "crystals_per_gpu": b_local, "parallelism": f"dp{world}",
                       "mode": mode_desc, "nmax": max(nmaxes)}}


def weak_leg(model, workload, mode, B, rank, world, dev, steps, warmup, barrier, st, use_graph, L, label):
    """A per-GPU-batch configuration (large cell, small batch, phonon): per-rank batches, weak scaling."""
    from dostransformer_b200 import dp
    import torch.distributed as dist
    NB = 3
    host = [b.pin_memory() for b in make_batches(rank, NB, B, workload)]
    nmax = max(int(torch.bincount(b.batch).max()) for b in host)
    if world > 1:
        t = torch.tensor([nmax], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        nmax = int(t.item())
    for b in host:
        if not hasattr(b, "max_num_nodes") or "max_num_nodes" not in b:
            b["max_num_nodes"] = int(torch.bincount(b.batch).max())
    old_nmax = model.max_num_nodes
    model.max_num_nodes = nmax
    run = Runner(model, mode, world, 1.0 / world, use_graph)
    resident = [b.clone().to(dev) for b in host]
    l0 = L.launch_count()
    sec, each = timed_steps(run, resident, steps, max(warmup, NB), barrier, st)
    launches = run.launches(L, l0)
    sec = max_over_ranks(sec, world, dev)
    mode_desc = run.describe()
    run.close()
    model.max_num_nodes = old_nmax
    n_nodes = sum(b.batch.numel() for b in host) / NB
    n_edges = sum(b.edge_index.shape[1] for b in host) / NB
    return {"metric": METRIC, "value": world * B * steps / sec, "unit": UNIT, "scaling": "weak", "n_gpus": world,
            "ms_per_step": sec / steps * 1e3, "ms_each_step_device": each, "steps": steps,
            "gpu_launches_per_step": launches / max(1, steps + max(warmup, NB)),
            "config": {"workload": label, "crystals_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                       "mean_nodes_per_batch": n_nodes, "mean_edges_per_batch": n_edges, "nmax": nmax,
                       "mode": mode_desc}}


def sweep_leg(model, rank, world, dev, n_eval, store_size, batch_size, barrier):
    """BASELINE config 5: forward-only DOS prediction sweep, sharded over the ranks (no collective).  Every rank holds a
    store of `store_size` distinct synthetic crystals packed in HBM and evaluates `n_eval` crystal ids (counter-hashed into
    the store, sorted by atom count into batches of `batch_size` assembled ON THE DEVICE from the ids), per-crystal
    evaluation (no phantom keys: the reference's batch_size-1 loaders), predictions kept on the device."""
    import numpy as np
    from dostransformer_b200.collate import PackedCrystals
    from dostransformer_b200.synthetic import make_edos_batch
    t_build = time.perf_counter()
    chunks = [make_edos_batch(min(2048, store_size - i), seed=7000 + 97 * rank + i, T=T) for i in range(0, store_size, 2048)]
    stores = [PackedCrystals.from_batch(c, device=dev) for c in chunks]
    t_build = time.perf_counter() - t_build
    # crystal id -> (store chunk, slot): a counter-based hash of the GLOBAL crystal id (splitmix64 finaliser)
    gid = np.arange(rank * n_eval, (rank + 1) * n_eval, dtype=np.uint64)
    z = gid * np.uint64(0x9E3779B97F4A7C15) + np.uint64(0xBF58476D1CE4E5B9)
    z ^= z >> np.uint64(31)
    slot = (z % np.uint64(store_size)).astype(np.int64)
    was_training, was_pc, was_nmax = model.training, model.per_crystal_eval, model.max_num_nodes
    model.eval()
    model.per_crystal_eval = True
    model.max_num_nodes = None
    plans = []
    for ci, stc in enumerate(stores):
        sel = slot[(slot // 2048) == ci] - ci * 2048
        order = np.argsort(stc.node_count[sel], kind="stable")
        sel = sel[order]
        plans += [(stc, torch.from_numpy(sel[i:i + batch_size].copy())) for i in range(0, len(sel), batch_size)]
    outs = []
    with torch.no_grad():
        for stc, ids in plans[:2]:
            model(stc.collate(ids))
        barrier()
        t0 = time.perf_counter()
        done = 0
        for stc, ids in plans:
            g = stc.collate(ids)
            dg, _, ds = model(g)
            outs.append(ds.clamp_min(0))          # utils.py:76
            if len(outs) > 8:
                outs.pop(0)
            done += int(ids.numel())
        barrier()
        sec = time.perf_counter() - t0
    model.per_crystal_eval = was_pc
    model.max_num_nodes = was_nmax
    model.train(was_training)
    sec = max_over_ranks(sec, world, dev)
    total = n_eval * world
    return {"metric": "inference sweep crystals/sec (forward only)", "value": total / sec, "unit": UNIT, "n_gpus": world,
            "seconds": sec, "crystals_evaluated": total, "batches_per_gpu": len(plans), "store_build_s": t_build,
            "config": {"workload": f"{MODEL_DESC} T={T}, inference-only DOS prediction sweep over {total} synthetic crystal "
                                   f"evaluations sharded over {world}xB200 (BASELINE configs[4]: 1 M at 8 GPUs), store of "
                                   f"{store_size} distinct crystals per GPU, ids -> on-device collate -> forward",
                       "batch": batch_size, "per_gpu": n_eval, "mode": "eager forward, per-crystal evaluation (no phantom keys), "
                       "host wall clock incl. launch overhead, max over ranks"}}


def inference_b1_leg(model, dev, steps, st):
    """The reference's evaluation loaders: batch_size 1 (main_eDOS.py:55-56), forward only; eager and graph replay."""
    from dostransformer_b200.graphed import GraphedStep
    from dostransformer_b200.synthetic import make_edos_batch
    sizes = [torch.tensor([n]) for n in (12, 20, 33)]
    gs = [make_edos_batch(1, seed=9000 + i, T=T, sizes=s).to(dev) for i, s in enumerate(sizes)]
    model.eval()
    model.per_crystal_eval = True
    res = {}
    with torch.no_grad():
        for name, fn in (("eager", lambda g: model(g)), ("graph", GraphedStep(model, "edos", train=False))):
            for g in gs:
                fn(g)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = max(steps, 12)
            a.record(st)
            for i in range(n):
                fn(gs[i % 3])
            b.record(st)
            torch.cuda.synchronize()
            res[name] = {"ms_per_crystal": a.elapsed_time(b) / n, "value": n / a.elapsed_time(b) * 1e3, "unit": UNIT}
    model.per_crystal_eval = False
    model.train()
    res["config"] = {"workload": f"{MODEL_DESC} T={T}, evaluation with batch_size 1 (main_eDOS.py:55-56), forward only, 1xB200"}
    return res


# ======================================================================================================== product arm
def run_product(args, rank: int, world: int, local_rank: int):
    import torch.distributed as dist
    from dostransformer_b200 import _lib as L
    from dostransformer_b200 import ops
    from dostransformer_b200.dp import GradReducer, live_named_parameters
    from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; dostransformer_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L.lib()
    pk = peaks()
    st = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    torch.manual_seed(0)
    model = DOSTransformer(GNN_LAYERS, T_LAYERS, 200, 41, 2, HIDDEN, dev, 0.0, n_energies=T, precision=args.precision).to(dev).train()

    # ------------------------------------------------------------------------------------------------ non-headline runs
    if args.workload == "sweep":
        res = sweep_leg(model, rank, world, dev, args.sweep_per_gpu, args.sweep_store, args.sweep_batch, barrier)
        if rank == 0:
            line = {"metric": res["metric"], "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": res["batches_per_gpu"],
                    "warmup": 2, "ms_per_step": res["seconds"] / res["batches_per_gpu"] * 1e3, "higher_is_better": True,
                    "scaling": "weak", "vs_baseline": None, "dtype": "bf16x3 operands, f32 accumulate", "data": "synthetic",
                    "config": res["config"], "detail": res}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.workload == "phonon":
        line = phonon_line(args, rank, world, dev, barrier, st, L)
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    B = args.batch
    strong = args.scaling == "strong"
    use_graph = {"on": True, "off": False, "auto": True}[args.graph]
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("DOST_BENCH_NO_SAMPLER"):
        sampler.start()

    if strong:
        if rank == 0:
            sampler.wait_ready()
        sampler.mark()
        res = strong_scaling_leg(model, rank, world, dev, args.steps, args.warmup, barrier, st, args.global_batch, use_graph, L)
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0:
            line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": "bf16x3 operands, f32 accumulate" if args.precision == "bf16x3" else args.precision,
                    "data": "synthetic", "config": res["config"], "clocks": clocks, "e2e": res["e2e"],
                    "gpu_launches": int(res["gpu_launches_per_step"] * args.steps), "ms_each_step_device": res["ms_each_step_device"]}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ------------------------------------------------------------------------------------------------ headline (weak scaling)
    NB = 3
    host = [b.pin_memory() for b in make_batches(rank if args.data_rank < 0 else args.data_rank, NB, B, args.workload)]
    nmax = max(int(torch.bincount(b.batch).max()) for b in host)
    n_nodes = sum(b.batch.numel() for b in host) / NB
    n_edges = sum(b.edge_index.shape[1] for b in host) / NB
    if world > 1:
        t = torch.tensor([nmax], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        nmax = int(t.item())
    if args.nmax > 0:
        nmax = max(nmax, args.nmax)
    model.max_num_nodes = nmax            # global padding length: the only cross-rank coupling besides the grads
    step = Runner(model, "edos", world, 1.0 / world, use_graph)
    resident = [b.clone().to(dev) for b in host]

    # ---------------------------------------------------------------- device-resident timing
    for i in range(max(args.warmup, NB)):      # (every batch signature once: graph capture / allocator warm-up)
        step(resident[i % NB])
    barrier()
    if rank == 0:
        sampler.wait_ready()     # a slow NVML attach must finish outside the timed region
    barrier()
    sampler.mark()
    l0 = L.launch_count()
    g0 = step.graph.launches if step.graph is not None else 0
    sec, dev_each = timed_steps(step, resident, args.steps, 0, barrier, st, args.ncu_window)
    launches = (L.launch_count() - l0) + ((step.graph.launches - g0) if step.graph is not None else 0)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:       # before any further step overwrites them
        dump_outputs(args.dump_outputs, step_outputs(model, step.last))
    sec = max_over_ranks(sec, world, dev)
    value = world * B * args.steps / sec

    # ---------------------------------------------------------------- end-to-end timing (host batches)
    h2d = host[0].nbytes()
    e2e_sec, per_step = e2e_steps(step, host, dev, args.steps, args.warmup, barrier)
    e2e_sec = max_over_ranks(e2e_sec, world, dev)
    e2e_val = world * B * args.steps / e2e_sec

    wl_desc = (f"{MODEL_DESC} T={T}, random-split shape (BASELINE configs[1]/[2]), {B} crystals per GPU" if args.workload == "edos"
               else f"{MODEL_DESC} T={T}, large-cell stress shape (BASELINE configs[3]: 200-400 atoms, 24 neighbours), {B} crystals per GPU")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32", "bf16x3": "bf16x3 operands, f32 accumulate", "bf16": "bf16 operands, f32 accumulate"}[
            args.precision], "data": "synthetic",
        "config": {"workload": wl_desc, "crystals_per_gpu": B,
                   "global_batch": B * world, "parallelism": f"dp{world}", "mean_nodes_per_batch": n_nodes,
                   "mean_edges_per_batch": n_edges, "nmax": nmax, "precision": PREC_DESC[args.precision],
                   "mode": step.describe(),
                   "l2_policy": "3 distinct batches rotated; per-step activations (>1 GB) exceed the 126 MB L2"},
        "clocks": clocks, "gpu_launches": int(launches), "ms_each_step_device": dev_each,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_sec / args.steps * 1e3, "ms_each_step": [round(x, 2) for x in per_step],
                "api": ("graphed.GraphedStep(model)(batch) [forward + ops.dos_loss + backward as one CUDA-graph replay]" if
                        step.graph is not None else "DOSTransformer(batch) + ops.dos_loss + loss.backward()") +
                       ", batch copied from pinned host memory on a copy stream one step ahead (double-buffered input pipeline), loss.item() every step; gc.freeze() after warm-up, cyclic GC "
                       "off inside the timed loop"},
    }
    fl = 3.0 * B * flops_per_crystal_fwd(n_nodes / B, n_edges / B, nmax)
    line["model_tflops"] = fl * args.steps / sec / 1e12
    headline_graph = step.graph is not None
    step.close()

    extras = not args.no_extras and args.workload == "edos" and B == 512

    # The side measurements hold collectives: a failure on one rank only would leave the others waiting.  A watchdog
    # bounds them: when it fires, rank 0 prints the headline line with what has finished and every rank exits.
    done = threading.Event()

    def watchdog():
        if not done.wait(args.extras_timeout):
            if rank == 0:
                line["extras_timed_out_after_s"] = args.extras_timeout
                print(json.dumps(line), flush=True)
            os._exit(0)
    if extras:
        threading.Thread(target=watchdog, daemon=True).start()

    def guarded(name, fn):
        """Side measurements never take the headline down; every rank runs them (they hold collectives)."""
        try:
            r = fn()
            if rank == 0:
                line[name] = r
        except Exception as ex:  # noqa: BLE001
            if rank == 0:
                line[name] = {"error": repr(ex)[:400]}

    if extras:
        # BASELINE configs[2] as written (strong scaling, global 512), configs[3] (large cell), configs[4] (sweep)
        guarded("strong_scaling", lambda: strong_scaling_leg(model, rank, world, dev, args.steps, args.warmup, barrier, st, 512,
                                                             True, L))
        guarded("large_cell", lambda: weak_leg(
            model, "large", "edos", 64, rank, world, dev, max(4, args.steps // 2), 3, barrier, st, use_graph, L,
            f"{MODEL_DESC} T={T}, large-cell stress shape (BASELINE configs[3]: 200-400 atoms, 24 neighbours), 64 crystals per GPU"))
        guarded("sweep", lambda: sweep_leg(model, rank, world, dev, args.sweep_per_gpu, args.sweep_store, args.sweep_batch, barrier))
    if world == 1 and extras:
        guarded("small_batch", lambda: {
            "train_b8_eager": weak_leg(model, "edos", "edos", 8, 0, 1, dev, args.steps, 3, barrier, st, False, L,
                                       f"{MODEL_DESC} T={T}, the reference's default batch of 8 crystals (utils.py:31), 1xB200"),
            "train_b8_graph": weak_leg(model, "edos", "edos", 8, 0, 1, dev, args.steps, 3, barrier, st, True, L,
                                       f"{MODEL_DESC} T={T}, the reference's default batch of 8 crystals (utils.py:31), 1xB200"),
            "train_b64_graph": weak_leg(model, "edos", "edos", 64, 0, 1, dev, args.steps, 3, barrier, st, True, L,
                                        f"{MODEL_DESC} T={T}, 64 crystals per GPU (config 3's per-GPU share at 8 GPUs), 1xB200"),
            "eval_b1": inference_b1_leg(model, dev, args.steps, st)})
        model.max_num_nodes = nmax
    if world == 1 and rank == 0:
        # BASELINE config 5 shape: forward-only DOS prediction, every crystal evaluated without padding (the reference's
        # eval loaders use batch_size 1), many crystals per launch, nothing read back per batch
        model.eval()
        model.per_crystal_eval = True
        with torch.no_grad():
            for i in range(2):
                model(resident[i % NB])
            torch.cuda.synchronize()
            i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            i0.record(st)
            for i in range(args.steps):
                model(resident[i % NB])
            i1.record(st)
            torch.cuda.synchronize()
        isec = i0.elapsed_time(i1) * 1e-3
        line["inference"] = {"value": B * args.steps / isec, "unit": UNIT, "ms_per_batch": isec / args.steps * 1e3,
                             "mode": "forward only, eval, per-crystal (no phantom keys), B crystals per launch"}
        model.per_crystal_eval = False
        model.train()
        # the step that follows the hot path (not part of the metric): fused AdamW over the live parameters, alone and in the
        # loop (fwd + bwd + AdamW every step: the weights' operand planes are re-split every step)
        from dostransformer_b200.optim import AdamW
        opt = AdamW(model.parameters(), lr=1e-4, weight_decay=1e-2)
        eager = Runner(model, "edos", 1, 1.0, False)
        esec, _ = timed_steps(eager, resident, args.steps, 3, barrier, st)
        line["eager_mode"] = {"value": B * args.steps / esec, "unit": UNIT, "ms_per_step": esec / args.steps * 1e3,
                              "what": "the same step issued kernel by kernel from Python (model(batch) + ops.dos_loss + "
                                      "loss.backward()), device-resident batches; bitwise the same results as the graph replay"}
        eager(resident[0])
        opt.step()
        torch.cuda.synchronize()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record(st)
        for _ in range(10):
            opt.step()
        o1.record(st)
        torch.cuda.synchronize()
        nlive = sum(p.numel() for p in model.parameters() if p.grad is not None)
        oms = o0.elapsed_time(o1) / 10
        line["optimizer"] = {"kind": "dost_adamw_step (fused multi-tensor AdamW, lr 1e-4, wd 1e-2)", "ms_per_step": oms,
                             "live_parameters": nlive, "gbytes_per_s": 28.0 * nlive / (oms * 1e-3) / 1e9}

        def opt_step(g):
            loss = eager(g)
            opt.step()
            return loss
        osec, _ = timed_steps(opt_step, resident, args.steps, 3, barrier, st)
        line["optimizer_in_loop"] = {"value": B * args.steps / osec, "unit": UNIT, "ms_per_step": osec / args.steps * 1e3,
                                     "what": "fwd + bwd + fused AdamW every step (weights change every step: their bf16 operand "
                                             "planes are re-split every step), eager, device-resident batches"}
        torch.manual_seed(0)     # the optimizer steps above moved the weights; nothing below depends on their values
        if extras:
            try:
                line["device_collate"] = device_collate_bench(host, dev, B, eager, args.steps, model)
            except Exception as ex:
                line["device_collate"] = {"error": repr(ex)}
        if args.precision == "bf16x3" and not args.no_alt:
            # the same step with plain bf16 operands (hi plane only), for reference: stated tolerance 5e-2 on gradients
            model.precision = "bf16"
            asec, _ = timed_steps(eager, resident, args.steps, 3, barrier, st)
            line["bf16_mode"] = {"value": B * args.steps / asec, "unit": UNIT, "ms_per_step": asec / args.steps * 1e3,
                                 "precision": PREC_DESC["bf16"]}
            model.precision = args.precision
        try:
            line.update(kernel_rooflines(B, pk, args.precision, ncu_traffic(args.precision)))
        except Exception as ex:  # keep the headline even if the side measurement fails
            line["roofline"] = {"error": repr(ex)}
        if extras:
            try:
                line["phonon"] = phonon_gpu_legs(dev, args.steps, barrier, st, L)
            except Exception as ex:
                line["phonon"] = {"error": repr(ex)[:400]}
        if not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            line["cpu_baseline"] = {k: v for k, v in cpu_leg("edos", args.cpu_sample, args.cpu_steps, 1, threads, 2000).items()}
            if extras:
                # the rows the reference actually runs: torch.set_num_threads(2) (main_eDOS.py:12, main_phDOS.py:12), its
                # default batch sizes (utils.py:31: 8; main_phDOS.py:52: 1), phonon in fp64
                line["cpu_baselines"] = {
                    "edos_b8_2threads": cpu_leg("edos", 8, 5, 1, 2, 2000),
                    "edos_b8_all_cores": cpu_leg("edos", 8, 8, 1, threads, 2000),
                    "phonon_fp64_b1_2threads": cpu_leg("phonon", 1, 15, 2, 2, 1000),
                    "phonon_fp64_b1_all_cores": cpu_leg("phonon", 1, 15, 2, threads, 1000)}
    done.set()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _phonon_model(dev):
    from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)       # main_phDOS.py:15-16
    try:
        torch.manual_seed(0)
        return DOSTransformer_phonon(3, 2, 118, 4, 256, dev, 0.0).to(dev).double().train()
    finally:
        torch.set_default_dtype(prev)


def phonon_gpu_legs(dev, steps, barrier, st, L):
    """BASELINE configs[0]'s model on the GPU: DOSTransformer_phonon, fp64 (FMA pipe), B = 1 (main_phDOS.py:52) and B = 64."""
    model = _phonon_model(dev)
    out = {}
    for B, graph in ((1, False), (1, True), (64, False), (64, True)):
        r = weak_leg(model, "phonon", "phonon", B, 0, 1, dev, max(steps, 8), 3, barrier, st, graph, L,
                     f"DOSTransformer_phonon hidden=256 L=3 t=2 T=51, fp64 (main_phDOS.py defaults), {B} crystal(s) per step, 1xB200")
        out[f"train_b{B}_{'graph' if graph else 'eager'}"] = r
    return out


def phonon_line(args, rank, world, dev, barrier, st, L):
    B = args.batch if args.batch != 512 else 1
    use_graph = {"on": True, "off": False, "auto": True}[args.graph]
    model = _phonon_model(dev)
    r = weak_leg(model, "phonon", "phonon", B, rank, world, dev, args.steps, args.warmup, barrier, st, use_graph, L,
                 f"DOSTransformer_phonon hidden=256 L=3 t=2 T=51, fp64 (main_phDOS.py defaults, BASELINE configs[0] on the GPU), "
                 f"{B} crystal(s) per GPU")
    return {"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": r["config"], "gpu_launches": int(r["gpu_launches_per_step"] * args.steps),
            "ms_each_step_device": r["ms_each_step_device"]}


def device_collate_bench(host, dev, B, step, steps, model):
    """SURVEY 8f-3: the batches' crystals packed once into HBM-resident tables; a step sends B crystal ids and the batch is
    assembled on the device (csrc/collate.cu).  Reports the assembly alone (CUDA events, bytes = read + written) and the
    end-to-end step that starts from host ids."""
    from dostransformer_b200.collate import PackedCrystals, split_batch
    graphs = [g for b in host for g in split_batch(b)]
    pk = PackedCrystals.from_graphs(graphs, device=dev)
    gen = torch.Generator().manual_seed(7)
    ids = [torch.randperm(len(pk), generator=gen)[:B].pin_memory() for _ in range(6)]
    for i in ids[:3]:
        b = pk.collate(i)
    torch.cuda.synchronize()
    st = torch.cuda.current_stream()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 30
    c0.record(st)
    for r in range(reps):
        b = pk.collate(ids[r % len(ids)])
    c1.record(st)
    torch.cuda.synchronize()
    cms = c0.elapsed_time(c1) / reps
    nbytes = 2.0 * b.nbytes()
    for i in ids:                                       # every batch shape once: allocator warm-up
        step(pk.collate(i)).item()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for r in range(steps):
        g = pk.collate(ids[r % len(ids)])
        step(g).item()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    return {"value": B * steps / sec, "unit": UNIT, "ms_per_step": sec / steps * 1e3, "h2d_bytes_per_step": 8 * B,
            "d2h_bytes_per_step": 4, "collate_ms": cms, "collate_gbytes_per_s": nbytes / (cms * 1e-3) / 1e9,
            "collate_launches": len(pk.tables) + 2, "store_bytes": pk.nbytes(), "crystals_in_store": len(pk),
            "note": "crystal ids from host memory -> PackedCrystals.collate (segmented copies on the device) -> fwd+bwd; "
                    "collate_ms includes the host-side launch cost of its kernels"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="product", choices=["product", "reference"])
    ap.add_argument("--batch", type=int, default=512, help="crystals per GPU (weak scaling)")
    ap.add_argument("--global-batch", type=int, default=512, help="global batch of --scaling strong")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak = the headline (per-GPU batch fixed); strong = BASELINE configs[2] as written (global batch "
                         "through the LPT sharder)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="whole-step CUDA-graph replay (auto = on, falling back to the eager step if a capture fails)")
    ap.add_argument("--cpu-sample", type=int, default=64, help="crystals per step of the CPU baseline sample")
    ap.add_argument("--cpu-steps", type=int, default=20, help="timed CPU baseline steps (bounded sample, ~10-20 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the extra bf16-mode measurement")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip the other BASELINE configurations")
    ap.add_argument("--extras-timeout", type=float, default=240.0, help="seconds after which the side measurements are abandoned")
    ap.add_argument("--workload", default="edos", choices=["edos", "large", "phonon", "sweep"],
                    help="edos = the headline configuration; large = BASELINE configs[3] (use --batch 64); phonon = configs[0] "
                         "on the GPU (fp64); sweep = configs[4] (forward-only prediction sweep)")
    ap.add_argument("--sweep-per-gpu", type=int, default=125000, help="crystal evaluations per GPU of the sweep (1 M at 8 GPUs)")
    ap.add_argument("--sweep-store", type=int, default=4096, help="distinct synthetic crystals per GPU in the sweep's store")
    ap.add_argument("--sweep-batch", type=int, default=1024)
    ap.add_argument("--nmax", type=int, default=0, help="(experiments) force a larger global padding length")
    ap.add_argument("--data-rank", type=int, default=-1, help="(experiments) generate the batches of another rank")
    ap.add_argument("--precision", default=os.environ.get("DOST_PRECISION", "bf16x3"), choices=["fp32", "bf16x3", "bf16"],
                    help="GEMM path: fp32 FMA pipe | tcgen05 bf16x3 (fp32 parity, default) | tcgen05 bf16")
    ap.add_argument("--ncu-window", action="store_true", help="bracket the first timed step with cudaProfilerStart/Stop (for "
                    "ncu --profile-from-start off; a number printed under a profiler is not a bench value)")
    ap.add_argument("--energies", type=int, default=T, help="energy-grid length (201 = the reference's eDOS grid; 1001 = the "
                    "long-grid variant of the large-cell stress configuration); not the headline line when changed")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps write the loss and the parameter gradients "
                    "of the last timed step as DIR/<name>.npy (float32, float64 for a float64 model; at most 64 MB in all, "
                    "a fixed seeded sample of every array beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "product" or args.scaling != "weak" or args.workload not in ("edos", "large")):
        ap.error("--dump-outputs covers the weak-scaling train-step line of the product (--workload edos or large)")
    if args.energies != T:
        globals()["T"] = args.energies
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_product(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
