"""Whole-step CUDA-graph replay (dostransformer_b200.graphed) against the eager step: same kernels, same order, so
losses and gradients must be BITWISE equal; bucket-padded batches must leave the real crystals' loss and gradients
unchanged up to fp32 summation order."""
import pytest
import torch

from dostransformer_b200 import ops
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
from dostransformer_b200.graphed import GraphedStep, batch_signature
from dostransformer_b200.optim import AdamW
from dostransformer_b200.synthetic import make_edos_batch, pad_edos_batch

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _model(h=128, seed=0, prec="bf16x3"):
    torch.manual_seed(seed)
    return DOSTransformer(2, 2, 200, 41, 2, h, torch.device(DEV), 0.0, precision=prec).to(DEV).train()


def _eager(m, g, weight=1.0):
    m.zero_grad(set_to_none=True)
    dg, _, ds = m(g)
    loss = ops.dos_loss(dg, ds, g.y_ft, mode="edos", beta=1.0)
    if weight != 1.0:
        loss = loss * weight
    loss.backward()
    return loss.detach().clone(), {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}


@pytest.mark.parametrize("prec", ["bf16x3", "fp32"])
def test_graph_replay_is_bitwise_the_eager_step(prec):
    m = _model(prec=prec)
    step = GraphedStep(m, "edos")
    sizes = torch.tensor([5, 9, 3, 12, 7, 8])
    a = [make_edos_batch(6, seed=10 + i, sizes=sizes).to(DEV) for i in range(3)]       # one signature, three batches
    b = [make_edos_batch(4, seed=20 + i, sizes=sizes[:4] + 2).to(DEV) for i in range(2)]  # a second signature
    assert batch_signature(a[0]) == batch_signature(a[1]) != batch_signature(b[0])
    for g in (a[0], b[0], a[1], b[1], a[2], a[0]):
        want_loss, want = _eager(m, g)
        got_loss = step(g)
        assert torch.equal(got_loss.detach(), want_loss)
        got = {k: p.grad for k, p in m.named_parameters() if p.grad is not None}
        assert set(got) == set(want)
        for k in want:
            assert torch.equal(got[k], want[k]), k
    assert step.captures == 2 and step.replays == 6 and step.launches > 0


def test_graph_replay_sees_optimizer_updates():
    """The weights' bf16 operand planes are re-split inside the graph: a replay after an optimizer step (fused AdamW
    writes through raw pointers) must equal the eager step on the updated weights."""
    m = _model()
    step = GraphedStep(m, "edos")
    opt = AdamW(m.parameters(), lr=1e-2, weight_decay=1e-2)
    g = make_edos_batch(5, seed=31, mean_atoms=8.0).to(DEV)
    l0 = step(g).detach().clone()
    for _ in range(3):
        opt.step()
        step(g)
    l1 = step(g).detach().clone()
    want_loss, want = _eager(m, g)
    assert torch.equal(l1, want_loss) and not torch.equal(l0, l1)
    step(g)
    for k, p in m.named_parameters():
        if p.grad is not None:
            assert torch.equal(p.grad, want[k]), k
    # a write that bypasses the version counter is seen too (the graph never trusts the cache)
    with torch.no_grad():
        m.fc.weight.data.mul_(1.5)
    l2 = step(g).detach().clone()
    ops.invalidate_weight_planes(m)
    want2, _ = _eager(m, g)
    assert torch.equal(l2, want2)


@pytest.mark.parametrize("prec,tol", [("fp32", 1e-4), ("bf16x3", 5e-3)])
def test_bucket_padding_leaves_the_real_crystals_unchanged(prec, tol):
    """Dummy crystals contribute exact zeros to every gradient; what differs from the unpadded step is the summation
    grouping (split-K chunks move with the row count).  fp32 path: fp32 rounding only (1e-4 on the cancellation-prone
    first-stack tensors).  bf16x3: the tensor-core accumulation order moves too and the same tensors amplify it to the
    level of that path's stated gradient floor (tests/test_gpu_model.py GRAD_FLOOR: rel-L2 2e-3 vs fp64; two bf16x3
    evaluations with different groupings may differ by twice that).  The semantic no-op itself is pinned on the CPU oracle
    (tests/test_host.py::test_bucket_padding_is_a_semantic_no_op_for_the_real_crystals)."""
    m = _model(h=128, prec=prec)
    g = make_edos_batch(7, seed=41, mean_atoms=9.0)
    p = pad_edos_batch(g, node_bucket=64, dummies=3)
    assert p.n_valid == 7 and p.system.numel() >= 10 and p.x.shape[0] % 64 == 0      # (the dummy count doubles until each fits)
    n = torch.bincount(p.batch)
    assert int(n[7:].max()) <= int(n[:7].max())
    want_loss, want = _eager(m, g.clone().to(DEV))
    step = GraphedStep(m, "edos")
    for _ in range(2):
        got_loss = step(p.clone().to(DEV))
    assert abs(got_loss.item() - want_loss.item()) <= 2e-6 * abs(want_loss.item())
    errs = {k: ((pr.grad.double() - want[k].double()).norm() / want[k].double().norm().clamp_min(1e-30)).item()
            for k, pr in m.named_parameters() if k in want}
    bad = {k: v for k, v in errs.items() if not v < tol}
    assert not bad, bad
    # model outputs of the real crystals are the unpadded ones
    m.eval()
    with torch.no_grad():
        dg_p, x_p, ds_p = m(p.clone().to(DEV))
        dg, x, ds = m(g.clone().to(DEV))
    # (1e-4 = the stated output tolerance: with more rows some small Linears move from the fp32 FMA kernel to the
    # bf16x3 tensor-core kernel, ops.planes_gemm_ok)
    assert (dg_p[:7] - dg).abs().max().item() <= 1e-4 * dg.abs().max().item()
    assert (x_p[:x.shape[0]] - x).abs().max().item() <= 1e-4 * x.abs().max().item()


def test_graphed_inference_matches_eager():
    m = _model().eval()
    m.per_crystal_eval = True
    step = GraphedStep(m, "edos", train=False)
    gs = [make_edos_batch(5, seed=50 + i, sizes=torch.tensor([4, 6, 2, 9, 5])).to(DEV) for i in range(3)]
    for g in gs:
        with torch.no_grad():
            want = m(g)
        got = step(g)
        for a, b in zip(got, want):
            assert torch.equal(a, b)
    assert step.captures == 1


def test_cached_index_tensors_outlive_captured_graphs():
    """ops._arange_i32 hands out views of one cached index tensor and replaces it when a larger one is needed.  A CUDA graph
    captured before the replacement still reads the OLD tensor on every replay: it must stay alive (it used to be freed,
    its block re-used, and the large-cell bench - second batch with more edges than the first - gathered through garbage
    indices: an illegal address)."""
    import torch
    from dostransformer_b200 import ops
    dev = torch.device("cuda")
    n1 = 5000
    a = torch.randn(n1, 64, device=dev)
    b = torch.randn(n1, 64, device=dev)
    out = torch.empty(n1, 64, device=dev)
    ops._axpy2(a, b, out)                         # warm-up outside the capture (creates / uses the cached index tensor)
    torch.cuda.synchronize()
    key = (str(a.device),)
    old = ops._ARANGE_CACHE[key]
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            ops._axpy2(a, b, out)                 # gather_rows with the identity index: reads the cached tensor
    torch.cuda.current_stream().wait_stream(s)
    big = ops._arange_i32(old.numel() + 1, a.device)   # outgrows the cache: a new tensor replaces the old one
    assert ops._ARANGE_CACHE[key].data_ptr() != old.data_ptr()
    del old, big
    junk = [torch.full((1 << 20,), -7, dtype=torch.int32, device=dev) for _ in range(8)]     # would re-use a freed block
    out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, a + b)
    del junk


def test_graph_replay_follows_the_models_padding_length():
    """model.max_num_nodes (the data-parallel global padding length set by the sharder) is a host integer baked into the
    captured launches: the graph cache is keyed on it, so a change between two steps with identical batch shapes gives the
    eager result for the NEW value (more phantom keys) instead of a stale replay."""
    m = _model()
    step = GraphedStep(m, "edos")
    g = make_edos_batch(5, seed=41, mean_atoms=8.0).to(DEV)
    losses = {}
    for nm in (None, g.max_num_nodes + 9, None, g.max_num_nodes + 9):
        m.max_num_nodes = nm
        want, _ = _eager(m, g)
        got = step(g)
        assert torch.equal(got.detach(), want), nm
        losses[nm] = want.item()
    m.max_num_nodes = None
    assert step.captures == 2 and losses[None] != losses[g.max_num_nodes + 9]


def test_bench_dumps_the_last_timed_step(tmp_path):
    """bench.py --steps K --dump-outputs DIR: the dumped loss and gradients are those of the K-th timed step (batch
    (K - 1) mod 3 of the rotation, not the warm-up's last), recomputed here eagerly from the same seeded model and batch."""
    import json
    import os
    import subprocess
    import sys
    import numpy as np
    from conftest import ROOT
    K, B = 5, 8
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(K), "--warmup", "0", "--batch", str(B),
                        "--no-extras", "--no-cpu-baseline", "--no-alt", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, DOST_BENCH_NO_SAMPLER="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == K and len(line["ms_each_step_device"]) == K
    batches = [make_edos_batch(B, seed=2000 + i, T=201) for i in range(3)]
    torch.manual_seed(0)
    m = DOSTransformer(3, 2, 200, 41, 2, 256, torch.device(DEV), 0.0, n_energies=201, precision="bf16x3").to(DEV).train()
    m.max_num_nodes = max(int(torch.bincount(b.batch).max()) for b in batches)
    loss, grads = _eager(m, batches[(K - 1) % 3].to(DEV))
    want = {"loss": loss, **{f"grad.{k}": v for k, v in grads.items()}}
    assert sorted(p.name[:-4] for p in out.iterdir()) == sorted(want)
    assert sum(p.stat().st_size for p in out.iterdir()) <= 64 << 20
    for k, v in want.items():
        got = np.load(out / f"{k}.npy")
        assert got.dtype == np.float32 and got.shape == tuple(v.shape), k
        got, v = torch.from_numpy(got).double(), v.cpu().double()
        assert ((got - v).norm() / v.norm().clamp_min(1e-30)).item() < 1e-5, k
