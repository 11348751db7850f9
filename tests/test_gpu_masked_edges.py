"""Masked phonon edges: a batch's ``edge_mask`` keeps only some edges, and ``phonon_topology(..., skin=s, masked=True)``
follows the phonon edge set inside one CUDA graph.

1. Kernels: dost_csr_build_masked and dost_gather_rows_masked against numpy bit for bit (the all-ones mask is bitwise the
   unmasked kernels); dost_edge_within against the numpy comparison, within 1 ulp of r_max too.
2. The model contract: the phonon model on a masked batch against the model on the subset batch.
3. The default path: a batch without edge_mask calls the same entry points and kernels; the eDOS model and
   dp.shard_batch refuse a mask.
4. The masked topology against phonon_graph_batch at moved geometries and across r_max; the flag; no host sync.
5. Replays: one capture across a crossing, each replay bitwise the eager masked step."""
import numpy as np
import pytest
import torch

from conftest import relerr
from dostransformer_b200 import _lib as L
from dostransformer_b200 import dp
from dostransformer_b200 import neighbors as NB
from dostransformer_b200 import ops
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
from dostransformer_b200.graphed import GraphedStep
from oracle import dost_oracle as O
from test_gpu_geometry_grad import GRAD_FLOOR, PHONON_FLOOR, _grade, _phonon_inputs, _phonon_oracle
from test_gpu_skin_topology import _complete, _crystals, _flag, _pair
from test_gpu_structure_step import EPS64, _check, _leaves, _perturb, _Phonon, _phonon_model, _step

pytestmark = pytest.mark.gpu
DEV = "cuda"
SIZES = {"B1": [1], "B5": [3, 1, 4, 2, 6], "B23": [2, 5, 1, 3, 4, 6, 2, 1, 5, 3, 2, 4, 6, 1, 3, 5, 2, 4, 3, 6, 1, 2, 5]}
# Parameter gradients and live edge_vec.grad rows of a masked batch are the subset batch's terms summed in another order
# (the weight-gradient GEMMs reduce over all E rows, the masked ones contributing exact zeros, tiled by E).  A sum of
# n <= 10^4 fp64 terms moves by at most n eps sum|terms| ~ 1e-12 sum|terms|; 1e-9 of the tensor's max leaves three orders
# of magnitude for cancellation and the chain through the layers.
FP64_ORDER = 1e-9


def _np(t):
    return t.detach().cpu().numpy()


# ------------------------------------------------------------------ 1. kernels
def _csr_numpy(key, mask, size):
    live = np.nonzero(mask != 0)[0]
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(key[live], minlength=size))]).astype(np.int32)
    perm = np.concatenate([live[np.argsort(key[live], kind="stable")], np.nonzero(mask == 0)[0]]).astype(np.int32)
    return rowptr, perm


def _gather_numpy(src, key, rowptr, mask):
    cnt = (rowptr[1:] - rowptr[:-1])[key]
    sc = np.where(cnt > 1, src.dtype.type(1) / np.maximum(cnt, 1).astype(src.dtype), src.dtype.type(1))
    out = src[key] * sc[:, None]
    return np.where((mask != 0)[:, None], out, 0).astype(src.dtype)


@pytest.mark.parametrize("case", ["random", "ones", "zeros", "empty_node", "E0"])
def test_masked_csr_and_gather_are_numpy_bit_for_bit(case):
    rng = np.random.default_rng(7)
    N, E = 37, (0 if case == "E0" else 1500)
    key = rng.integers(0, N, E).astype(np.int32)
    mask = {"random": rng.integers(0, 2, E), "ones": np.ones(E), "zeros": np.zeros(E), "E0": np.ones(0),
            "empty_node": key != 5}[case].astype(np.uint8)
    k, m = torch.from_numpy(key).to(DEV), torch.from_numpy(mask).to(DEV)
    csr, mx = ops.csr_build(k, N, want_max=True, mask=m)
    rowptr, perm = _csr_numpy(key, mask, N)
    assert np.array_equal(_np(csr.rowptr), rowptr) and np.array_equal(_np(csr.perm), perm), case
    assert int(mx) == int((rowptr[1:] - rowptr[:-1]).max())
    if case == "empty_node":
        assert rowptr[6] == rowptr[5]
    for dtype, W in ((torch.float64, 64), (torch.float64, 3), (torch.float32, 256), (torch.float32, 5)):
        src = torch.randn(N, W, dtype=dtype, generator=torch.Generator().manual_seed(W)).to(DEV)
        for deg in (None, csr.rowptr):
            got = ops.gather_rows_raw(src, k, deg_rowptr=deg, mask=m)
            want = _gather_numpy(_np(src), key, rowptr if deg is not None else np.zeros(N + 1, np.int32), mask)
            assert got.cpu().numpy().tobytes() == want.tobytes(), (case, dtype, W)
            assert bool((got[~m.bool()] == 0).all())
            if case == "ones":           # bitwise the unmasked kernels
                assert torch.equal(got, ops.gather_rows_raw(src, k, deg_rowptr=deg))
    if case == "ones":
        plain, pmx = ops.csr_build(k, N, want_max=True)
        assert torch.equal(plain.rowptr, csr.rowptr) and torch.equal(plain.perm, csr.perm) and torch.equal(pmx, mx)


def test_edge_within_is_the_fill_comparison():
    r = 4.0
    rng = np.random.default_rng(8)
    near = [np.nextafter(r, 0.0), r, np.nextafter(r, 8.0), np.nextafter(np.nextafter(r, 0.0), 0.0), 0.0, np.nan, np.inf]
    d = np.concatenate([rng.uniform(0.0, 4.5, 5000), near])
    mask = torch.empty(d.size, dtype=torch.uint8, device=DEV)
    L.check(L.lib().dost_edge_within(L.p(torch.from_numpy(d).to(DEV)), d.size, r, L.p(mask), L.stream()))
    assert np.array_equal(_np(mask), (d < r).astype(np.uint8))
    assert _np(mask)[-7:].tolist() == [1, 0, 0, 1, 1, 0, 0]


# ------------------------------------------------------------------ 2. the model contract
def _model(H, prec="fp64", p=0.0):
    torch.set_default_dtype(torch.float64 if prec == "fp64" else torch.float32)       # (restored by the conftest guard)
    torch.manual_seed(H)
    kw = {} if prec == "fp64" else {"precision": prec}
    return DOSTransformer_phonon(2, 1, 118, 4, H, torch.device(DEV), p, **kw).to(DEV).train()


def _run(model, g):
    """Forward + loss + backward on a batch whose edge_vec is a leaf: (outputs, loss, parameter grads, edge_vec.grad)."""
    model.zero_grad(set_to_none=True)
    out = model(g)
    loss = ops.dos_loss(out[0], out[2], g.phdos, mode="phonon")
    loss.backward()
    grads = {k: q.grad.clone() for k, q in model.named_parameters() if q.grad is not None}
    return [o.detach() for o in out], loss.detach(), grads, g.edge_vec.grad.clone()


def _candidate_batch(sizes, seed, dtype):
    """The list at 4.5 A of a seeded batch with bonds, a random mask that keeps the identity edges and drops at least one
    bond, and the batch of the kept edges."""
    while True:               # (a lone atom in a wide cell has no bond: take the next seed)
        _, lattice, pos, node_ptr, x, system, ph = _phonon_inputs(seed, sizes)
        full = NB.phonon_graph_batch(lattice, pos, node_ptr, x.to(DEV, dtype), r_max=4.5, system=system.to(DEV),
                                     phdos=ph.to(DEV, dtype))
        ei, sh = full.edge_index, full.edge_shift
        identity = (ei[0] == ei[1]) & (sh == 0).all(dim=1)
        if bool((~identity).any()):
            break
        seed += 1000
    drop = ~identity & (torch.rand(ei.shape[1], generator=torch.Generator().manual_seed(seed)) >= 0.6).to(DEV)
    drop[int(torch.nonzero(~identity)[0])] = True
    keep = ~drop
    vec = full.edge_vec.detach().to(dtype)

    def batch(mask):
        g = full.clone()
        g.edge_vec = vec.clone().requires_grad_()
        if mask is None:
            return g
        g["edge_mask"] = mask
        return g

    sub = batch(None)
    sub.edge_index, sub.edge_shift = ei[:, keep], sh[keep]
    sub.edge_vec = vec[keep].clone().requires_grad_()
    return batch, keep, identity, sub


@pytest.mark.parametrize("H", [64, 256])
@pytest.mark.parametrize("B", list(SIZES))
def test_masked_batch_is_the_subset_batch_fp64(H, B):
    model = _model(H)
    batch, keep, identity, sub = _candidate_batch(SIZES[B], 50 + H + len(SIZES[B]), torch.float64)
    assert bool((~keep).any())
    want = _run(model, sub)
    for mask in (keep.to(torch.uint8), keep):                   # uint8 or bool
        got = _run(model, batch(mask))
        assert all(torch.equal(u, v) for u, v in zip(got[0], want[0])), (H, B)   # dos_global, x, dos_system
        assert torch.equal(got[1], want[1])
        assert got[2].keys() == want[2].keys()
        for k in want[2]:
            assert relerr(got[2][k], want[2][k]) <= FP64_ORDER, (k, relerr(got[2][k], want[2][k]))
        ev = got[3]
        assert bool((ev[~keep] == 0).all())                    # masked rows: exact zeros
        live_id, want_id = identity[keep], want[3]
        for rows in (live_id, ~live_id):                        # the ~1e12 self-loop rows and the others, each on its own
            if bool(rows.any()):
                assert relerr(ev[keep][rows], want_id[rows]) <= FP64_ORDER
    # all ones: bitwise the unmasked batch, outputs and every gradient
    plain = _run(model, batch(None))
    ones = _run(model, batch(torch.ones_like(keep)))
    assert all(torch.equal(u, v) for u, v in zip(ones[0], plain[0])) and torch.equal(ones[1], plain[1])
    assert all(torch.equal(ones[2][k], plain[2][k]) for k in plain[2]) and torch.equal(ones[3], plain[3])


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_masked_batch_is_the_subset_batch_fp32_and_bf16x3(prec):
    model = _model(64, prec)
    batch, keep, identity, sub = _candidate_batch(SIZES["B5"], 60, torch.float32)
    want = _run(model, sub)
    got = _run(model, batch(keep.to(torch.uint8)))
    for u, v in zip(got[0], want[0]):
        assert relerr(u, v) < 1e-4
    for k in want[2]:
        _grade(k, got[2][k], want[2][k], GRAD_FLOOR[prec])
    assert bool((got[3][~keep] == 0).all())
    _grade("edge_vec", got[3][keep][~identity[keep]], want[3][~identity[keep]], GRAD_FLOOR[prec])
    plain = _run(model, batch(None))
    ones = _run(model, batch(torch.ones_like(keep)))
    assert all(torch.equal(u, v) for u, v in zip(ones[0], plain[0]))
    assert all(torch.equal(ones[2][k], plain[2][k]) for k in plain[2]) and torch.equal(ones[3], plain[3])


# ------------------------------------------------------------------ 3. the default path
class _Calls:
    """A stand-in for the loaded library that records the entry points called through it."""

    def __init__(self, lib):
        self.lib, self.names = lib, []

    def __getattr__(self, name):
        if name.startswith("dost_"):
            self.names.append(name)
        return getattr(self.lib, name)


def _entry_points_and_kernels(model, g, monkeypatch):
    calls = _Calls(L.lib())
    monkeypatch.setattr(L, "lib", lambda: calls)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _run(model, g)
        torch.cuda.synchronize()
    monkeypatch.undo()
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "dost" in e.name]
    return calls.names, kernels


def test_without_edge_mask_the_same_entry_points_and_kernels_run(monkeypatch):
    model = _model(64)
    batch, keep, _, _ = _candidate_batch(SIZES["B5"], 70, torch.float64)
    plain, plain_k = _entry_points_and_kernels(model, batch(None), monkeypatch)
    masked, masked_k = _entry_points_and_kernels(model, batch(torch.ones_like(keep)), monkeypatch)
    assert not any(n.endswith("_masked") for n in plain)
    # the masked batch calls the masked siblings in the same places, and nothing else changes
    assert [n.replace("_masked", "") for n in masked] == plain
    assert masked.count("dost_csr_build_masked") == 2 and masked.count("dost_gather_rows_masked") == 2   # 2 layers
    assert len(plain_k) == len(masked_k) and len(plain_k) > 0


def test_edos_model_and_shard_batch_refuse_an_edge_mask():
    from dostransformer_b200.synthetic import make_edos_batch
    torch.manual_seed(0)
    model = DOSTransformer(2, 1, 200, 41, 2, 128, torch.device(DEV), 0.0).to(DEV)
    g = make_edos_batch(3, seed=1).to(DEV)
    g["edge_mask"] = torch.ones(g.edge_index.shape[1], dtype=torch.uint8, device=DEV)
    with pytest.raises(NotImplementedError):
        model(g)
    with pytest.raises(NotImplementedError):
        dp.shard_batch(g, 2, 51)


# ------------------------------------------------------------------ 4. the masked topology
def _masked(d, skin=0.5):
    return NB.phonon_topology(d.lattice, d.pos, d.node_ptr, skin=skin, masked=True)


def _grad_bound(g, node_ptr, N):
    """Per-entry bounds for pos / lattice gradients summed over the candidates instead of the fresh list: the same nonzero
    terms g_e (edge_vec.grad of the fresh batch, identity edges dropped), sums of n terms within n eps sum|terms|."""
    ei, sh = g.edge_index, g.edge_shift
    a = g.edge_vec.grad.abs().masked_fill(((ei[0] == ei[1]) & (sh == 0).all(dim=1))[:, None], 0.0)
    S_pos = torch.zeros(N, 3, dtype=torch.float64, device=DEV).index_add_(0, ei[0], a).index_add_(0, ei[1], a)
    crystal = torch.repeat_interleave(torch.arange(node_ptr.numel() - 1, device=DEV), node_ptr[1:] - node_ptr[:-1])
    S_lat = torch.zeros(node_ptr.numel() - 1, 3, 3, dtype=torch.float64, device=DEV).index_add_(
        0, crystal[ei[0]], sh.abs().double()[:, :, None] * a[:, None, :])
    n = 2 * ei.shape[1]
    return n * EPS64 * S_pos, n * EPS64 * S_lat


def _against_fresh(model, topo, lat, p, x, per, node_ptr, oracle=None):
    """The masked topology's step at (lat, p) against the step on phonon_graph_batch there."""
    la, pa = _leaves(lat, p)
    ga = NB.phonon_graph_batch(la, pa, node_ptr, x, **per)
    ga.edge_vec.retain_grad()
    model.zero_grad(set_to_none=True)
    want_out = [o.detach() for o in model(ga)]
    want = _step(model, ga, "phonon", la, pa)
    lb, pb = _leaves(lat, p)
    gb = topo.batch(lb, pb, x, **per)
    keep = gb.edge_mask.bool()
    assert torch.equal(gb.edge_index[:, keep], ga.edge_index) and torch.equal(gb.edge_shift[keep], ga.edge_shift)
    assert torch.equal(gb.edge_vec[keep], ga.edge_vec)
    model.zero_grad(set_to_none=True)
    got_out = [o.detach() for o in model(gb)]
    assert all(torch.equal(u, v) for u, v in zip(got_out, want_out))
    got = _step(model, gb, "phonon", lb, pb)
    assert torch.equal(got[0], want[0])
    for k in want[1]:
        assert relerr(got[1][k], want[1][k]) <= FP64_ORDER, k
    b_pos, b_lat = _grad_bound(ga, node_ptr, p.shape[0])
    assert bool(((got[2] - want[2]).abs() <= b_pos).all()) and bool(((got[3] - want[3]).abs() <= b_lat).all())
    if oracle is not None:
        sd, cells, xr, system, ph, sizes = oracle
        _, _, _, r_pos, r_lat = _phonon_oracle(sd, _crystals(lat, p, node_ptr), lat, p, xr, system, ph, sizes)
        _grade("pos", got[2], r_pos, PHONON_FLOOR)
        _grade("lattice", got[3], r_lat, PHONON_FLOOR)
    return keep


def test_masked_topology_is_the_fresh_list_at_moved_geometries():
    d = _Phonon()
    model = _phonon_model()
    sd = {k: v.cpu() for k, v in O.state_dict_of(model).items()}
    _, _, _, _, xr, system, ph = _phonon_inputs(31, [3, 1, 4, 2, 6])
    oracle = (sd, d.cells, xr, system, ph, [3, 1, 4, 2, 6])
    topo = _masked(d)
    assert topo.src.numel() > NB.phonon_topology(d.lattice, d.pos, d.node_ptr).src.numel()
    base = _against_fresh(model, topo, d.lattice, d.pos, d.x, d.per, d.node_ptr, oracle)
    changed = 0
    for seed in range(4):
        lat, p = _perturb(d.lattice, d.pos, 200 + seed, 0.001, 0.03)
        assert _complete(topo, lat, p, 4.0), seed
        keep = _against_fresh(model, topo, lat, p, d.x, d.per, d.node_ptr, oracle if seed == 0 else None)
        changed += int(not torch.equal(keep, base))
        assert topo.matches(lat, p)
    assert changed > 0                                        # bonds did cross r_max
    assert _flag(topo) == 0


def test_a_bond_crossing_r_max_is_followed_both_ways():
    lattice, pos, node_ptr, x = _pair()
    per = {"system": torch.zeros(1, dtype=torch.int64, device=DEV),
           "phdos": torch.rand(1, 51, dtype=torch.float64, generator=torch.Generator().manual_seed(3)).to(DEV)}
    model = _phonon_model()
    topo = NB.phonon_topology(lattice, pos, node_ptr, skin=0.5, masked=True)
    held = NB.phonon_topology(lattice, pos, node_ptr, skin=0.5)
    assert topo.src.numel() == 4
    crossed = pos.clone()
    crossed[1, 0] = 5.1                                       # 3.9 A -> 4.1 A: the bond leaves r_max
    lives = []
    for p in (pos, crossed, pos):
        lives.append(int(_against_fresh(model, topo, lattice, p, x, per, node_ptr).sum()))
        held.batch(lattice, p, x, **per)
        assert _flag(topo) == 0
    assert lives == [4, 2, 4] and _flag(held) == 1           # the held skin topology flags what the masked one follows
    topo.batch(lattice, pos + 0.3, x, **per)                  # a move past the completeness bound
    assert _flag(topo) == 1
    topo.batch(lattice, pos, x, **per)
    assert _flag(topo) == 1                                   # sticky
    topo.clear()
    assert _flag(topo) == 0
    assert _flag(NB.phonon_topology(lattice, pos + 0.3, node_ptr, skin=0.5, masked=True)) == 0   # a rebuild starts clear
    with pytest.raises(ValueError):
        NB.phonon_topology(lattice, pos, node_ptr, masked=True)


def test_masked_batch_does_not_synchronise():
    d = _Phonon()
    topo = _masked(d)
    la, pa = _leaves(*_perturb(d.lattice, d.pos, 3, 0.001, 0.03))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        topo.batch(la, pa, d.x, **d.per)
    finally:
        torch.cuda.set_sync_debug_mode("default")


# ------------------------------------------------------------------ 5. replays
def _crossing_geometries(d, topo, n, base_seed):
    geoms = [_perturb(d.lattice, d.pos, base_seed + i, 0.001, 0.03) for i in range(n)]
    masks = [topo.batch(*g, d.x, **d.per).edge_mask.clone() for g in geoms]
    topo.clear()
    assert any(not torch.equal(masks[0], m) for m in masks[1:])     # the live set changes between the geometries
    return geoms


def test_replays_across_a_crossing_are_the_eager_masked_step():
    d = _Phonon()
    model = _phonon_model()
    eager_topo, topo = _masked(d), _masked(d)
    geoms = _crossing_geometries(d, eager_topo, 4, 220)
    step = GraphedStep(model, "phonon", structure=True)
    far = _perturb(d.lattice, d.pos, 230, 0.0, 0.6)
    for i, (lat, p) in enumerate(geoms + [far] + geoms[:1]):
        la, pa = _leaves(lat, p)
        want = _step(model, eager_topo.batch(la, pa, d.x, **d.per), "phonon", la, pa)
        _check(step(topo, lat, p, d.x, **d.per), want, step, model, i)
        assert torch.equal(topo.stale, eager_topo.stale) and _flag(topo) == (1 if i >= 4 else 0), i
    assert step.captures == 1 and step.replays == 6


def test_inference_and_dropout_replays_of_a_masked_topology():
    d = _Phonon()
    model = _phonon_model()
    model.eval()
    topo = _masked(d)
    geoms = _crossing_geometries(d, topo, 3, 240)
    step = GraphedStep(model, "phonon", train=False, structure=True)
    for i, (lat, p) in enumerate(geoms):
        with torch.no_grad():
            want = model(topo.batch(lat, p, d.x, **d.per))
        got = step(topo, lat, p, d.x, **d.per)
        assert all(torch.equal(u, v) for u, v in zip(got, want)), i
    assert step.captures == 1 and _flag(topo) == 0
    model = _phonon_model(p=0.1)
    eager_topo, topo = _masked(d), _masked(d)
    step = GraphedStep(model, "phonon", structure=True)
    for i, (lat, p) in enumerate(geoms):
        torch.manual_seed(250 + i)
        la, pa = _leaves(lat, p)
        want = _step(model, eager_topo.batch(la, pa, d.x, **d.per), "phonon", la, pa)
        torch.manual_seed(250 + i)
        _check(step(topo, lat, p, d.x, **d.per), want, step, model, ("dropout", i))
    assert step.captures == 1 and _flag(topo) == 0
