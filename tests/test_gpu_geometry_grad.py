"""GPU tests of the geometry gradients: the two backward kernels against fp64 torch autograd, the pos / lattice reduction,
both models end to end against the fp64 oracle chain (tests/test_geometry_grad_abi.py, pinned there by finite
differences), finite differences of the models' own losses, and the guarantee that nothing changes when no input asks
for a gradient."""
import math

import numpy as np
import pytest
import torch

from conftest import relerr
from dostransformer_b200 import _lib as L
from dostransformer_b200 import neighbors as NB
from dostransformer_b200 import ops
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
from dostransformer_b200.synthetic import CrystalBatch
from oracle import dost_oracle as O
from oracle import neighbors_oracle as NO
from test_geometry_grad_abi import knn_edges, oracle_edge_vec, oracle_gaussian, oracle_nbr_dist, oracle_topology

pytestmark = pytest.mark.gpu
DEV = "cuda"
EPS = {torch.float32: 2.0 ** -24, torch.float64: 2.0 ** -53}
GRAD_FLOOR = {"fp32": (1e-4, 3e-4), "bf16x3": (2e-3, 1e-2)}       # test_gpu_model.py: (relative L2, max-norm)
PHONON_FLOOR = (1e-4, 3e-4)                                        # test_phonon_small_golden_fp64: fp32 softmax in fp64


def _rel_l2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _grade(name, got, ref, floor, noise=(0.0, 0.0)):
    e_l2, e_inf = _rel_l2(got, ref), relerr(got, ref)
    assert e_l2 < max(floor[0], 3 * noise[0]) and e_inf < max(floor[1], 3 * noise[1]), (name, e_l2, e_inf, noise)


def _cells(seed, sizes, a_lo=3.0, a_hi=5.5):
    rng = np.random.default_rng(seed)
    cells = [NO.random_crystal(rng, n, a_lo, a_hi) for n in sizes]
    lattice = torch.tensor(np.stack([c[0] for c in cells]), dtype=torch.float64, device=DEV)
    pos = torch.tensor(np.concatenate([c[1] for c in cells]), dtype=torch.float64, device=DEV)
    node_ptr = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int64, device=DEV)
    return cells, lattice, pos, node_ptr


# ------------------------------------------------------------------ 1. kernel level
def _features_grad_ref(v, W, dv):
    """fp64 autograd of features -> Linear (no bias: it does not enter d_edge_vec) with dv at the pre-activation."""
    v = v.detach().double().cpu().requires_grad_()
    (O.phonon_edge_features(v) @ W.double().cpu().T * dv.double().cpu()).sum().backward()
    return v.grad


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("H", [48, 256])
def test_phonon_edge_encode_bwd_kernel(dtype, H):
    gen = torch.Generator().manual_seed(H)
    special = torch.tensor([[0.0, 0.0, 0.0], [1e-13, 0.0, 0.0], [0.0, -1e-13, 0.0], [0.3, -1.1, 0.5], [2.0, 0.0, 0.0],
                            [0.0, 0.0, -2.0], [1.2, 2.1, -1.9], [2.5, 1.0, 0.0], [4.0, 0.0, 0.0], [0.0, -4.0, 0.0],
                            [3.0, 3.0, 3.0], [0.0, 0.0, 7.5]], dtype=torch.float64)
    rnd = torch.randn(300, 3, generator=gen, dtype=torch.float64)
    rnd = rnd / rnd.norm(dim=1, keepdim=True) * (5.0 * torch.rand(300, 1, generator=gen, dtype=torch.float64))
    v = torch.cat([special, rnd]).to(dtype)
    E = v.shape[0]
    W = torch.randn(H, 4, generator=gen, dtype=torch.float64).to(dtype)
    dv = torch.randn(E, H, generator=gen, dtype=torch.float64).to(dtype)
    vd, Wd, dvd = v.to(DEV), W.to(DEV), dv.to(DEV)
    runs = []
    for _ in range(2):
        out = torch.empty(E, 3, dtype=dtype, device=DEV)
        L.check(L.lib().dost_phonon_edge_encode_bwd(L.dt(vd), L.p(vd), E, L.p(Wd), L.p(dvd), H, L.p(out), L.stream()))
        runs.append(out.cpu())
    assert torch.equal(runs[0], runs[1])                                  # bitwise reproducible
    ref = _features_grad_ref(v, W, dv)
    # per row: |got - ref| <= 64 eps B_e with B_e = (sqrt3 / max(|v|, 1e-12) + pi/4 (1 + sqrt3)) sum_c |dv_c| max_k |W_ck|,
    # the size of J^T g; 64 eps covers the H/32-term lane sums, the 5-level butterfly and the ~10 rounded ops of J (and, in
    # fp32, the fp32 value of the clamp 1e-12 and of pi, each within 1 ulp)
    ln = v.double().norm(dim=1)
    B = (math.sqrt(3) / ln.clamp_min(1e-12) + math.pi / 4 * (1 + math.sqrt(3))) * (dv.double().abs() @ W.double().abs().amax(1))
    err = (runs[0].double() - ref).abs().amax(1)
    assert bool((err <= 64 * EPS[dtype] * B).all()), (err / B).max().item()
    # the self-interaction zero vector: sqrt(3) * 1e12 * (dv . W[:, 1:4]), what the reference produces
    want0 = math.sqrt(3) / 1e-12 * (dv[0].double() @ W[:, 1:].double())
    assert float((runs[0][0].double() - want0).abs().max()) <= 64 * EPS[dtype] * float(B[0])


def test_phonon_edge_encode_autograd_fp64():
    """The autograd node: edge_vec, weight, bias and slope gradients against torch autograd of features -> Linear ->
    PReLU, fp64 (gates are taken from the same fp64 pre-activation, so no gate flips)."""
    gen = torch.Generator().manual_seed(1)
    E, H = 700, 64
    v = torch.randn(E, 3, generator=gen, dtype=torch.float64) * 1.8
    v[::25] = 0.0                                                         # self-interaction rows
    W = torch.randn(H, 4, generator=gen, dtype=torch.float64)
    b = torch.randn(H, generator=gen, dtype=torch.float64)
    a = torch.tensor([0.25], dtype=torch.float64)
    d_out = torch.randn(E, H, generator=gen, dtype=torch.float64)
    leaves = [t.to(DEV).requires_grad_() for t in (v, W, b, a)]
    (ops.phonon_edge_encode(*leaves) * d_out.to(DEV)).sum().backward()
    refs = [t.clone().requires_grad_() for t in (v, W, b, a)]
    (torch.nn.functional.prelu(O.phonon_edge_features(refs[0]) @ refs[1].T + refs[2], refs[3]) * d_out).sum().backward()
    for name, got, ref in zip(("edge_vec", "weight", "bias", "slope"), leaves, refs):
        keep = slice(None) if name != "edge_vec" else (v.norm(dim=1) > 0)
        # fp64 sums of up to n = E H = 4.5e4 terms in another order: ~ sqrt(n) eps sum|t| ~ n eps |max| = 5e-12 -> 1e-10
        assert relerr(got.grad.cpu()[keep], ref.grad[keep]) < 1e-10, name
    selfs = v.norm(dim=1) == 0
    assert relerr(leaves[0].grad.cpu()[selfs], refs[0].grad[selfs]) < 1e-10


def test_gaussian_expand_bwd_kernel():
    gen = torch.Generator().manual_seed(2)
    d = torch.cat([torch.tensor([0.0, 0.2, 4.0, 8.0, 9.0, 1e-9]), 9.0 * torch.rand(2000, generator=gen, dtype=torch.float64)])
    d_out = torch.randn(d.numel(), 41, generator=gen).float()
    dd, gd = d.to(DEV), d_out.to(DEV)
    runs = []
    for _ in range(2):
        out = torch.empty(d.numel(), dtype=torch.float64, device=DEV)
        L.check(L.lib().dost_gaussian_expand_bwd(L.p(gd), L.p(dd), d.numel(), 0.0, 0.2, 41, 0.2, L.p(out), L.stream()))
        runs.append(out.cpu())
    assert torch.equal(runs[0], runs[1])
    x = d.clone().requires_grad_()
    phi = oracle_gaussian(x)
    (phi * d_out.double()).sum().backward()
    # per element: a 41-term fp64 sum of terms each ~8 rounded ops (exp within 2 ulp of libm's): <= 64 eps sum |terms|
    mu = torch.tensor(np.arange(0.0, 8.0 + 0.2, 0.2))
    terms = (d_out.double() * phi.detach() * (-2 * (d[:, None] - mu) / 0.04)).abs().sum(1)
    assert bool(((runs[0] - x.grad).abs() <= 64 * EPS[torch.float64] * terms + 1e-300).all())
    # and through the autograd node of neighbors.gaussian_expand
    xg = dd.clone().requires_grad_()
    (NB.gaussian_expand(xg, 0.0, 8.0, 0.2) * gd).sum().backward()
    assert torch.equal(xg.grad.cpu(), runs[0])


def test_pos_and_lattice_reduction():
    sizes = [1, 4, 2, 7]
    cells, lattice, pos, node_ptr = _cells(21, sizes)
    lat, p = lattice.clone().requires_grad_(), pos.clone().requires_grad_()
    nl = NB.phonon_edges(lat, p, node_ptr, 4.0)
    src, dst = nl["edge_index"]
    identity = (src == dst) & (nl["edge_shift"] == 0).all(dim=1)
    gen = torch.Generator().manual_seed(3)
    g = torch.randn(src.numel(), 3, generator=gen, dtype=torch.float64).to(DEV)
    g[identity] *= 1e12                       # what dost_phonon_edge_encode_bwd gives the self-interaction rows

    def grads(dvec):
        lat.grad = p.grad = None
        torch.autograd.backward(nl["edge_vec"], dvec, retain_graph=True)
        return p.grad.clone(), lat.grad.clone()

    d_pos, d_lat = grads(g)
    again = grads(g)
    assert torch.equal(d_pos, again[0]) and torch.equal(d_lat, again[1])          # bitwise reproducible
    no_id = grads(g.masked_fill(identity[:, None], 0.0))
    assert torch.equal(d_pos, no_id[0]) and torch.equal(d_lat, no_id[1])         # identity edges contribute exactly 0
    topo = oracle_topology(cells, 4.0, True)
    assert torch.equal(topo["src"], src.cpu()) and torch.equal(topo["dst"], dst.cpu())
    rl, rp = lattice.detach().cpu().clone().requires_grad_(), pos.detach().cpu().clone().requires_grad_()
    oracle_edge_vec(rl, rp, topo).backward(g.cpu())
    # per entry: an fp64 sum of <= deg terms in another order, deg <= 256: 256 eps times the sum of |terms|
    ga = g.cpu().masked_fill(identity.cpu()[:, None], 0.0).abs()
    bp = torch.zeros_like(rp).index_add_(0, topo["dst"], ga).index_add_(0, topo["src"], ga)
    bl = torch.zeros(len(sizes), 3, 3, dtype=torch.float64).index_add_(
        0, topo["crystal"], topo["shift"].abs().double()[:, :, None] * ga[:, None, :])
    assert bool(((d_pos.cpu() - rp.grad).abs() <= 256 * EPS[torch.float64] * bp).all())
    assert bool(((d_lat.cpu() - rl.grad).abs() <= 256 * EPS[torch.float64] * bl).all())
    assert bool((d_pos[node_ptr[0]:node_ptr[1]] == 0).all())                     # a 1-atom crystal: only its own images


# ------------------------------------------------------------------ 2. phonon model
def _phonon_inputs(seed, sizes):
    cells, lattice, pos, node_ptr = _cells(seed, sizes)
    gen = torch.Generator().manual_seed(seed)
    N, C = sum(sizes), len(sizes)
    x = torch.zeros(N, 118, dtype=torch.float64)
    x[torch.arange(N), torch.randint(0, 118, (N,), generator=gen)] = 1.0 + 200.0 * torch.rand(N, generator=gen,
                                                                                           dtype=torch.float64)
    system = torch.randint(0, 7, (C,), generator=gen)
    ph = torch.rand(C, 51, generator=gen, dtype=torch.float64)
    return cells, lattice, pos, node_ptr, x, system, ph / ph.amax(dim=1, keepdim=True)


def _phonon_device_step(model, lattice, pos, node_ptr, x, system, ph, want_geo=True):
    lat = lattice.clone().requires_grad_(want_geo)
    p = pos.clone().requires_grad_(want_geo)
    g = NB.phonon_graph_batch(lat, p, node_ptr, x.to(DEV), system=system.to(DEV), phdos=ph.to(DEV))
    g.x.requires_grad_(want_geo)
    if want_geo:
        g.edge_vec.retain_grad()
    model.zero_grad(set_to_none=True)
    dg, _, ds = model(g)
    loss = ops.dos_loss(dg, ds, g.phdos, mode="phonon")
    loss.backward()
    return g, lat, p, loss, dg, ds


def _phonon_oracle(sd, cells, lattice, pos, x, system, ph, sizes):
    topo = oracle_topology(cells, 4.0, True)
    rl, rp = lattice.detach().cpu().clone().requires_grad_(), pos.detach().cpu().clone().requires_grad_()
    ev = oracle_edge_vec(rl, rp, topo)
    ev.retain_grad()
    rx = x.clone().requires_grad_()
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    g = CrystalBatch(x=rx, edge_index=torch.stack([topo["src"], topo["dst"]]), edge_vec=ev, batch=batch, system=system)
    leaf = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in sd.items()}
    dg, _, ds = O.phonon_forward(leaf, g, training=True)
    O.phonon_loss(dg, ds, ph).backward()
    return topo, ev.grad, rx.grad, rp.grad, rl.grad


@pytest.mark.parametrize("H", [64, 256])
@pytest.mark.parametrize("sizes", [[1], [3, 1, 4, 2, 6], [2, 5, 1, 3, 4, 6, 2, 1, 5, 3, 2, 4, 6, 1, 3, 5, 2, 4, 3, 6, 1, 2, 5]],
                         ids=["B1", "B5", "B23"])
def test_phonon_model_geometry_gradients(H, sizes):
    torch.set_default_dtype(torch.float64)
    cells, lattice, pos, node_ptr, x, system, ph = _phonon_inputs(30 + len(sizes), sizes)
    torch.manual_seed(H)
    model = DOSTransformer_phonon(2, 1, 118, 4, H, torch.device(DEV), 0.0)
    sd = O.state_dict_of(model)
    model.to(DEV).train()
    g, lat, p, _, _, _ = _phonon_device_step(model, lattice, pos, node_ptr, x, system, ph)
    topo, r_ev, r_x, r_pos, r_lat = _phonon_oracle(sd, cells, lattice, pos, x, system, ph, sizes)
    assert torch.equal(g.edge_index.cpu(), torch.stack([topo["src"], topo["dst"]]))
    selfs = (topo["src"] == topo["dst"]) & (topo["shift"] == 0).all(dim=1)
    ev_grad = g.edge_vec.grad.cpu()
    # self-loop rows (~1e12, the clamp's 1/1e-12) and the other rows, each graded against its own norm
    _grade("edge_vec (self loops)", ev_grad[selfs], r_ev[selfs], PHONON_FLOOR)
    if bool((~selfs).any()):
        _grade("edge_vec", ev_grad[~selfs], r_ev[~selfs], PHONON_FLOOR)
    _grade("x", g.x.grad, r_x, PHONON_FLOOR)
    if len(sizes) > 1:
        _grade("pos", p.grad, r_pos, PHONON_FLOOR)
        _grade("lattice", lat.grad, r_lat, PHONON_FLOOR)
    else:      # a lone 1-atom crystal sees only its own images: its pos.grad is 0
        _grade("lattice", lat.grad, r_lat, PHONON_FLOOR)
    off = np.concatenate([[0], np.cumsum(sizes)])
    for i in [i for i, n in enumerate(sizes) if n == 1]:
        # the same edges summed in the same order as centre and as neighbour: exactly 0
        assert bool((p.grad[off[i]] == 0).all())


# ------------------------------------------------------------------ 3. eDOS model
def _edos_inputs(seed, sizes):
    cells, lattice, pos, node_ptr = _cells(seed, sizes, 3.5, 6.0)
    gen = torch.Generator().manual_seed(seed)
    C = len(sizes)
    feats = torch.randn(sum(sizes), 200, generator=gen)
    glob = torch.randn(2 * C, generator=gen)
    system = torch.randint(0, 7, (C,), generator=gen)
    y = torch.rand(C * 201, generator=gen)
    return cells, lattice, pos, node_ptr, feats, glob, system, y


def _edos_oracle(sd, cells, lattice, pos, feats, glob, system, y, sizes, dtype):
    topo = oracle_topology(cells, 8.0, False)
    picks = knn_edges(topo, 12)
    rl, rp = lattice.detach().cpu().clone().requires_grad_(), pos.detach().cpu().clone().requires_grad_()
    ea = oracle_gaussian(oracle_nbr_dist(oracle_edge_vec(rl, rp, topo), picks, 8.0)).reshape(-1, 41).to(dtype)
    ea.retain_grad()
    C, N = len(sizes), sum(sizes)
    cry = torch.repeat_interleave(torch.arange(C), torch.tensor(sizes))
    rows = torch.arange(N) + cry
    x = torch.zeros(N + C, 200, dtype=dtype)
    x[rows] = feats.to(dtype)
    x.requires_grad_()
    off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.tensor(sizes).cumsum(0)])
    centre = torch.arange(N).repeat_interleave(12)
    nbr = torch.where(picks >= 0, topo["dst"][picks.clamp_min(0)], off[cry][:, None]).reshape(-1)
    ei = torch.stack([centre + cry[centre], nbr + cry[nbr]])
    rg = glob.to(dtype).clone().requires_grad_()
    batch = torch.repeat_interleave(torch.arange(C), torch.tensor(sizes) + 1)
    g = CrystalBatch(x=x, edge_index=ei, edge_attr=ea, batch=batch, glob=rg, system=system)
    leaf = {k: (v.to(dtype).clone().requires_grad_() if v.is_floating_point() else v) for k, v in sd.items()}
    dg, _, ds = O.edos_forward(leaf, g, training=True)
    O.edos_loss(dg, ds, y.to(dtype)).backward()
    return ei, {"x": x.grad, "edge_attr": ea.grad, "glob": rg.grad, "pos": rp.grad, "lattice": rl.grad}


def _edos_device_step(model, lattice, pos, node_ptr, feats, glob, system, y, want_geo=True):
    lat = lattice.clone().requires_grad_(want_geo)
    p = pos.clone().requires_grad_(want_geo)
    gl = glob.to(DEV).clone().requires_grad_(want_geo)
    g = NB.edos_graph_batch(lat, p, node_ptr, feats.to(DEV), glob=gl, system=system.to(DEV), y_ft=y.to(DEV))
    g.x.requires_grad_(want_geo)
    if want_geo:
        g.edge_attr.retain_grad()
    model.zero_grad(set_to_none=True)
    dg, _, ds = model(g)
    loss = ops.dos_loss(dg, ds, g.y_ft, mode="edos")
    loss.backward()
    return g, lat, p, gl, loss, dg, ds


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_edos_model_geometry_gradients(prec):
    sizes = [3, 7, 1, 12, 5]
    cells, lattice, pos, node_ptr, feats, glob, system, y = _edos_inputs(40, sizes)
    torch.manual_seed(4)
    model = DOSTransformer(2, 1, 200, 41, 2, 128, torch.device(DEV), 0.0, precision=prec)
    sd = O.state_dict_of(model)
    model.to(DEV).train()
    g, lat, p, gl, _, _, _ = _edos_device_step(model, lattice, pos, node_ptr, feats, glob, system, y)
    ei, r64 = _edos_oracle(sd, cells, lattice, pos, feats, glob, system, y, sizes, torch.float64)
    _, r32 = _edos_oracle(sd, cells, lattice, pos, feats, glob, system, y, sizes, torch.float32)
    assert torch.equal(g.edge_index.cpu(), ei)
    got = {"x": g.x.grad, "edge_attr": g.edge_attr.grad, "glob": gl.grad, "pos": p.grad, "lattice": lat.grad}
    for k in got:
        # the floor, or 3x the reference's own fp32-vs-fp64 noise when that is larger (test_gpu_model._check_grads)
        _grade(k, got[k], r64[k], GRAD_FLOOR[prec], (_rel_l2(r32[k], r64[k]), relerr(r32[k], r64[k])))


# ------------------------------------------------------------------ 4. finite differences of the models' losses
def _fd_check(loss_at, topo_at, ad_pos, ad_lat, loss0, c_ulps, hs):
    """Central differences at the 3 position and 2 lattice coordinates of largest analytic gradient.  h is the largest of
    ``hs`` at which the topology is unchanged.  The loss carries fp32 rounding noise of at most c_ulps fp32 ulps of |loss|
    (the fp32 softmax; for the fp32 eDOS model every op), so the difference quotient is good to c_ulps 2^-24 |loss| / h,
    plus a truncation h^2/6 |L'''|: |L'''| / |L'| <~ 3 / w^2 for features of width w (1 A cutoff ramp, 0.2 A Gaussians),
    which the hs keep below 2e-3 |grad|."""
    coords = [("pos", int(i)) for i in ad_pos.abs().flatten().argsort(descending=True)[:3]]
    coords += [("lattice", int(i)) for i in ad_lat.abs().flatten().argsort(descending=True)[:2]]
    base = topo_at(None, 0, 0.0)
    for which, flat in coords:
        ad = (ad_pos if which == "pos" else ad_lat).flatten()[flat].item()
        for h in hs:
            if all(topo_at(which, flat, s * h) == base for s in (1, -1)):
                break
        else:
            pytest.fail(f"topology changes within {hs[-1]} A of {which}[{flat}]")
        fd = (loss_at(which, flat, h) - loss_at(which, flat, -h)) / (2 * h)
        tol = c_ulps * 2.0 ** -24 * abs(loss0) / h + 2e-3 * abs(ad)
        assert abs(fd - ad) <= tol, (which, flat, h, fd, ad, tol)


def _perturbed(lattice, pos, which, flat, d):
    lat, p = lattice.clone(), pos.clone()
    if which == "pos":
        p.view(-1)[flat] += d
    elif which == "lattice":
        lat.view(-1)[flat] += d
    return lat, p


def test_finite_differences_of_both_models():
    torch.set_default_dtype(torch.float64)
    sizes = [3, 2, 4]
    cells, lattice, pos, node_ptr, x, system, ph = _phonon_inputs(50, sizes)
    torch.manual_seed(5)
    model = DOSTransformer_phonon(2, 1, 118, 4, 64, torch.device(DEV), 0.0).to(DEV).train()
    _, lat, p, loss0, _, _ = _phonon_device_step(model, lattice, pos, node_ptr, x, system, ph)

    def ph_loss(which, flat, d):
        la, pp = _perturbed(lattice, pos, which, flat, d)
        with torch.no_grad():
            g = NB.phonon_graph_batch(la, pp, node_ptr, x.to(DEV), system=system.to(DEV), phdos=ph.to(DEV))
            dg, _, ds = model(g)
            return ops.dos_loss(dg, ds, g.phdos, mode="phonon").item()

    def ph_topo(which, flat, d):
        la, pp = _perturbed(lattice, pos, which, flat, d)
        nl = NB.phonon_edges(la, pp, node_ptr, 4.0)
        return (nl["edge_index"].cpu().numpy().tobytes(), nl["edge_shift"].cpu().numpy().tobytes())

    # fp64 model with the reference's fp32 softmax: <= ~64 fp32 ulps of the loss across the 3 x t_layers attentions
    _fd_check(ph_loss, ph_topo, p.grad, lat.grad, loss0.item(), 64, (1e-2, 5e-3, 2.5e-3))

    torch.set_default_dtype(torch.float32)
    sizes = [4, 6, 3]
    cells, lattice, pos, node_ptr, feats, glob, system, y = _edos_inputs(51, sizes)
    torch.manual_seed(6)
    model = DOSTransformer(2, 1, 200, 41, 2, 64, torch.device(DEV), 0.0, precision="fp32").to(DEV).train()
    _, lat, p, _, loss0, _, _ = _edos_device_step(model, lattice, pos, node_ptr, feats, glob, system, y)

    def ed_loss(which, flat, d):
        la, pp = _perturbed(lattice, pos, which, flat, d)
        with torch.no_grad():
            g = NB.edos_graph_batch(la, pp, node_ptr, feats.to(DEV), glob=glob.to(DEV), system=system.to(DEV),
                                    y_ft=y.to(DEV))
            dg, _, ds = model(g)
            return ops.dos_loss(dg, ds, g.y_ft, mode="edos").item()

    def ed_topo(which, flat, d):
        la, pp = _perturbed(lattice, pos, which, flat, d)
        e = NB.edos_edges(la, pp, node_ptr)
        return e["edge_index"].cpu().numpy().tobytes()

    # fp32 model: the fp32-rounded bond features and every fp32 op, <= ~1024 fp32 ulps of the loss
    _fd_check(ed_loss, ed_topo, p.grad, lat.grad, loss0.item(), 1024, (5e-3, 2.5e-3, 1.25e-3))


# ------------------------------------------------------------------ 5. nothing changes when nothing asks for it
def _param_grads(model):
    return {k: q.grad.clone() for k, q in model.named_parameters() if q.grad is not None}


def test_no_input_grad_is_bitwise_unchanged_and_launches_no_new_kernel():
    torch.set_default_dtype(torch.float64)
    sizes = [3, 1, 4]
    _, lattice, pos, node_ptr, x, system, ph = _phonon_inputs(60, sizes)
    torch.manual_seed(7)
    pm = DOSTransformer_phonon(2, 1, 118, 4, 64, torch.device(DEV), 0.0).to(DEV).train()
    torch.set_default_dtype(torch.float32)
    _, elat, epos, enode, feats, glob, esys, y = _edos_inputs(61, [3, 5, 2])
    torch.manual_seed(8)
    em = DOSTransformer(2, 1, 200, 41, 2, 128, torch.device(DEV), 0.0).to(DEV).train()

    def steps(want_geo):
        out = []
        _, _, _, loss, dg, ds = _phonon_device_step(pm, lattice, pos, node_ptr, x, system, ph, want_geo)
        out.append((loss.detach(), dg.detach(), ds.detach(), _param_grads(pm)))
        _, _, _, _, loss, dg, ds = _edos_device_step(em, elat, epos, enode, feats, glob, esys, y, want_geo)
        out.append((loss.detach(), dg.detach(), ds.detach(), _param_grads(em)))
        return out

    plain, geo = steps(False), steps(True)
    for a, b in zip(plain, geo):
        assert all(torch.equal(u, v) for u, v in zip(a[:3], b[:3]))
        assert a[3].keys() == b[3].keys() and all(torch.equal(a[3][k], b[3][k]) for k in a[3])

    new = ("phonon_edge_encode_bwd_kernel", "gaussian_expand_bwd_kernel")

    def kernels(want_geo):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            steps(want_geo)
            torch.cuda.synchronize()
        return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}

    without, with_geo = kernels(False), kernels(True)
    assert not [n for n in without if any(k in n for k in new)]
    assert all(any(k in n for n in with_geo) for k in new)                 # the profiler does see them when asked


def test_frozen_parameters_with_geometry_gradients_only():
    torch.set_default_dtype(torch.float64)
    sizes = [2, 5]
    _, lattice, pos, node_ptr, x, system, ph = _phonon_inputs(70, sizes)
    torch.manual_seed(9)
    model = DOSTransformer_phonon(2, 1, 118, 4, 64, torch.device(DEV), 0.0).to(DEV).train()
    _, lat, p, _, _, _ = _phonon_device_step(model, lattice, pos, node_ptr, x, system, ph)
    want = (p.grad.clone(), lat.grad.clone())
    model.requires_grad_(False)
    _, lat, p, _, _, _ = _phonon_device_step(model, lattice, pos, node_ptr, x, system, ph)
    assert all(q.grad is None for q in model.parameters())
    # the same kernels on the same inputs for the input gradients; only the parameter products are skipped
    assert relerr(p.grad, want[0]) < 1e-12 and relerr(lat.grad, want[1]) < 1e-12
