"""CPU tests: the oracle restatement against the golden vectors produced by the reference's own code,
against the live reference when /root/reference is present, and self-consistency of the restated
third-party primitives (SURVEY.md section 8c)."""
import math

import pytest
import torch

from conftest import load_golden, relerr
from dostransformer_b200.synthetic import CrystalBatch, make_edos_batch, make_phonon_batch
from oracle import dost_oracle as O
from oracle import reference_loader, shims


def _batch_from(fx):
    return CrystalBatch(**fx["batch"])


def test_oracle_matches_golden_edos_small():
    fx = load_golden("edos_small.pt")
    g = _batch_from(fx)
    outs, loss, grads = O.run_train_step(O.edos_forward, O.edos_loss, fx["state_dict"], g, g.y_ft)
    assert relerr(outs[0], fx["dos_global"]) < 2e-6
    assert relerr(outs[2], fx["dos_system"]) < 2e-6
    assert relerr(outs[1], fx["x"]) < 2e-6
    assert abs(loss.item() - fx["loss"].item()) < 1e-6
    assert set(grads) == set(fx["grads64"])
    for k, ref64 in fx["grads64"].items():
        tol = max(1e-4, 3 * fx["grads_noise"][k][0])        # relerr(the reference's fp32 gradient, ref64)
        assert relerr(grads[k], ref64) < tol, k


def test_oracle_fp64_matches_golden_arbiter():
    fx = load_golden("edos_small.pt")
    g = _batch_from(fx)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in fx["state_dict"].items()}
    g64 = g.clone()
    for k in g64.keys():
        v = getattr(g64, k)
        if torch.is_tensor(v) and v.is_floating_point():
            setattr(g64, k, v.double())
    outs, loss, grads = O.run_train_step(O.edos_forward, O.edos_loss, p64, g64, g64.y_ft)
    assert relerr(outs[0], fx["dos_global64"]) < 1e-12
    assert relerr(outs[2], fx["dos_system64"]) < 1e-12
    for k, ref in fx["grads64"].items():
        assert relerr(grads[k], ref) < 1e-9, k


def test_oracle_matches_golden_phonon_small():
    fx = load_golden("phonon_small.pt")
    g = _batch_from(fx)
    outs, loss, grads = O.run_train_step(O.phonon_forward, O.phonon_loss, fx["state_dict"], g, g.phdos)
    assert relerr(outs[0], fx["dos_global"]) < 1e-10
    assert relerr(outs[2], fx["dos_system"]) < 1e-10
    assert abs(loss.item() - fx["loss"].item()) < 1e-10
    for k, ref in fx["grads64"].items():
        assert relerr(grads[k], ref) < 1e-7, k


def test_dead_parameters_listed():
    fx = load_golden("edos_small.pt")
    dead = fx["dead"]
    assert len(dead) == 45                     # 3 x 7 node_mlp_1 + 6 layers x 4 attention projections
    assert all(("node_mlp_1" in k) or ("self_attn" in k) for k in dead)
    fxp = load_golden("phonon_small.pt")
    assert len(fxp["dead"]) == 46 and "alpha" in fxp["dead"]


@pytest.mark.skipif(not reference_loader.available(),
                    reason="the original project's model code is not available (DOST_REFERENCE_ROOT or oracle/_ref/)")
def test_oracle_matches_live_reference():
    EDOS, PHONON, _ = reference_loader.load()
    torch.manual_seed(5)
    m = EDOS(2, 2, 200, 41, 2, 64, torch.device("cpu"), 0.0)
    g = make_edos_batch(6, seed=77, mean_atoms=8.0, max_atoms=30)
    dg, x, ds = m(g)
    dg2, x2, ds2 = O.edos_forward(O.state_dict_of(m), g)
    assert relerr(dg2, dg) < 2e-6 and relerr(ds2, ds) < 2e-6 and relerr(x2, x) < 2e-6
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(6)
    mp = PHONON(3, 2, 118, 4, 32, torch.device("cpu"), 0.0)
    gp = make_phonon_batch(4, seed=78)
    dg, x, ds = mp(gp)
    dg2, x2, ds2 = O.phonon_forward(O.state_dict_of(mp), gp)
    assert relerr(dg2, dg) < 1e-12 and relerr(ds2, ds) < 1e-12


def test_phantom_key_identity():
    """SURVEY 0.1-4: zero-padded rows become LN.bias keys; the packed restatement with (Nmax-n) analytic phantom
    keys equals the padded attention."""
    torch.manual_seed(0)
    H, T = 32, 9
    n = [3, 7, 1]
    nmax = max(n)
    gamma, beta = torch.randn(H, dtype=torch.float64), torch.randn(H, dtype=torch.float64)
    q = torch.randn(len(n), T, H, dtype=torch.float64)
    xs = [torch.randn(k, H, dtype=torch.float64) for k in n]
    dense = torch.zeros(len(n), nmax, H, dtype=torch.float64)
    for i, x in enumerate(xs):
        dense[i, : n[i]] = x
    ln = lambda t: torch.nn.functional.layer_norm(t, (H,), gamma, beta, 1e-5)
    assert torch.equal(ln(torch.zeros(1, H, dtype=torch.float64))[0], beta)       # LN(0) == bias exactly
    ref = O.attention(q, ln(dense))
    for i, x in enumerate(xs):
        k = ln(x)
        s = (q[i] @ k.T) * H ** -0.5
        sb = (q[i] @ beta) * H ** -0.5
        c = nmax - n[i]
        m = torch.maximum(s.max(dim=1).values, sb)
        e = torch.exp(s - m[:, None])
        eb = c * torch.exp(sb - m)
        out = (e @ k + eb[:, None] * beta[None]) / (e.sum(1) + eb)[:, None]
        assert relerr(out, ref[i]) < 1e-6      # fp32 softmax inside O.attention


def test_scatter_restatements_against_dense():
    torch.manual_seed(1)
    E, N, W = 57, 9, 5
    src = torch.randn(E, W, dtype=torch.float64)
    idx = torch.randint(0, N - 2, (E,))             # leaves empty destinations
    onehot = torch.zeros(N, E, dtype=torch.float64)
    onehot[idx, torch.arange(E)] = 1
    assert relerr(O.segment_sum(src, idx, N), onehot @ src) < 1e-13
    cnt = onehot.sum(1).clamp(min=1)
    assert relerr(O.segment_mean(src, idx, N), (onehot @ src) / cnt[:, None]) < 1e-13
    assert relerr(shims.scatter_mean(src, idx, dim=0, dim_size=N), O.segment_mean(src, idx, N)) < 1e-15
    rowptr, perm = O.csr_by_key(idx, N)
    for s in range(N):
        seg = perm[rowptr[s]:rowptr[s + 1]]
        assert torch.equal(seg, torch.nonzero(idx == s).squeeze(1))


def test_to_dense_batch_restatement():
    batch = torch.tensor([0, 0, 0, 1, 2, 2])
    x = torch.arange(12.0).view(6, 2)
    dense, n, nmax = O.pad_crystals(x, batch)
    d2, mask = shims.to_dense_batch(x, batch)
    assert torch.equal(dense, d2) and nmax == 3 and mask.sum() == 6
    assert torch.equal(dense[1, 1:], torch.zeros(2, 2))


def test_phonon_edge_features_restatement():
    v = torch.tensor([[0.0, 0.0, 0.0], [1.0, 2.0, 2.0], [0.0, 0.0, 3.9], [5.0, 0.0, 0.0]], dtype=torch.float64)
    ref = shims.smooth_cutoff(v.norm(dim=1) / 4.0)[:, None] * shims.spherical_harmonics(
        shims._Irreps(1), v, True, normalization="component")
    out = O.phonon_edge_features(v)
    assert relerr(out, ref) < 1e-14
    assert torch.allclose(out[0], torch.tensor([1.0, 0, 0, 0], dtype=torch.float64))   # self-interaction edge
    assert out[3].abs().max() == 0                                                     # beyond the cutoff
    assert abs(out[1, 1:].norm().item() - out[1, 0].item() * math.sqrt(3)) < 1e-12


def test_losses():
    torch.manual_seed(2)
    B, T = 4, 11
    pg, ps = torch.rand(B, T), torch.rand(B, T)
    y = torch.rand(B * T) - 0.2
    yy = y.clamp(min=0).view(B, T)
    ref = ((yy - pg) ** 2).mean(1).sqrt().mean() + 0.5 * ((yy - ps) ** 2).mean(1).sqrt().mean()
    assert abs(O.edos_loss(pg, ps, y, 0.5) - ref) < 1e-7
    ph = torch.rand(B, T)
    ref = ((ph - pg) ** 2).mean().sqrt() + ((ph - ps) ** 2).mean().sqrt()
    assert abs(O.phonon_loss(pg, ps, ph, 1.0) - ref) < 1e-7


# ---------------------------------------------------------------------------------------------- graph construction oracle
def test_neighbor_oracle_known_lattices():
    """The brute-force neighbour oracle on lattices with textbook answers (the reference has no fixtures for its
    third-party neighbour finders: parity unpinned, see oracle/neighbors_oracle.py)."""
    import numpy as np
    from oracle import neighbors_oracle as NO
    # simple cubic, a = 3: 6 first neighbours at 3, 12 second at 3*sqrt(2); with self-interaction also the atom itself
    L = np.eye(3) * 3.0
    pos = np.zeros((1, 3))
    nl = NO.neighbor_list(L, pos, 3.5, self_interaction=True)
    assert len(nl["dist"]) == 7 and np.count_nonzero(nl["dist"] == 0.0) == 1 and np.count_nonzero(nl["dist"] == 3.0) == 6
    assert (nl["shift"][nl["dist"] == 0.0] == 0).all()
    nl = NO.neighbor_list(L, pos, 4.5, self_interaction=False)
    assert len(nl["dist"]) == 18 and np.allclose(np.sort(nl["dist"])[6:], 3.0 * np.sqrt(2.0))
    # canonical order: shifts ascend lexicographically for the single (i, j) pair
    key = nl["shift"][:, 0] * 100 + nl["shift"][:, 1] * 10 + nl["shift"][:, 2]
    assert (np.diff(key) > 0).all()
    assert np.array_equal(nl["vec"], nl["shift"].astype(np.float64) * 3.0)
    # fcc (conventional cell, 4 atoms, a = 4): 12 nearest neighbours at a / sqrt(2) for every atom
    Lf = np.eye(3) * 4.0
    pf = np.array([[0, 0, 0], [0, 2, 2], [2, 0, 2], [2, 2, 0]], dtype=np.float64)
    bonds, feats = NO.edos_edges(Lf, pf, radius=8.0, k=12)
    assert bonds.shape == (48, 2) and feats.shape == (48, 41) and feats.dtype == np.float32
    nlf = NO.neighbor_list(Lf, pf, 8.0, self_interaction=False)
    idx, dist = NO.knn_from_list(nlf, 4, 12, 8.0)
    assert np.allclose(dist, 4.0 / np.sqrt(2.0)) and (bonds[:, 0] == np.repeat(np.arange(4), 12)).all()
    # the Gaussian filter peaks at the centre closest to the distance (2.828 -> centre 14 = 2.8)
    assert (feats.argmax(axis=1) == 14).all()
    # a sparse cell: fewer than 12 images within the radius -> padded with index 0 / distance radius + 1
    Ls = np.eye(3) * 7.5
    bonds, feats = NO.edos_edges(Ls, np.array([[0.0, 0.0, 0.0], [3.0, 0.0, 0.0]]), radius=8.0, k=12)
    nls = NO.neighbor_list(Ls, np.array([[0.0, 0.0, 0.0], [3.0, 0.0, 0.0]]), 8.0, self_interaction=False)
    per_atom = np.bincount(nls["src"], minlength=2)
    assert (per_atom < 12).all()
    idx, dist = NO.knn_from_list(nls, 2, 12, 8.0)
    assert (dist[0, per_atom[0]:] == 9.0).all() and (idx[0, per_atom[0]:] == 0).all() and (np.diff(dist, axis=1) >= 0).all()
