"""Geometry gradients without a GPU: the C ABI of the two backward kernels (include/dost.h, ctypes, exports), and the fp64
oracle chain the GPU tests grade against, pinned by central finite differences.

The oracle chain is the reference's own arithmetic on a fixed topology: the brute-force neighbour list of
oracle/neighbors_oracle.py gives (src, dst, shift) and the picked k nearest; torch forms edge_vec = pos[dst] - pos[src] +
shift @ lattice (identity edges held at their constant 0); then the phonon features (oracle.dost_oracle
phonon_edge_features) or |edge_vec| -> the fp64 Gaussian expansion (mat2graph.py:162-179) of the eDOS bonds."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from dostransformer_b200 import _lib as L
from oracle import dost_oracle as O
from oracle import neighbors_oracle as NO

DECLS = {
    "dost_phonon_edge_encode_bwd": "int dtype, const void* edge_vec, long long E, const void* weight, const void* dv, int H, "
                                   "void* d_edge_vec, dost_stream_t stream",
    "dost_gaussian_expand_bwd": "const float* d_out, const double* dist, long long n, double dmin, double step, int nfilt, "
                                "double var, double* d_dist, dost_stream_t stream",
}
CTYPE = {"int": C.c_int, "long long": C.c_longlong, "double": C.c_double}


def test_header_ctypes_and_exports_of_the_geometry_backward_agree():
    with open(os.path.join(ROOT, "include", "dost.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    lib = L.load()
    for name, params in DECLS.items():
        (got,) = re.findall(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", text)
        decl = [" ".join(p.split()) for p in got.split(",")]
        assert decl == [p.strip() for p in params.split(",")], name
        res, args = L._SIGNATURES[name]
        want = [CTYPE.get(p.rsplit(" ", 1)[0], C.c_void_p) for p in decl]
        assert res is C.c_int and args == want, name
        assert name in L.EXPORTED_SYMBOLS and getattr(lib, name).argtypes == args
    assert lib.dost_abi_version() == 15                 # additive entry points: the ABI version is unchanged


def test_geometry_backward_kernels_reject_bad_arguments_without_a_launch():
    lib = L.load()
    assert lib.dost_phonon_edge_encode_bwd(L.F64, None, 1, None, None, 64, None, None) != 0
    assert b"phonon_edge_encode_bwd" in lib.dost_last_error()
    assert lib.dost_gaussian_expand_bwd(None, None, 1, 0.0, 0.2, 41, 0.2, None, None) != 0
    assert b"gaussian_expand_bwd" in lib.dost_last_error()


# ------------------------------------------------------------------ the oracle chain (also used by the GPU tests)
def oracle_topology(cells, cutoff, self_interaction):
    """Canonical (i, j, S) list of a batch of crystals from the numpy oracle: src, dst (batch rows), shift, crystal [E]
    as int64 tensors, plus the per-crystal lists for the k-nearest picks."""
    src, dst, shf, cry, lists, off = [], [], [], [], [], 0
    for c, (Lc, pc) in enumerate(cells):
        nl = NO.neighbor_list(Lc, pc, cutoff, self_interaction=self_interaction)
        src.append(nl["src"] + off)
        dst.append(nl["dst"] + off)
        shf.append(nl["shift"])
        cry.append(np.full(len(nl["src"]), c, dtype=np.int64))
        lists.append((nl, len(pc)))
        off += len(pc)
    t = lambda xs, shape: torch.tensor(np.concatenate(xs) if xs else np.zeros(shape, dtype=np.int64))
    return {"src": t(src, (0,)), "dst": t(dst, (0,)), "shift": t(shf, (0, 3)).reshape(-1, 3), "crystal": t(cry, (0,)),
            "lists": lists}


def oracle_edge_vec(lattice, pos, topo):
    """edge_vec = pos[dst] - pos[src] + shift @ lattice[crystal] (utils.py:271-273); the identity edges (i, i, 0) are the
    constant 0 whatever the geometry."""
    src, dst, shift = topo["src"], topo["dst"], topo["shift"]
    ev = pos[dst] - pos[src] + torch.einsum("ei,eij->ej", shift.to(pos.dtype), lattice[topo["crystal"]])
    identity = (src == dst) & (shift == 0).all(dim=1)
    return torch.where(identity[:, None], torch.zeros_like(ev), ev)


def knn_edges(topo, k):
    """Edge ids (into the batch list) of the k nearest picks of every atom, -1 for padded slots (mat2graph.py:217-231:
    stable sort by distance)."""
    picks, e0 = [], 0
    for nl, n in topo["lists"]:
        for i in range(n):
            m = np.nonzero(nl["src"] == i)[0]
            order = m[np.argsort(nl["dist"][m], kind="stable")[:k]]
            row = np.full(k, -1, dtype=np.int64)
            row[:len(order)] = order + e0
            picks.append(row)
        e0 += len(nl["src"])
    return torch.tensor(np.stack(picks)) if picks else torch.zeros(0, k, dtype=torch.int64)


def oracle_nbr_dist(ev, picks, radius):
    """[N,k] distances of the picks, padded slots the constant radius + 1 (mat2graph.py:223-229)."""
    d = ev.norm(dim=1)
    safe = picks.clamp_min(0)
    return torch.where(picks >= 0, d[safe], torch.full_like(d[safe], radius + 1.0))


def oracle_gaussian(dist, radius=8.0, step=0.2):
    """GaussianDistance(0, radius, step).expand in fp64 (the fp32 cast of the reference counts as the identity)."""
    filt = torch.tensor(np.arange(0.0, radius + step, step), dtype=dist.dtype)
    return torch.exp(-(dist[..., None] - filt) ** 2 / step ** 2)


def _cells(kind, seed, sizes):
    rng = np.random.default_rng(seed)
    out = []
    for n in sizes:
        if kind == "cubic":
            Lc = np.eye(3) * 3.7
            out.append((Lc, rng.uniform(0, 1, (n, 3)) @ Lc))
        else:
            out.append(NO.random_crystal(rng, n, 3.2, 5.0))
    return out


def _same_topology(a, b):
    return all(torch.equal(a[k], b[k]) for k in ("src", "dst", "shift"))


@pytest.mark.parametrize("kind", ["cubic", "triclinic"])
@pytest.mark.parametrize("model", ["phonon", "edos"])
def test_oracle_chain_matches_central_differences(kind, model):
    # the cubic eDOS cells are dense enough that the 12 picks end below the lattice constant: the self images (6 at a, 12 at
    # a sqrt 2) are exact ties that a lattice perturbation reorders, a genuine kink of the fixed-k selection
    cells = _cells(kind, 5 if kind == "cubic" else 6, [2, 1, 3] if (kind != "cubic" or model == "phonon") else [6, 5, 7])
    cutoff, radius, k = 4.0, 8.0, 12
    self_int = model == "phonon"
    lattice = torch.tensor(np.stack([c[0] for c in cells]), dtype=torch.float64, requires_grad=True)
    pos = torch.tensor(np.concatenate([c[1] for c in cells]), dtype=torch.float64, requires_grad=True)
    topo = oracle_topology(cells, cutoff if self_int else radius, self_int)
    picks = None if self_int else knn_edges(topo, k)
    gen = torch.Generator().manual_seed(7)
    w = torch.randn((topo["src"].numel(), 4) if self_int else (pos.shape[0], k, 41), generator=gen, dtype=torch.float64)

    def loss(lat, p, topo_=topo):
        ev = oracle_edge_vec(lat, p, topo_)
        f = O.phonon_edge_features(ev) if self_int else oracle_gaussian(oracle_nbr_dist(ev, picks, radius), radius)
        return (w * f).sum()

    loss(lattice, pos).backward()
    # central differences, h = 1e-5, S = sum |w|: rounding eps S / h ~ 1e-11 S; truncation h^2/6 |f'''| <= 1e-8 S, the third
    # derivative of a 0.2 A-wide Gaussian being <= ~5e2 / A^3 (the phonon features' are O(10)); observed <= 3e-12 S
    h = 1e-5
    tol = 1e-8 * float(w.abs().sum())
    coords = [("pos", a, c) for a in (0, 2, 5) for c in range(3)] + [("lattice", b, (r, c)) for b in (0, 2) for r, c in
                                                                       ((0, 0), (1, 2), (2, 1))]
    for which, i, c in coords:
        fd = []
        for sgn in (1.0, -1.0):
            lat, p = lattice.detach().clone(), pos.detach().clone()
            if which == "pos":
                p[i, c] += sgn * h
            else:
                lat[i][c] += sgn * h
            cells_h = [(lat[b].numpy(), p[o:o + len(cc[1])].numpy())
                       for b, (cc, o) in enumerate(zip(cells, np.cumsum([0] + [len(x[1]) for x in cells])[:-1]))]
            topo_h = oracle_topology(cells_h, cutoff if self_int else radius, self_int)
            assert _same_topology(topo, topo_h), (which, i, c)        # the FD stays on the fixed topology
            if not self_int:
                assert torch.equal(knn_edges(topo_h, k), picks), (which, i, c)
            fd.append(loss(lat, p).item())
        got = (pos.grad[i, c] if which == "pos" else lattice.grad[i][c]).item()
        assert abs((fd[0] - fd[1]) / (2 * h) - got) <= tol, (which, i, c, (fd[0] - fd[1]) / (2 * h), got)
