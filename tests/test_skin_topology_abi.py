"""Skin topologies without a GPU: the C ABI of the re-pick and check kernels (include/dost.h, ctypes, exports), and numpy
restatements of what they compute, on the brute-force lists of oracle/neighbors_oracle.py:

* the re-pick: the candidate list at radius + skin, its distances recomputed at the new geometry by the arithmetic
  contract, filtered at radius, then ``knn_from_list``, is ``edos_edges`` at the new geometry bit for bit;
* the completeness test: whenever it passes, every pair within the cutoff at the new geometry is a candidate."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from dostransformer_b200 import _lib as L
from oracle import neighbors_oracle as NO
from test_structure_step_abi import contract_geometry

DECLS = {
    "dost_knn_reselect": "const double* lattice, const double* pos, const int64_t* node_ptr, const int64_t* crystal_of, "
                         "const int32_t* cand_ptr, const int64_t* cand_dst, const int64_t* cand_shift, long long N, int k, "
                         "double cutoff, double pad_dist, double* cand_len, double* cand_vec, int64_t* out_pick, "
                         "double* out_dist, int64_t* out_nbr, int64_t* out_shift, int64_t* out_edge_index, "
                         "dost_stream_t stream",
    "dost_topology_check": "const double* lattice, const double* pos, const double* lattice0, const double* pos0, "
                           "const int64_t* node_ptr, long long C, double cutoff, double skin, const int64_t* crystal_of, "
                           "const int64_t* cand_src, const int64_t* cand_dst, const int64_t* cand_shift, "
                           "const uint8_t* cand_held, long long n_cand, int32_t* flag, dost_stream_t stream",
}
CTYPE = {"int": C.c_int, "long long": C.c_longlong, "double": C.c_double}
SLACK = 1e-9            # the relative slack of dost_topology_check


def test_header_ctypes_and_exports_of_the_skin_kernels_agree():
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


def test_skin_kernels_reject_bad_arguments_without_a_launch():
    lib = L.load()
    nul = [None] * 7
    assert lib.dost_knn_reselect(*nul, 1, 12, 8.0, 9.0, *([None] * 8)) != 0
    assert b"knn_reselect" in lib.dost_last_error()
    assert lib.dost_knn_reselect(*nul, 0, 12, 8.0, 9.0, *([None] * 8)) == 0              # nothing to do
    assert lib.dost_topology_check(*([None] * 5), 1, 4.0, 0.5, *([None] * 5), 0, None, None) != 0
    assert b"topology_check" in lib.dost_last_error()
    assert lib.dost_topology_check(*([None] * 5), 0, 4.0, 0.5, *([None] * 5), 0, None, None) == 0


# ------------------------------------------------------------------ numpy restatements
def skin_bound(L0, p0, L1, p1, cutoff):
    """(eps, delta, bound) of dost_topology_check for one crystal: eps = ||L0^-1 (L - L0)||_F, delta = max_i |(f_i - f0_i) L|
    with f = p L^-1, and the radius (cutoff + 2 delta) / (1 - eps) within which every pair now within the cutoff was at
    the build (inf for eps >= 1)."""
    eps = np.linalg.norm(np.linalg.inv(L0) @ (L1 - L0))
    df = p1 @ np.linalg.inv(L1) - p0 @ np.linalg.inv(L0)
    delta = np.linalg.norm(df @ L1, axis=1).max() if len(p1) else 0.0
    return eps, delta, ((cutoff + 2.0 * delta) / (1.0 - eps) if eps < 1.0 else np.inf)


def skin_complete(L0, p0, L1, p1, cutoff, skin):
    """True when dost_topology_check leaves the flag clear for this crystal (without the phonon crossing test)."""
    eps, _, bound = skin_bound(L0, p0, L1, p1, cutoff)
    return bool(eps < 1.0 and bound * (1.0 + SLACK) < cutoff + skin)


def candidates(L0, p0, cutoff, skin, self_interaction):
    return NO.neighbor_list(L0, p0, cutoff + skin, self_interaction=self_interaction)


def repick(cand, L1, p1, radius, k):
    """dost_knn_reselect for one crystal: the candidates' distances at (L1, p1) by the contract, filtered at d < radius,
    then the stable k nearest (knn_from_list).  Returns (idx [n,k], dist [n,k], pick [n,k] candidate ids, -1 padded)."""
    n = len(p1)
    _, d = contract_geometry(L1[None], p1, np.zeros(n, dtype=np.int64), cand["src"], cand["dst"], cand["shift"], 0.0)
    keep = np.nonzero(d < radius)[0]
    nl = {"src": cand["src"][keep], "dst": cand["dst"][keep], "dist": d[keep]}
    idx, dist = NO.knn_from_list(nl, n, k, radius)
    pick = np.full((n, k), -1, dtype=np.int64)
    for i in range(n):
        m = np.nonzero(nl["src"] == i)[0]
        order = np.argsort(nl["dist"][m], kind="stable")[:k]
        pick[i, :len(order)] = keep[m][order]
    return idx, dist, pick


def move(rng, L0, p0, dl, dp):
    return L0 + dl * rng.standard_normal((3, 3)), p0 + dp * rng.standard_normal(p0.shape)


def pair_keys(nl):
    return {(int(i), int(j), *map(int, s)) for i, j, s in zip(nl["src"], nl["dst"], nl["shift"])}


@pytest.mark.parametrize("seed", range(4))
def test_repick_from_the_candidates_is_the_fresh_edos_list(seed):
    rng = np.random.default_rng(100 + seed)
    radius, k, skin = 8.0, 12, 2.0
    L0, p0 = NO.random_crystal(rng, int(rng.integers(1, 9)), 3.0, 6.0)
    cand = candidates(L0, p0, radius, skin, False)
    changed = 0
    for t in range(6):
        L1, p1 = move(rng, L0, p0, 0.004 * t, 0.04 * t)
        assert skin_complete(L0, p0, L1, p1, radius, skin), t
        idx, dist, pick = repick(cand, L1, p1, radius, k)
        bonds, feats = NO.edos_edges(L1, p1, radius, k)
        assert np.array_equal(bonds[:, 1], idx.reshape(-1)) and np.array_equal(bonds[:, 0], np.repeat(np.arange(len(p1)), k))
        assert NO.gaussian_expand(dist).reshape(-1, 41).tobytes() == feats.tobytes()
        fresh = NO.neighbor_list(L1, p1, radius, self_interaction=False)
        assert np.array_equal(NO.knn_from_list(fresh, len(p1), k, radius)[1], dist)
        # each candidate is picked at most once (the backward's plain stores rely on it)
        assert len(np.unique(pick[pick >= 0])) == int((pick >= 0).sum())
        changed += int(not np.array_equal(pick, repick(cand, L0, p0, radius, k)[2]))
    assert changed > 0                                    # the moves do change which neighbours are picked


@pytest.mark.parametrize("seed", range(6))
def test_completeness_test_implies_the_fresh_list_is_among_the_candidates(seed):
    rng = np.random.default_rng(200 + seed)
    passed = failed = 0
    for _ in range(12):
        n = int(rng.integers(1, 6))
        L0, p0 = NO.random_crystal(rng, n, 3.0, 6.0)
        cutoff, skin = float(rng.choice([4.0, 8.0])), float(rng.uniform(0.0, 1.5))
        si = bool(rng.integers(0, 2))
        cand = pair_keys(candidates(L0, p0, cutoff, skin, si))
        for scale in (0.0, 0.02, 0.1, 0.4):
            L1, p1 = move(rng, L0, p0, 0.2 * scale, scale)
            if skin_complete(L0, p0, L1, p1, cutoff, skin):
                passed += 1
                assert pair_keys(NO.neighbor_list(L1, p1, cutoff, self_interaction=si)) <= cand
            else:
                failed += 1
    assert passed > 0 and failed > 0


def test_bound_is_tight_for_a_pure_strain_and_a_rigid_translation():
    L0 = np.diag([5.0, 6.0, 7.0])
    p0 = np.array([[0.5, 0.5, 0.5], [2.0, 3.0, 1.0]])
    eps, delta, _ = skin_bound(L0, p0, 1.01 * L0, 1.01 * p0, 4.0)        # homogeneous strain: no fractional move
    assert abs(eps - 0.01 * np.sqrt(3)) < 1e-12 and delta < 1e-12
    eps, delta, _ = skin_bound(L0, p0, L0, p0 + 0.3, 4.0)                 # rigid translation by (0.3, 0.3, 0.3)
    assert eps == 0.0 and abs(delta - 0.3 * np.sqrt(3)) < 1e-12
    assert not skin_complete(L0, p0, L0, p0 + 0.3, 4.0, 2 * 0.3 * np.sqrt(3))   # at the bound: flagged (conservative)
