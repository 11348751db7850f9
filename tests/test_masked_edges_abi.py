"""Masked phonon edges without a GPU: the C ABI of the masked CSR build, the masked gather and the membership kernel
(include/dost.h, ctypes, exports), and numpy restatements of what they compute:

* the masked CSR: the live entries sorted as ``csr_by_key`` sorts the filtered keys, the masked entries after rowptr[N];
* the membership: at moved geometries where the completeness test passes, the candidates within r_max + skin at the
  build, filtered by their contract length < r_max, are the oracle's phonon list there - indices, shifts and order."""
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
from test_skin_topology_abi import candidates, move, skin_complete
from test_structure_step_abi import contract_geometry

DECLS = {
    "dost_csr_build_masked": "const int32_t* key, const uint8_t* mask, long long n, long long size, int32_t* rowptr, "
                             "int32_t* perm, int32_t* maxcount, void* workspace, size_t workspace_bytes, "
                             "dost_stream_t stream",
    "dost_gather_rows_masked": "int dtype, const void* src, long long ld, const int32_t* idx, const int32_t* deg_rowptr, "
                               "const uint8_t* mask, const void* add, long long ld_add, long long R, int W, void* out, "
                               "long long ldo, dost_stream_t stream",
    "dost_edge_within": "const double* edge_len, long long n, double cutoff, uint8_t* mask, dost_stream_t stream",
}
CTYPE = {"int": C.c_int, "long long": C.c_longlong, "double": C.c_double, "size_t": C.c_size_t}


def test_header_ctypes_and_exports_of_the_masked_kernels_agree():
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


def test_masked_kernels_reject_bad_arguments_without_a_launch():
    lib = L.load()
    assert lib.dost_csr_build_masked(None, None, 4, 2, None, None, None, None, 0, None) != 0
    assert b"csr_build_masked" in lib.dost_last_error()
    assert lib.dost_gather_rows_masked(1, None, 8, None, None, None, None, 0, 3, 8, None, 8, None) != 0
    assert b"gather_rows_masked" in lib.dost_last_error()
    assert lib.dost_gather_rows_masked(1, None, 8, None, None, None, None, 0, 0, 8, None, 8, None) == 0   # nothing to do
    assert lib.dost_edge_within(None, 5, 4.0, None, None) != 0
    assert b"edge_within" in lib.dost_last_error()
    assert lib.dost_edge_within(None, 0, 4.0, None, None) == 0


# ------------------------------------------------------------------ numpy restatements
def masked_csr(key, mask, size):
    """dost_csr_build_masked in numpy: (rowptr [size+1] of the live entries, perm [n]: the live entries in (key, index)
    order, then the masked entries in index order)."""
    live = np.nonzero(mask != 0)[0]
    rowptr, perm = O.csr_by_key(torch.from_numpy(key[live].astype(np.int64)), size)
    return rowptr.numpy(), np.concatenate([live[perm.numpy()], np.nonzero(mask == 0)[0]]).astype(np.int64)


@pytest.mark.parametrize("seed", range(4))
def test_masked_csr_restatement(seed):
    rng = np.random.default_rng(300 + seed)
    size = int(rng.integers(1, 40))
    n = int(rng.integers(0, 400))
    key = rng.integers(0, size, n)
    for mask in (rng.integers(0, 2, n), np.ones(n, dtype=np.int64), np.zeros(n, dtype=np.int64)):
        rowptr, perm = masked_csr(key, mask, size)
        live = int((mask != 0).sum())
        assert rowptr[-1] == live and sorted(perm.tolist()) == list(range(n))
        assert bool((mask[perm[:live]] != 0).all()) and bool((mask[perm[live:]] == 0).all())
        assert np.array_equal(perm[live:], np.sort(perm[live:]))
        for s in range(size):           # each live segment: that key's live entries, ascending
            seg = perm[rowptr[s]:rowptr[s + 1]]
            assert np.array_equal(seg, np.nonzero((key == s) & (mask != 0))[0])
        if live == n:                   # all ones: the unmasked sort
            r0, p0 = O.csr_by_key(torch.from_numpy(key.astype(np.int64)), size)
            assert np.array_equal(rowptr, r0.numpy()) and np.array_equal(perm, p0.numpy())


def live_candidates(cand, L1, p1, r_max):
    """The masked topology's live set at (L1, p1): the candidates' contract lengths compared as the fill compares."""
    n = len(p1)
    _, d = contract_geometry(L1[None], p1, np.zeros(n, dtype=np.int64), cand["src"], cand["dst"], cand["shift"], 0.0)
    return d < r_max


@pytest.mark.parametrize("seed", range(6))
def test_live_candidates_are_the_fresh_phonon_list(seed):
    rng = np.random.default_rng(400 + seed)
    r_max, skin = 4.0, 0.5
    checked = crossed = 0
    for _ in range(8):
        L0, p0 = NO.random_crystal(rng, int(rng.integers(1, 7)), 3.0, 6.0)
        cand = candidates(L0, p0, r_max, skin, True)
        held = live_candidates(cand, L0, p0, r_max)
        for t in range(5):
            L1, p1 = move(rng, L0, p0, 0.002 * t, 0.05 * t)
            if not skin_complete(L0, p0, L1, p1, r_max, skin):
                continue
            keep = live_candidates(cand, L1, p1, r_max)
            fresh = NO.neighbor_list(L1, p1, r_max, self_interaction=True)
            assert np.array_equal(cand["src"][keep], fresh["src"]) and np.array_equal(cand["dst"][keep], fresh["dst"])
            assert np.array_equal(cand["shift"][keep], fresh["shift"])
            checked += 1
            crossed += int(not np.array_equal(keep, held))
    assert checked > 0 and crossed > 0                  # some moves do take bonds across r_max

