"""Structure steps without a GPU: the C ABI of the fixed-topology geometry kernels (include/dost.h, ctypes, exports), and
the arithmetic contract they follow, restated per entry in numpy on a fixed (src, dst, shift) list, against the edge vectors
and distances of oracle/neighbors_oracle.py bit for bit."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from dostransformer_b200 import _lib as L
from oracle import neighbors_oracle as NO

DECLS = {
    "dost_edge_geometry": "const double* lattice, const double* pos, const int64_t* crystal_of, const int64_t* src, "
                          "const int64_t* dst, const int64_t* shift, long long n, double pad, double* edge_vec, "
                          "double* edge_len, dost_stream_t stream",
    "dost_edge_geometry_bwd": "const double* d_vec, const double* d_len, const double* edge_vec, const double* edge_len, "
                              "const int64_t* src, const int64_t* dst, const int64_t* shift, long long n, int with_lattice, "
                              "double* g, dost_stream_t stream",
}
CTYPE = {"int": C.c_int, "long long": C.c_longlong, "double": C.c_double}


def test_header_ctypes_and_exports_of_the_edge_geometry_agree():
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


def test_edge_geometry_kernels_reject_bad_arguments_without_a_launch():
    lib = L.load()
    assert lib.dost_edge_geometry(None, None, None, None, None, None, 1, 9.0, None, None, None) != 0
    assert b"edge_geometry" in lib.dost_last_error()
    assert lib.dost_edge_geometry_bwd(None, None, None, None, None, None, None, 1, 0, None, None) != 0
    assert b"edge_geometry_bwd" in lib.dost_last_error()
    assert lib.dost_edge_geometry(None, None, None, None, None, None, 0, 9.0, None, None, None) == 0      # nothing to do


def contract_geometry(lattice, pos, crystal_of, src, dst, shift, pad):
    """dost_edge_geometry in numpy: per entry v = (pos[dst] - pos[src]) + s, s_c = (Sx L0c + Sy L1c) + Sz L2c,
    d = sqrt((vx^2 + vy^2) + vz^2), each operation rounded on its own (numpy does not fuse); dst < 0: v = 0, d = pad."""
    ok = dst >= 0
    j = np.where(ok, dst, 0)
    Lc = lattice[crystal_of[src]]                                                    # [n,3,3]
    S = shift.astype(np.float64)
    s = (S[:, 0:1] * Lc[:, 0] + S[:, 1:2] * Lc[:, 1]) + S[:, 2:3] * Lc[:, 2]
    v = (pos[j] - pos[src]) + s
    d = np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])
    return np.where(ok[:, None], v, 0.0), np.where(ok, d, pad)


@pytest.mark.parametrize("self_interaction,cutoff", [(True, 4.0), (False, 8.0)])
def test_contract_restatement_reproduces_the_oracle_list_bit_for_bit(self_interaction, cutoff):
    rng = np.random.default_rng(11)
    cells = [NO.random_crystal(rng, n, 3.0, 6.0) for n in (1, 4, 2, 6)] + [(np.eye(3) * 9.5, rng.uniform(0, 9.5, (3, 3)))]
    lattice = np.stack([c[0] for c in cells])
    pos = np.concatenate([c[1] for c in cells])
    src, dst, shift, vec, dist, cry, off = [], [], [], [], [], [], 0
    for c, (Lc, pc) in enumerate(cells):
        nl = NO.neighbor_list(Lc, pc, cutoff, self_interaction=self_interaction)
        src.append(nl["src"] + off)
        dst.append(nl["dst"] + off)
        shift.append(nl["shift"])
        vec.append(nl["vec"])
        dist.append(nl["dist"])
        cry.append(np.full(len(pc), c, dtype=np.int64))
        off += len(pc)
    src, dst, shift = np.concatenate(src), np.concatenate(dst), np.concatenate(shift)
    v, d = contract_geometry(lattice, pos, np.concatenate(cry), src, dst, shift, cutoff + 1.0)
    assert v.tobytes() == np.concatenate(vec).tobytes() and d.tobytes() == np.concatenate(dist).tobytes()
    if self_interaction:
        identity = (src == dst) & (shift == 0).all(axis=1)
        assert identity.any() and (v[identity] == 0).all()
    # padded slots: the pad distance and a zero vector, whatever the geometry
    pv, pd = contract_geometry(lattice, pos, np.concatenate(cry), src[:3], np.full(3, -1), shift[:3], cutoff + 1.0)
    assert (pv == 0).all() and (pd == cutoff + 1.0).all()
