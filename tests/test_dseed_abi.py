"""The ``_dseed`` siblings of the seeded entry points (include/dost.h): each takes the plain entry point's arguments with
``const unsigned long long* seed_offset`` inserted right after ``seed``, in the header, in the ctypes binding and in the
library's exports.  No GPU needed."""
import os
import re

from conftest import ROOT
from dostransformer_b200 import _lib as L

SEEDED = ("dost_xattn_fwd", "dost_xattn_bwd", "dost_xattn_softmax_fwd", "dost_xattn_softmax_bwd", "dost_softmax_fwd",
          "dost_softmax_bwd", "dost_softmax_fwd_planes", "dost_softmax_bwd_planes", "dost_attn_fused_fwd")


def _declared_params():
    with open(os.path.join(ROOT, "include", "dost.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    out = {}
    for name, params in re.findall(r"\b(dost_\w+)\s*\(([^)]*)\)\s*;", text):
        out[name] = [" ".join(p.split()) for p in params.split(",")]
    return out


def test_every_seeded_entry_point_has_a_dseed_sibling_with_the_offset_after_the_seed():
    decl = _declared_params()
    assert {n for n in decl if any(p.endswith(" seed") for p in decl[n])} == set(SEEDED) | {n + "_dseed" for n in SEEDED}
    for name in SEEDED:
        plain, dseed = decl[name], decl[name + "_dseed"]
        i = plain.index("unsigned long long seed")
        assert dseed == plain[:i + 1] + ["const unsigned long long* seed_offset"] + plain[i + 1:], name
        res, args = L._SIGNATURES[name]
        res_d, args_d = L._SIGNATURES[name + "_dseed"]
        assert res_d is res and args_d == args[:i + 1] + [L.C.c_void_p] + args[i + 1:], name
        assert name + "_dseed" in L.EXPORTED_SYMBOLS


def test_library_exports_the_dseed_siblings():
    lib = L.load()
    for name in SEEDED:
        assert getattr(lib, name + "_dseed").argtypes == L._SIGNATURES[name + "_dseed"][1]
