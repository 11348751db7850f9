"""C ABI of the attention-map kernels (include/dost.h): declarations, ctypes binding and exports agree.  No GPU needed."""
import ctypes as C
import os
import re

from conftest import ROOT
from dostransformer_b200 import _lib as L

DECLS = {
    "dost_xattn_probs": "int dtype, const void* q, long long q_sstride, const void* kv, const void* phantom, const int32_t* ptr, "
                        "const int32_t* nmax, const float* lse, void* out, int cols, int S, int B, int T, int H, double scale, "
                        "double drop_p, unsigned long long mask_seed, const unsigned long long* seed_offset, dost_stream_t stream",
    "dost_attn_maps_from_planes": "const void* p_hi, const void* p_lo, long long ld_p, long long rows, int cols, int T, int B, "
                                  "const int32_t* ptr, const int32_t* nmax, float* out, double drop_p, "
                                  "unsigned long long mask_seed, const unsigned long long* seed_offset, dost_stream_t stream",
}
CTYPE = {"int": C.c_int, "long long": C.c_longlong, "double": C.c_double, "unsigned long long": C.c_ulonglong}


def test_header_ctypes_and_exports_of_the_map_kernels_agree():
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
        # the mask seed is followed by the optional device word of the forward it reproduces
        i = decl.index("unsigned long long mask_seed")
        assert decl[i + 1] == "const unsigned long long* seed_offset"
        assert name in L.EXPORTED_SYMBOLS and getattr(lib, name).argtypes == args


def test_map_kernels_reject_bad_arguments_without_a_launch():
    lib = L.load()
    assert lib.dost_attn_maps_from_planes(None, None, 8, 1, 1, 1, 1, None, None, None, 0.0, 0, None, None) != 0
    assert b"attn_maps_from_planes" in lib.dost_last_error()
    assert lib.dost_xattn_probs(0, None, 0, None, None, None, None, None, None, 1, 1, 1, 1, 32, 1.0, 0.0, 0, None, None) != 0
    assert b"xattn_probs" in lib.dost_last_error()
