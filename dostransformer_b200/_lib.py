"""ctypes binding of libdost_b200.so (the C ABI declared in include/dost.h).

There is no CPU fallback: if the shared library is missing or a CUDA device is not visible, every
op raises.  Build the library with ``python -m dostransformer_b200.build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# DOST_B200_LIB: an alternative build of the same library (A/B timing of kernel variants on one box)
LIB_PATH = os.environ.get("DOST_B200_LIB") or os.path.join(_HERE, "libdost_b200.so")

F32, F64 = 0, 1
ACT_NONE, ACT_RELU, ACT_LEAKY, ACT_PRELU = 0, 1, 2, 3
KC, MC = 0, 1
PREC_FMA, PREC_BF16X3, PREC_BF16 = 0, 1, 2
PRECISIONS = {"fp32": PREC_FMA, "bf16x3": PREC_BF16X3, "bf16": PREC_BF16}

_lib: Optional[C.CDLL] = None
ABI_VERSION = 15
DEVERR_MESSAGES = {1: "an index (edge_index / batch / system) is outside its table",
                   2: "a crystal has more atoms than the padding length given by the host (max_num_nodes)"}


class Seg(C.Structure):
    _fields_ = [("base", C.c_void_p), ("ld", C.c_longlong), ("idx", C.c_void_p), ("div", C.c_int),
                ("width", C.c_int)]


class Gemm(C.Structure):
    _fields_ = [
        ("dtype", C.c_int), ("M", C.c_int), ("N", C.c_int), ("K", C.c_int), ("batch", C.c_int),
        ("a_mode", C.c_int), ("a_nseg", C.c_int), ("a", Seg * 3), ("a_bstride", C.c_longlong),
        ("b_mode", C.c_int), ("b", Seg), ("b_bstride", C.c_longlong),
        ("bias", C.c_void_p), ("act", C.c_int), ("act_slope", C.c_double), ("prelu_slope", C.c_void_p),
        ("out_pre", C.c_void_p), ("ld_pre", C.c_longlong),
        ("dact_saved", C.c_void_p), ("ld_dact", C.c_longlong), ("dact_kind", C.c_int), ("dact_slope", C.c_double),
        ("residual", C.c_void_p), ("ld_res", C.c_longlong),
        ("out", C.c_void_p), ("ldc", C.c_longlong), ("c_bstride", C.c_longlong),
        ("accumulate", C.c_int), ("split_k", C.c_int), ("precision", C.c_int),
    ]


class PlanesC(C.Structure):
    _fields_ = [("hi", C.c_void_p), ("lo", C.c_void_p), ("ld", C.c_longlong), ("rows", C.c_longlong), ("width", C.c_int)]


class GemmBf16(C.Structure):
    _fields_ = [
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("a_mode", C.c_int), ("a_nseg", C.c_int), ("a", PlanesC * 3),
        ("b_mode", C.c_int), ("b", PlanesC),
        ("bias", C.c_void_p),
        ("rowbias", C.c_void_p), ("ld_rowbias", C.c_longlong), ("rowbias_div", C.c_int),
        ("act", C.c_int), ("act_slope", C.c_float), ("prelu_slope", C.c_void_p),
        ("out_pre", C.c_void_p), ("ld_pre", C.c_longlong),
        ("dact_hi", C.c_void_p), ("ld_dact", C.c_longlong), ("dact_slope", C.c_float),
        ("residual", C.c_void_p), ("ld_res", C.c_longlong),
        ("out", C.c_void_p), ("ldc", C.c_longlong), ("accumulate", C.c_int),
        ("out_hi", C.c_void_p), ("out_lo", C.c_void_p), ("ld_op", C.c_longlong),
        ("split_k", C.c_int), ("precision", C.c_int),
        ("batch", C.c_int), ("a_bstride", C.c_longlong), ("b_bstride", C.c_longlong), ("c_bstride", C.c_longlong),
        ("res_bstride", C.c_longlong),
        ("b_rowoff", C.c_void_p), ("c_rowoff", C.c_void_p), ("c_rowlim", C.c_void_p),
        ("colsum", C.c_void_p),
        ("out_gate", C.c_void_p), ("dact_gate", C.c_void_p), ("ld_gate", C.c_longlong),
    ]


_SIGNATURES = {
    "dost_abi_version": (C.c_int, []),
    "dost_last_error": (C.c_char_p, []),
    "dost_launch_count": (C.c_longlong, []),
    "dost_reset_launch_count": (None, []),
    "dost_device_errors_init": (C.c_int, []),
    "dost_device_errors": (C.c_uint, [C.c_int]),
    "dost_imax_scalar": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "dost_cast_i64_i32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "dost_csr_workspace_bytes": (C.c_size_t, [C.c_longlong, C.c_longlong]),
    "dost_csr_build": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_size_t, C.c_void_p]),
    "dost_gemm_workspace_bytes": (C.c_size_t, [C.POINTER(Gemm)]),
    "dost_gemm": (C.c_int, [C.POINTER(Gemm), C.c_void_p, C.c_size_t, C.c_void_p]),
    "dost_gemm_bf16_workspace_bytes": (C.c_size_t, [C.POINTER(GemmBf16)]),
    "dost_gemm_bf16": (C.c_int, [C.POINTER(GemmBf16), C.c_void_p, C.c_size_t, C.c_void_p]),
    "dost_split_planes": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong,
                                    C.c_void_p]),
    "dost_split_planes_multi": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "dost_split_planes_colsum_workspace_bytes": (C.c_size_t, [C.c_longlong, C.c_int, C.c_longlong]),
    "dost_split_planes_colsum": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong,
                                           C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dost_ln_fwd_planes": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "dost_ln_bwd_planes_workspace_bytes": (C.c_size_t, [C.c_longlong, C.c_int]),
    "dost_ln_bwd_planes": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p,
                                     C.c_size_t, C.c_void_p]),
    "dost_rowdot_fwd": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "dost_rowdot_bwd_workspace_bytes": (C.c_size_t, [C.c_longlong, C.c_int]),
    "dost_rowdot_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int,
                                  C.c_void_p, C.c_size_t, C.c_void_p]),
    "dost_colsum_planes_workspace_bytes": (C.c_size_t, [C.c_longlong, C.c_int]),
    "dost_colsum_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_size_t, C.c_void_p]),
    "dost_ln_fwd": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "dost_ln_bwd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_longlong, C.c_int]),
    "dost_ln_bwd": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong,
                              C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dost_colsum_workspace_bytes": (C.c_size_t, [C.c_int, C.c_longlong, C.c_longlong]),
    "dost_colsum": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p,
                              C.c_size_t, C.c_void_p]),
    "dost_prelu_bwd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_longlong]),
    "dost_prelu_bwd": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong,
                                 C.c_void_p, C.c_size_t, C.c_void_p]),
    "dost_segment_reduce": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_longlong,
                                      C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p]),
    "dost_gather_rows": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p]),
    "dost_phonon_edge_feat": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]),
    "dost_phonon_edge_encode": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "dost_xattn_fwd": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_double, C.c_double, C.c_ulonglong, C.c_void_p]),
    "dost_xattn_bwd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "dost_xattn_bwd": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_double,
                                 C.c_double, C.c_ulonglong, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dost_xattn_kv_ext_build": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_longlong, C.c_void_p]),
    "dost_xattn_kv_ext_split": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p]),
    "dost_xattn_kv_pad_split": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "dost_xattn_softmax_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_double,
                                         C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_double, C.c_ulonglong, C.c_void_p]),
    "dost_xattn_softmax_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int,
                                         C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_longlong, C.c_double, C.c_ulonglong,
                                         C.c_void_p]),
    "dost_softmax_fwd": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_double,
                                   C.c_double, C.c_ulonglong, C.c_void_p]),
    "dost_softmax_bwd": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_double,
                                   C.c_double, C.c_ulonglong, C.c_void_p]),
    "dost_softmax_fwd_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_double,
                                          C.c_double, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "dost_softmax_bwd_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_double,
                                          C.c_double, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "dost_attn_fused_supported": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "dost_attn_fused_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_double,
                                      C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int,
                                      C.c_double, C.c_ulonglong, C.c_void_p, C.c_void_p]),
    "dost_softmax_bwd_from_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int,
                                               C.c_double, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "dost_xattn_probs": (C.c_int, [C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_ulonglong,
                                   C.c_void_p, C.c_void_p]),
    "dost_attn_maps_from_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_int, C.c_int,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_ulonglong, C.c_void_p,
                                             C.c_void_p]),
    "dost_eval_metrics": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dost_adamw_step": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                  C.c_double, C.c_double, C.c_double, C.c_longlong, C.c_void_p]),
    "dost_loss_fwd": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p]),
    "dost_loss_bwd": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dost_collate_ptr": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "dost_collate_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong,
                                    C.c_longlong, C.c_void_p, C.c_void_p]),
    "dost_collate_index": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dost_neighbor_count": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_double, C.c_int,
                                      C.c_void_p, C.c_void_p]),
    "dost_neighbor_fill": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_double, C.c_int,
                                     C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "dost_knn_select": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_double,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dost_gaussian_expand": (C.c_int, [C.c_void_p, C.c_longlong, C.c_double, C.c_double, C.c_int, C.c_double, C.c_void_p,
                                       C.c_void_p]),
}


def _with_seed_offset(args):
    """The argument list of a dost_<name>_dseed sibling: `const unsigned long long* seed_offset` after the seed."""
    i = args.index(C.c_ulonglong) + 1
    return args[:i] + [C.c_void_p] + args[i:]


for _name in ("dost_xattn_fwd", "dost_xattn_bwd", "dost_xattn_softmax_fwd", "dost_xattn_softmax_bwd", "dost_softmax_fwd",
              "dost_softmax_bwd", "dost_softmax_fwd_planes", "dost_softmax_bwd_planes", "dost_attn_fused_fwd"):
    _res, _args = _SIGNATURES[_name]
    _SIGNATURES[_name + "_dseed"] = (_res, _with_seed_offset(_args))

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def load(path: str = LIB_PATH) -> C.CDLL:
    """dlopen the library and attach the signatures.  Does not need a GPU."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(path):
        raise RuntimeError(f"{path} not found: the CUDA extension is not built (python -m dostransformer_b200.build). "
                           "dostransformer_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.dost_abi_version() != ABI_VERSION:
        raise RuntimeError("libdost_b200.so ABI version mismatch")
    _lib = lib
    return lib


_cuda_checked = False


def lib() -> C.CDLL:
    """The loaded library, for compute calls: requires a visible CUDA device (checked once per process)."""
    global _cuda_checked
    L = _lib if _lib is not None else load()
    if not _cuda_checked:
        if not torch.cuda.is_available():
            raise RuntimeError("dostransformer_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        torch.cuda.init()
        check(L.dost_device_errors_init(), "device_errors_init")
        _cuda_checked = True
    return L


def poll_device_errors() -> None:
    """Raises if a kernel of an EARLIER, completed launch flagged invalid input (no device synchronisation: the flags live
    in mapped host memory).  Called at the start of every ops.build_graph; call it after torch.cuda.synchronize() to
    check the most recent step."""
    if _lib is None:
        return
    mask = int(_lib.dost_device_errors(1))
    if mask:
        msgs = [m for bit, m in DEVERR_MESSAGES.items() if mask & bit]
        raise RuntimeError("dostransformer_b200: a kernel skipped invalid input: " + "; ".join(msgs))


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().dost_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libdost_b200 {what} failed (rc={rc}): {msg}")


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_get_device = getattr(torch._C, "_cuda_getDevice", None)


def dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    raise TypeError(f"dostransformer_b200 supports float32/float64 tensors, got {t.dtype}")


def p(t: Optional[torch.Tensor]):
    """Device pointer of a tensor (honours storage offset) or NULL."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("dostransformer_b200: tensor is not on a CUDA device (no CPU fallback)")
    if _get_device is not None and t.get_device() != _get_device():
        # kernels launch on the CURRENT device's current stream: a tensor of another device would be dereferenced there
        raise RuntimeError(f"dostransformer_b200: tensor on cuda:{t.get_device()} but the current device is "
                           f"cuda:{_get_device()}; wrap the call in torch.cuda.device(tensor.device)")
    return C.c_void_p(t.data_ptr())




def stream():
    """cudaStream_t of torch's current stream on the current device (the raw-pointer query is ~10x cheaper than
    building a torch.cuda.Stream object; it is called once per kernel launch)."""
    if _raw_stream is not None and _get_device is not None:
        return _raw_stream(_get_device())
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


_switches = {}


def switch(name: str) -> bool:
    """Environment switch (DOST_NO_*), read once per process; reload_switches() re-reads them."""
    v = _switches.get(name)
    if v is None:
        v = _switches[name] = bool(os.environ.get(name))
    return v


def reload_switches() -> None:
    _switches.clear()


def launch_count() -> int:
    return int(load().dost_launch_count())


def reset_launch_count() -> None:
    load().dost_reset_launch_count()
