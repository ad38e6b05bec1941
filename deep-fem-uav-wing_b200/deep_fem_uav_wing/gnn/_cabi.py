"""ctypes binding of ``libdfw_b200.so`` (C ABI declared in ``include/dfw_b200.h``).

The shared library is the product: there is no CPU or PyTorch fallback behind these calls.
If it has not been built, importing this module raises immediately with the build command.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_double, c_float, c_int, c_int64, c_size_t, c_uint64, c_void_p

_PKG_ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
LIB_PATH = os.environ.get("DFW_B200_LIB", os.path.join(_PKG_ROOT, "lib", "libdfw_b200.so"))

DFW_F32, DFW_BF16 = 0, 1
EP_RELU, EP_LAYERNORM, EP_RESIDUAL, EP_DROPOUT, EP_SEED_IS_PTR, EP_TRANSPOSE_W, EP_OUT_BF16 = 1, 2, 4, 8, 16, 32, 64

# name -> (restype, argtypes); must list every symbol of include/dfw_b200.h
SIGNATURES = {
    "dfw_last_error": (ctypes.c_char_p, []),
    "dfw_abi_version": (c_int, []),
    "dfw_csr_ws_bytes": (c_size_t, [c_int64, c_int64]),
    "dfw_csr_build": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_size_t, c_void_p]),
    "dfw_csr_transpose": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_size_t, c_void_p]),
    "dfw_faces_ws_bytes": (c_size_t, [c_int64, c_int64]),
    "dfw_faces_to_csr": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dfw_node_features_ws_bytes": (c_size_t, [c_int64]),
    "dfw_node_features": (c_int, [c_void_p, c_void_p, c_void_p, ctypes.POINTER(c_float), c_int, c_int, c_void_p, c_void_p, c_int64,
                                  c_void_p, c_size_t, c_void_p]),
    "dfw_node_features_batched_ws_bytes": (c_size_t, [c_int64]),
    "dfw_node_features_batched": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p,
                                          c_void_p, c_size_t, c_void_p]),
    "dfw_graphsage_forward_ws_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64, c_int64, c_int, c_int]),
    "dfw_graphsage_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, ctypes.POINTER(c_void_p), c_int, c_int64, c_int64, c_int64,
                                      c_int64, c_int64, c_int64, c_float, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dfw_sage_aggregate": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                   c_int, c_void_p]),
    "dfw_sage_aggregate_scaled": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int,
                                          c_void_p]),
    "dfw_agg_plan_sizes": (c_int, [c_int64, c_int64, ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), ctypes.POINTER(c_int64)]),
    "dfw_agg_plan_max_block_edges": (c_int, []),
    "dfw_agg_plan_build": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_size_t, c_void_p]),
    "dfw_sage_aggregate_tc": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int,
                                      c_void_p]),
    "dfw_linear_fwd": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                               c_float, c_void_p, c_float, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "dfw_linear_ws_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int]),
    "dfw_linear_tc_eligible": (c_int, [c_int64, c_int64, c_int64, c_int64, c_int]),
    "dfw_epilogue_bwd_ws_bytes": (c_size_t, [c_int64, c_int64]),
    "dfw_epilogue_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_float, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                 c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "dfw_linear_bwd_input": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int,
                                     c_void_p, c_size_t, c_void_p]),
    "dfw_linear_bwd_weight_ws_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64]),
    "dfw_linear_bwd_weight": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                      c_int64, c_int64, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "dfw_sage_layer_fwd_ws_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int]),
    "dfw_sage_layer_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_float, c_float, c_uint64, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int64, c_int64, c_int64, c_int64, c_int, c_void_p, c_size_t, c_void_p]),
    "dfw_sage_layer_bwd_ws_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int, c_int]),
    "dfw_sage_layer_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_float, c_uint64, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int, c_void_p, c_size_t, c_void_p]),
    "dfw_mlp2_fwd_ws_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64, c_int]),
    "dfw_mlp2_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_uint64, c_int, c_int, c_void_p, c_void_p,
                             c_int64, c_int64, c_int64, c_int64, c_int, c_void_p, c_size_t, c_void_p]),
    "dfw_mlp2_bwd_ws_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64, c_int, c_int, c_int]),
    "dfw_mlp2_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_uint64, c_int, c_int,
                             c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int,
                             c_void_p, c_size_t, c_void_p]),
    "dfw_masked_mse_ws_bytes": (c_size_t, [c_int64, c_int64]),
    "dfw_masked_mse_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p,
                                   c_size_t, c_void_p]),
    "dfw_masked_mse_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int,
                                   c_void_p, c_void_p]),
    "dfw_stress_metrics_ws_bytes": (c_size_t, [c_int64, c_int64]),
    "dfw_stress_metrics": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_size_t,
                                   c_void_p]),
    "dfw_vertex_normals_ws_bytes": (c_size_t, [c_int64, c_int64]),
    "dfw_vertex_normals": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dfw_case_stress_summary_ws_bytes": (c_size_t, [c_int64, c_int64]),
    "dfw_case_stress_summary": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_double, c_double, c_int,
                                        c_void_p, c_void_p, c_size_t, c_void_p]),
    "dfw_cast": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_void_p]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"libdfw_b200.so not found at {LIB_PATH}. This package has no CPU/PyTorch fallback: build the CUDA "
            "library first (python -c 'import __graft_entry__ as g; g.build()' at the repo root, or "
            "make -C deep-fem-uav-wing_b200/csrc)."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


class DfwError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        raise DfwError(lib.dfw_last_error().decode("utf-8", "replace"))
