"""ctypes binding of libgps_b200.so (the C ABI declared in include/gps_b200.h).

The library is the product: there is no CPU or eager-PyTorch fallback.  If the shared object is
missing or fails to load, importing a function from here raises immediately.
"""
from __future__ import annotations

import ctypes as C
import os

import torch  # noqa: F401  (loads libcudart.so.12 into the process before our library resolves it)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgps_b200.so")

GPS_OK, GPS_ERR_ARG, GPS_ERR_UNSUPPORTED, GPS_ERR_CUDA = 0, -1, -2, -3
LOCAL = {"None": 0, "CustomGatedGCN": 1, "GINE": 2, "GCN": 3}
GLOBAL = {"None": 0, "Transformer": 1, "Performer": 2}
ACT = {"relu": 0, "gelu": 1}
PRECISION = {"fp32": 0, "bf16": 1}

_fp = C.c_void_p  # device pointers travel as void*


class GpsGraph(C.Structure):
    _fields_ = [("N", C.c_int64), ("E", C.c_int64), ("B", C.c_int64),
                ("dst_ptr", _fp), ("dst_src", _fp), ("dst_eid", _fp),
                ("src_ptr", _fp), ("src_dst", _fp), ("src_eid", _fp), ("graph_ptr", _fp)]


class GpsBatchNorm(C.Structure):
    _fields_ = [("weight", _fp), ("bias", _fp), ("running_mean", _fp), ("running_var", _fp),
                ("num_batches_tracked", _fp), ("grad_weight", _fp), ("grad_bias", _fp)]


class GpsLinear(C.Structure):
    _fields_ = [("weight", _fp), ("bias", _fp), ("grad_weight", _fp), ("grad_bias", _fp)]


class GpsPlanes(C.Structure):
    _fields_ = [("hi", _fp), ("lo", _fp), ("ld", C.c_int64)]


class GpsLayerArgs(C.Structure):
    _fields_ = [
        ("d", C.c_int64), ("heads", C.c_int64),
        ("local_type", C.c_int32), ("global_type", C.c_int32), ("act", C.c_int32),
        ("training", C.c_int32), ("precision", C.c_int32), ("reserved0", C.c_int32),
        ("dropout", C.c_float), ("attn_dropout", C.c_float),
        ("seed", C.c_uint64), ("offset", C.c_uint64),
        ("gine_eps", C.c_float), ("reserved1", C.c_int32),
        ("graph", GpsGraph),
        ("x", _fp), ("edge_attr", _fp), ("x_out", _fp), ("edge_out", _fp),
        ("gcn_A", GpsLinear), ("gcn_B", GpsLinear), ("gcn_C", GpsLinear), ("gcn_D", GpsLinear),
        ("gcn_E", GpsLinear),
        ("bn_node_x", GpsBatchNorm), ("bn_edge_e", GpsBatchNorm),
        ("gine_lin0", GpsLinear), ("gine_lin1", GpsLinear),
        ("attn_in", GpsLinear), ("attn_out", GpsLinear),
        ("perf_q", GpsLinear), ("perf_k", GpsLinear), ("perf_v", GpsLinear),
        ("perf_proj", _fp), ("perf_features", C.c_int64), ("perf_dim_head", C.c_int64),
        ("norm1_local", GpsBatchNorm), ("norm1_attn", GpsBatchNorm), ("norm2", GpsBatchNorm),
        ("ff1", GpsLinear), ("ff2", GpsLinear),
        ("grad_x_out", _fp), ("grad_edge_out", _fp), ("grad_x", _fp), ("grad_edge_attr", _fp),
        ("saved", _fp), ("saved_bytes", C.c_int64),
        ("workspace", _fp), ("workspace_bytes", C.c_int64),
        ("offset_dev", _fp),
        ("gcn_conv", GpsLinear),
        ("ev_grads_early", _fp),
        ("x_planes_in", GpsPlanes), ("e_planes_in", GpsPlanes), ("x_planes_out", GpsPlanes), ("e_planes_out", GpsPlanes),
        ("wplanes", _fp), ("wplanes_bytes", C.c_int64), ("wplanes_valid", C.c_int32), ("reserved2", C.c_int32),
        ("ev_grads_mid", _fp), ("ev_grads_done", _fp),
        ("pe", _fp), ("pe_dim", C.c_int64), ("grad_pe", _fp), ("es_r0", GpsLinear), ("es_r1", GpsLinear),
    ]

ES_FLAG = 1   # GpsLayerArgs.reserved1 bit 0: EquivStableLapPE edge gate


class GpsLayerPlan(C.Structure):
    _fields_ = [("saved_bytes", C.c_int64), ("fwd_workspace_bytes", C.c_int64),
                ("bwd_workspace_bytes", C.c_int64), ("fwd_launches", C.c_int64),
                ("bwd_launches", C.c_int64), ("wplanes_bytes", C.c_int64)]


# every symbol include/gps_b200.h declares: name -> (restype, argtypes)
_i64, _i32, _f32, _u64 = C.c_int64, C.c_int32, C.c_float, C.c_uint64
SYMBOLS = {
    "gps_last_error": (C.c_char_p, []),
    "gps_abi_version": (C.c_int, []),
    "gps_build_arch": (C.c_char_p, []),
    "gps_graph_bytes": (_i64, [_i64, _i64, _i64]),
    "gps_graph_build": (C.c_int, [_fp, _fp, _i64, _i64, _i64, _fp, _i64, C.POINTER(GpsGraph), _fp]),
    "gps_layer_plan": (C.c_int, [C.POINTER(GpsLayerArgs), C.POINTER(GpsLayerPlan)]),
    "gps_layer_forward": (C.c_int, [C.POINTER(GpsLayerArgs), _fp]),
    "gps_layer_backward": (C.c_int, [C.POINTER(GpsLayerArgs), _fp]),
    "gps_linear_forward": (C.c_int, [_fp, _i64, _fp, _i64, _fp, _fp, _i64, _i64, _i64, _i64, _i32, _i32, _fp]),
    "gps_gemm": (C.c_int, [_fp, _i64, _i32, _fp, _i64, _i32, _fp, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _fp]),
    "gps_gatedgcn_aggregate_forward": (C.c_int, [C.POINTER(GpsGraph), _i64, _fp, _fp, _fp, _fp, _i64, _fp, _fp,
                                                 _fp, _fp, _fp]),
    "gps_es_gate_forward": (C.c_int, [C.POINTER(GpsGraph), _fp, _i64, _i64, _i32] + [_fp] * 6 + [_fp]),
    "gps_gatedgcn_es_aggregate_forward": (C.c_int, [C.POINTER(GpsGraph), _i64, _fp, _fp, _fp, _fp, _i64, _fp, _fp,
                                                    _fp, _fp, _fp, _fp]),
    "gps_es_gate_backward_workspace_bytes": (_i64, [_i64, _i64]),
    "gps_es_gate_backward": (C.c_int, [_i64, _i64, _i32] + [_fp] * 12 + [_fp, _i64, _fp]),
    "gps_es_pe_backward": (C.c_int, [C.POINTER(GpsGraph), _fp, _i64, _fp, _fp, _fp]),
    "gps_gine_aggregate_forward": (C.c_int, [C.POINTER(GpsGraph), _i64, _fp, _fp, _f32, _fp, _fp]),
    "gps_attention_forward": (C.c_int, [C.POINTER(GpsGraph), _i64, _i64, _fp, _fp, _fp, _i64, _fp, _i64, _fp,
                                        _f32, _u64, _u64, _fp]),
    "gps_attention_backward": (C.c_int, [C.POINTER(GpsGraph), _i64, _i64, _fp, _fp, _fp, _i64, _fp, _fp, _i64,
                                         _fp, _fp, _fp, _fp, _fp, _i64, _f32, _u64, _u64, _fp]),
    "gps_attention_forward_tc": (C.c_int, [C.POINTER(GpsGraph), _i64, _i64, _fp, _fp, _i64, _fp, _i64, _fp, _f32, _u64, _u64,
                                           _i32, _fp]),
    "gps_dropout_mask": (C.c_int, [_fp, _i64, _i64, _f32, _u64, _u64, _i32, _fp]),
    "gps_to_planes": (C.c_int, [_fp, _i64, _i64, _i64, _fp, _fp, _i64, _fp]),
    "gps_gemm_planes": (C.c_int, [_fp, _fp, _i64, _i32, _fp, _fp, _i64, _i32, _fp, _i64, _fp, _fp, _i64, _i64, _i64, _i64,
                                  _i32, _i32, _fp, _fp]),
    "gps_fallback_count": (C.c_ulonglong, []),
    # not in the header's stage list but part of the ABI: launch counter for bench.py
    "gps_launch_count": (C.c_ulonglong, []),
    "gps_debug_set": (None, [C.c_int]),
    "gps_debug_tma": (None, [C.c_int, _fp]),
    "gps_debug_attn": (None, [_fp]),
}

_lib = None


def load():
    """Loads libgps_b200.so (once).  Raises if it is missing: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m graphgps_b200.build` "
            "(nvcc, sm_100a). graphgps_b200 has no CPU/eager fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.gps_abi_version() != 3:
        raise RuntimeError("libgps_b200.so ABI version mismatch")
    _lib = lib
    return lib


class GpsError(RuntimeError):
    pass


def check(rc: int, what: str):
    if rc == GPS_OK:
        return
    msg = load().gps_last_error().decode("utf-8", "replace")
    if rc == GPS_ERR_UNSUPPORTED:
        raise NotImplementedError(f"{what}: {msg}")
    if rc == GPS_ERR_ARG:
        raise ValueError(f"{what}: {msg}")
    raise GpsError(f"{what}: {msg}")


def ptr(t):
    """Device (or host) address of a tensor, 0 for None."""
    return 0 if t is None else t.data_ptr()
