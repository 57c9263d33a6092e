"""ctypes binding of libcheckerpose_b200.so (the C ABI declared in include/checkerpose_b200.h).

The library is the product: if it is missing or fails to load, importing this module raises --
there is no eager-PyTorch or CPU fallback behind any op.
"""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

c_i32, c_i64, c_f32, c_vp, c_sz = C.c_int, C.c_int64, C.c_float, C.c_void_p, C.c_size_t


class ChainLayer(C.Structure):
    _fields_ = [("w_packed", c_vp), ("bias", c_vp), ("kin", c_i32), ("nout", c_i32), ("act", c_i32), ("slope", c_f32),
                ("w_stride", c_i64), ("b_stride", c_i32)]


class ChainParams(C.Structure):
    _fields_ = [
        ("prologue", c_i32), ("B", c_i32), ("N", c_i32),
        ("src", c_vp), ("ld_src", c_i32), ("C", c_i32),
        ("z", c_vp), ("ld_z", c_i32), ("Co", c_i32), ("idx", c_vp), ("graph_sel", c_vp), ("K", c_i32), ("agg_slope", c_f32),
        ("patches", c_vp), ("Hp", c_i32), ("Wp", c_i32), ("E", c_i32), ("tap_step", c_i32),
        ("x_id", c_vp), ("y_id", c_vp), ("mask", c_vp),
        ("graph_feat", c_vp), ("ld_gf", c_i32), ("Cg", c_i32),
        ("a_out", c_vp), ("ld_a_out", c_i32),
        ("num_layers", c_i32),
        ("layers", ChainLayer * 3),
        ("out_mode", c_i32), ("out", c_vp), ("ld_out", c_i32), ("n_valid", c_i32),
    ]


class GraphPlanStruct(C.Structure):
    _fields_ = [("G", c_i32), ("N", c_i32), ("K", c_i32), ("KP", c_i32), ("T", c_i32), ("umax", c_i32), ("max_unique", c_i32),
                ("ucount", c_vp), ("ulist", c_vp), ("prog", c_vp)]


class EdgeConvParams(C.Structure):
    _fields_ = [
        ("B", c_i32), ("N", c_i32),
        ("z", c_vp), ("ld_z", c_i32), ("Co", c_i32),
        ("plan", GraphPlanStruct), ("graph_sel", c_vp), ("agg_slope", c_f32),
        ("a_out", c_vp), ("ld_a_out", c_i32),
        ("layer", ChainLayer),
        ("out_mode", c_i32), ("out", c_vp), ("ld_out", c_i32), ("n_valid", c_i32),
    ]


class GemmX3Params(C.Structure):
    _fields_ = [
        ("mode", c_i32),
        ("a1", c_vp), ("ld1", c_i32), ("k1", c_i32),
        ("a2", c_vp), ("ld2", c_i32), ("k2", c_i32),
        ("H", c_i32), ("W", c_i32), ("Ho", c_i32), ("Wo", c_i32), ("KH", c_i32), ("KW", c_i32), ("pad", c_i32),
        ("M", c_i64), ("K", c_i32),
        ("w_hi", c_vp), ("w_lo", c_vp),
        ("bias", c_vp), ("act", c_i32), ("slope", c_f32),
        ("out", c_vp), ("ld_out", c_i32), ("Nout", c_i32),
    ]


class ConvBf16Params(C.Structure):
    _fields_ = [
        ("mode", c_i32),
        ("a1", c_vp), ("ld1", c_i32), ("k1", c_i32),
        ("H", c_i32), ("W", c_i32), ("Ho", c_i32), ("Wo", c_i32), ("KH", c_i32), ("KW", c_i32), ("pad", c_i32),
        ("M", c_i64), ("K", c_i32),
        ("w_packed", c_vp),
        ("bias", c_vp), ("act", c_i32), ("slope", c_f32),
        ("out", c_vp), ("ld_out", c_i32), ("Nout", c_i32),
    ]


SLAB_MAX_TAPS, SLAB_MAX_PHASES = 9, 4


class SlabPhase(C.Structure):
    _fields_ = [("ntaps", c_i32), ("wtap", c_i32 * SLAB_MAX_TAPS), ("shift", c_i32 * SLAB_MAX_TAPS), ("out_off", c_i32)]


class ConvSlabParams(C.Structure):
    _fields_ = [
        ("x", c_vp), ("B", c_i32), ("Hp", c_i32), ("Wp", c_i32), ("C", c_i32), ("ldx", c_i32),
        ("w_packed", c_vp), ("K", c_i32),
        ("bias", c_vp), ("act", c_i32), ("slope", c_f32),
        ("out", c_vp), ("ld_out", c_i32), ("Nout", c_i32),
        ("num_phases", c_i32), ("phase", SlabPhase * SLAB_MAX_PHASES),
        ("vy0", c_i32), ("vy1", c_i32), ("vx0", c_i32), ("vx1", c_i32),
        ("compact", c_i32), ("out_sb", c_i64), ("out_sy", c_i32), ("out_sx", c_i32),
        ("seg_w", c_vp), ("seg_b", c_vp), ("seg_out", c_vp), ("seg_n", c_i32),
    ]


class QueryDecodeParams(C.Structure):
    _fields_ = [
        ("B", c_i32), ("N", c_i32),
        ("src", c_vp), ("ld_src", c_i32), ("kin", c_i32),
        ("w1_packed", c_vp), ("b1", c_vp), ("nmid", c_i32), ("slope", c_f32),
        ("w2", c_vp), ("b2", c_vp), ("nout", c_i32),
        ("logits", c_vp), ("ld_logits", c_i32),
        ("plane", c_i32), ("Ltot", c_i32),
        ("x_bits", c_vp), ("y_bits", c_vp), ("x_id", c_vp), ("y_id", c_vp), ("x_id_kp", c_vp), ("y_id_kp", c_vp),
        ("perm", c_vp), ("graph_sel", c_vp),
        ("w1_stride", c_i64), ("b1_stride", c_i32), ("w2_stride", c_i32), ("b2_stride", c_i32),
    ]


# name -> (restype, argtypes); must list every symbol of include/checkerpose_b200.h
SIGNATURES = {
    "cp_last_error_string": (C.c_char_p, []),
    "cp_version": (c_i32, []),
    "cp_device_arch": (c_i32, []),
    "cp_pack_weight_split": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "cp_gemm_x3": (c_i32, [C.POINTER(GemmX3Params), c_vp]),
    "cp_edge_aggregate_staged_f32": (c_i32, [c_vp, C.POINTER(GraphPlanStruct), c_vp, c_f32, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "cp_pnp_ransac": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_i32, C.c_uint64, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "cp_query_decode_fwd": (c_i32, [C.POINTER(QueryDecodeParams), c_vp]),
    "cp_conv_bf16": (c_i32, [C.POINTER(ConvBf16Params), c_vp]),
    "cp_conv_slab": (c_i32, [C.POINTER(ConvSlabParams), c_vp]),
    "cp_zero_border_nhwc": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "cp_upsample2x_cat_nhwc_to": (c_i32, [c_vp, c_i64, c_i64, c_i64, c_i32, c_vp, c_i64, c_i64, c_i64, c_i32, c_i32, c_vp, c_i64, c_i64,
                                          c_i64, c_i32, c_i32, c_i32, c_vp]),
    "cp_graph_sel": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp]),
    "cp_knn": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "cp_transpose_cn_to_nc": (c_i32, [c_vp, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "cp_transpose_nc_to_cn": (c_i32, [c_vp, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "cp_convert": (c_i32, [c_vp, c_i32, c_vp, c_i32, c_i64, c_vp]),
    "cp_graph_feature": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "cp_fold_edgeconv": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_f32, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "cp_packed_weight_bytes": (c_sz, [c_i32, c_i32]),
    "cp_pack_weight": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_vp]),
    "cp_linear_f32": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp, c_i32, c_f32, c_vp, c_i32, c_i64, c_i32, c_vp]),
    "cp_edge_aggregate": (c_i32, [c_vp, c_i32, c_vp, c_vp, c_f32, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "cp_chain_fwd": (c_i32, [C.POINTER(ChainParams), c_vp]),
    "cp_sample_taps": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_vp]),
    "cp_upsample2x_cat_nhwc": (c_i32, [c_vp, c_i64, c_i64, c_i64, c_i32, c_vp, c_i64, c_i64, c_i64, c_i32, c_i32, c_vp, c_i32,
                                       c_i32, c_i32, c_vp]),
    "cp_decode_init": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "cp_decode_refine": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "cp_transpose_scatter_bf16": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "cp_bias_add_rows_bf16": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_i32, c_vp]),
    "cp_permute_rows": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_i32, c_vp]),
    "cp_graph_plan_kp": (c_i32, [c_i32]),
    "cp_edgeconv_ring_rows": (c_i32, [c_i32]),
    "cp_graph_plan_build": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cp_edgeconv_fwd": (c_i32, [C.POINTER(EdgeConvParams), c_vp]),
    "cp_correspondences": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "cp_correspondences_pack": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "cp_correspondences_unpack": (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "cp_fps": (c_i32, [c_vp, c_i32, c_i32, C.POINTER(C.c_double), C.c_double, c_vp, c_vp, c_vp, c_vp]),
    "cp_threshold": (c_i32, [c_vp, c_f32, c_i32, c_vp, c_i32, c_i64, c_vp]),
    "cp_id_to_bits": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    "cp_group_argmax": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_vp]),
    "cp_bits_to_id": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_i64, c_i64, c_i64, c_i32, c_f32, c_i32, c_vp, c_i32, c_vp]),
}

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -m checkerpose_b200.build` (or __graft_entry__.build()). "
        "checkerpose_b200 has no fallback path.")

lib = C.CDLL(LIB_PATH)
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)   # AttributeError here == the .so does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = lib.cp_last_error_string()
        raise RuntimeError(f"checkerpose_b200 {what} failed ({status}): {msg.decode() if msg else '?'}")
