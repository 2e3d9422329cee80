"""ctypes binding of libstdadk.so (include/stdadk.h).  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# STDADK_LIB: an alternative build of the same library (e.g. the -DSTDADK_PF_DEBUG profiling build of tools/)
LIB_PATH = os.environ.get("STDADK_LIB") or os.path.join(_HERE, "libstdadk.so")
MAX_Q = 8

WENDLAND, GAUSSIAN, TRIANGULAR = 0, 1, 2
LOSS_NONE, LOSS_MSE, LOSS_PINBALL = 0, 1, 2
BASIS_CODE = {"wendland": WENDLAND, "gaussian": GAUSSIAN, "triangular": TRIANGULAR}
# stnf/models/st_interp.py:56-60
CALIBRATION = {"wendland": 1.0, "gaussian": 0.223477, "triangular": 0.654714}

fp = C.c_void_p  # device pointers travel as integers


SETTLED_STEP, SETTLED_X = 1, 2       # stdadk_bwd_args.settled bits (STDADK_SETTLED_*)


class Basis(C.Structure):
    _fields_ = [("knots4", fp), ("tknots2", fp), ("k_s", C.c_int32), ("k_t", C.c_int32), ("p_cov", C.c_int32),
                ("basis_fn", C.c_int32)]


class Points(C.Structure):
    _fields_ = [("coords", fp), ("t", fp), ("xcov", fp), ("index", fp), ("grid_nx", C.c_int32), ("grid_ny", C.c_int32),
                ("grid_nt", C.c_int32), ("_pad", C.c_int32), ("row_begin", C.c_int64), ("n_rows", C.c_int64)]


class Layer(C.Structure):
    _fields_ = [("w_img", fp), ("bias", fp), ("gamma", fp), ("beta", fp), ("n_in", C.c_int32), ("n_out", C.c_int32),
                ("ln_eps", C.c_float), ("layer_id", C.c_int32), ("w_img_lo", fp)]


class Dropout(C.Structure):
    _fields_ = [("p", C.c_float), ("step", C.c_uint32), ("seed", C.c_uint64), ("step_ptr", fp),
                ("key_offset", C.c_uint64)]


class Head(C.Structure):
    _fields_ = [("w", fp), ("b", fp), ("q", C.c_int32), ("loss_type", C.c_int32), ("y", fp),
                ("taus", C.c_float * MAX_Q), ("inv_count", C.c_float), ("nc_weight", C.c_float),
                ("nc_power", C.c_int32), ("_pad", C.c_int32), ("yhat", fp), ("dyhat", fp), ("loss_acc", fp)]


class FwdArgs(C.Structure):
    _fields_ = [("basis", C.POINTER(Basis)), ("pts", Points), ("a_img", fp), ("layer", Layer), ("drop", Dropout),
                ("out_img", fp), ("stats", fp), ("head", C.POINTER(Head)), ("addend", fp), ("feat_img", fp), ("x_img", fp),
                ("a_img_lo", fp), ("out_img_lo", fp)]


class BwdArgs(C.Structure):
    _fields_ = [("basis", C.POINTER(Basis)), ("pts", Points), ("a_img", fp), ("layer", Layer), ("drop", Dropout),
                ("stats", fp), ("head", C.POINTER(Head)), ("d_head_w", fp), ("d_head_b", fp), ("dz_next_img", fp),
                ("wt_next_img", fp), ("n_next", C.c_int32), ("settled", C.c_int32), ("dz_img", fp), ("d_bias", fp),
                ("d_gamma", fp), ("d_beta", fp), ("addend", fp), ("x_img", fp), ("a_img_lo", fp), ("dz_next_img_lo", fp),
                ("wt_next_img_lo", fp), ("dz_img_lo", fp)]


class WgradArgs(C.Structure):
    _fields_ = [("basis", C.POINTER(Basis)), ("pts", Points), ("a_img", fp), ("dz_img", fp), ("n_in", C.c_int32),
                ("n_out", C.c_int32), ("dw", fp), ("stride_o", C.c_int64), ("stride_i", C.c_int64), ("a_img_lo", fp),
                ("dz_img_lo", fp)]


class KnotGradArgs(C.Structure):
    _fields_ = [("basis", C.POINTER(Basis)), ("pts", Points), ("dz_img", fp), ("w1s_img", fp), ("n_out", C.c_int32),
                ("_pad", C.c_int32), ("d_centers", fp), ("d_log_bw", fp), ("dz_img_lo", fp), ("w1s_img_lo", fp)]


class AdamWArgs(C.Structure):
    _fields_ = [("p", fp), ("g", fp), ("m", fp), ("v", fp), ("shadow", fp), ("n", C.c_int64),
                ("n_groups", C.c_int32), ("zero_grad", C.c_int32), ("group_end", C.POINTER(C.c_int64)), ("hyper", fp),
                ("sqnorms", fp), ("step_count", fp), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("ema_decay", C.c_float), ("loss_acc", fp), ("loss_sum", fp), ("loss_last", fp), ("fuse_norm", C.c_int32),
                ("state_early", C.c_int32), ("norm_ws", fp)]


MAX_LEVELS = 8


class SparseArgs(C.Structure):
    _fields_ = [("pts", Points), ("knots4", fp), ("n_levels", C.c_int32), ("basis_fn", C.c_int32), ("n_out", C.c_int32),
                ("p_cov", C.c_int32), ("side", C.c_int32 * MAX_LEVELS), ("offset", C.c_int32 * MAX_LEVELS),
                ("thetap", C.c_float * MAX_LEVELS), ("w1t", fp), ("zs", fp), ("dz_img", fp), ("dw1t", fp),
                ("celllist", fp), ("celllist_k_s", C.c_int32), ("_pad", C.c_int32), ("d_centers", fp), ("d_log_bw", fp)]


class PackDesc(C.Structure):
    _fields_ = [("src", fp), ("row_stride", C.c_int64), ("col_stride", C.c_int64), ("rows", C.c_int64),
                ("cols", C.c_int64), ("img", fp), ("part", C.c_int32), ("_pad", C.c_int32)]


MAX_HIDDEN = 4


class PredictArgs(C.Structure):
    _fields_ = [("basis", C.POINTER(Basis)), ("pts", Points), ("n_layers", C.c_int32), ("_pad", C.c_int32),
                ("layers", Layer * MAX_HIDDEN), ("head", C.POINTER(Head))]


class FieldArgs(C.Structure):
    _fields_ = [("basis", C.POINTER(Basis)), ("sites", fp), ("grid_nx", C.c_int32), ("grid_ny", C.c_int32),
                ("n_sites", C.c_int64), ("n_times", C.c_int32), ("k_begin", C.c_int32), ("k_end", C.c_int32),
                ("n_layers", C.c_int32), ("site_begin", C.c_int64), ("site_end", C.c_int64),
                ("layers", Layer * MAX_HIDDEN), ("w1", fp), ("w1_row_stride", C.c_int64), ("w1_col_stride", C.c_int64),
                ("head", C.POINTER(Head)), ("row_base", C.c_int64), ("zt_ws", fp), ("out_k_stride", C.c_int64)]


MAX_PEERS = 8


class PeerAllreduceArgs(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("g", fp), ("n", C.c_int64), ("recv", fp * MAX_PEERS),
                ("step_count", fp), ("n_groups", C.c_int32), ("mode", C.c_int32), ("group_end", C.POINTER(C.c_int64)),
                ("sqnorms", fp), ("workspace", fp)]


_lib = None

_PROTOS = {
    "stdadk_version": (C.c_int, []),
    "stdadk_last_error": (C.c_char_p, []),
    "stdadk_sizeof": (C.c_size_t, [C.c_int]),
    "stdadk_image_floats": (C.c_size_t, [C.c_int64, C.c_int64]),
    "stdadk_knots_prepare": (C.c_int, [fp, fp, fp, C.c_float, C.c_int, fp, fp]),
    "stdadk_tknots_prepare": (C.c_int, [fp, fp, C.c_int, fp, fp]),
    "stdadk_basis_fwd": (C.c_int, [C.POINTER(Basis), C.POINTER(Points), fp, fp, fp]),
    "stdadk_pack_image": (C.c_int, [fp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, fp, fp]),
    "stdadk_unpack_image": (C.c_int, [fp, C.c_int64, C.c_int64, fp, fp]),
    "stdadk_pack_images": (C.c_int, [C.POINTER(PackDesc), C.c_int, fp]),
    "stdadk_predict_supported": (C.c_int, [C.POINTER(PredictArgs)]),
    "stdadk_predict": (C.c_int, [C.POINTER(PredictArgs), fp]),
    "stdadk_predict_field_supported": (C.c_int, [C.POINTER(FieldArgs)]),
    "stdadk_predict_field": (C.c_int, [C.POINTER(FieldArgs), fp]),
    "stdadk_peer_allreduce": (C.c_int, [C.POINTER(PeerAllreduceArgs), fp]),
    "stdadk_layer_fwd": (C.c_int, [C.POINTER(FwdArgs), fp]),
    "stdadk_layer_bwd": (C.c_int, [C.POINTER(BwdArgs), fp]),
    "stdadk_wgrad": (C.c_int, [C.POINTER(WgradArgs), fp]),
    "stdadk_dense_basis_supported": (C.c_int, [C.c_int32] * 6),
    "stdadk_dense_max_knots": (C.c_int32, [C.c_int32] * 5),
    "stdadk_knot_grad": (C.c_int, [C.POINTER(KnotGradArgs), fp]),
    "stdadk_sqnorm_ws_floats": (C.c_size_t, []),
    "stdadk_grad_sqnorm": (C.c_int, [fp, C.c_int64, C.c_int, C.POINTER(C.c_int64), fp, fp, fp]),
    "stdadk_adamw_ema_step": (C.c_int, [C.POINTER(AdamWArgs), fp]),
    "stdadk_celllist_ws_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "stdadk_celllist_build": (C.c_int, [fp, C.c_int32, C.POINTER(C.c_int32), C.c_int32, fp, C.c_size_t, fp]),
    "stdadk_sparse_l1_fwd": (C.c_int, [C.POINTER(SparseArgs), fp]),
    "stdadk_sparse_l1_wgrad": (C.c_int, [C.POINTER(SparseArgs), fp]),
}
EXPORTED = list(_PROTOS)


def lib():
    """Load libstdadk.so once; a missing library is an error, never a fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  st_dadk_b200 has no CPU or PyTorch fallback path.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            if not hasattr(L, name):
                continue
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        # (stdadk_sizeof index, struct); index 13 is unused
        structs = [(0, Basis), (1, Points), (2, Layer), (3, Dropout), (4, Head), (5, FwdArgs), (6, BwdArgs), (7, WgradArgs),
                   (8, KnotGradArgs), (9, AdamWArgs), (10, PackDesc), (11, SparseArgs), (12, PredictArgs),
                   (14, PeerAllreduceArgs), (15, FieldArgs)]
        for i, st in structs:
            if L.stdadk_sizeof(i) != C.sizeof(st):
                raise RuntimeError(f"libstdadk ABI mismatch: {st.__name__} is {C.sizeof(st)} B in the binding, "
                                   f"{L.stdadk_sizeof(i)} B in the library")
        _lib = L
    return _lib


def check(code: int, what: str):
    if code != 0:
        msg = lib().stdadk_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libstdadk {what} failed (code {code}): {msg}")
