"""ctypes binding of libtoda_b200.so (C ABI declared in include/toda_b200.h).

There is no CPU fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtoda_b200.so")

c_int, c_i64, c_f32, c_vp, c_sz = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t
_IP = ctypes.POINTER(ctypes.c_int)
_FP = ctypes.POINTER(ctypes.c_float)
# toda_alloc_fn: (rows, ctx) -> device pointer of the output the library asks for once it knows its size
ALLOC_FN = ctypes.CFUNCTYPE(c_vp, c_sz, c_vp)

# name -> (restype, argtypes); must list every symbol include/toda_b200.h declares
SIGNATURES = {
    "toda_last_error": (ctypes.c_char_p, []),
    "toda_version": (c_int, []),
    "toda_launch_count": (ctypes.c_longlong, []),
    "toda_device_info": (c_int, [_IP, _IP, _IP]),
    "toda_index_bytes": (c_sz, [c_int] * 4),
    "toda_index_insert": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_vp]),
    "toda_index_insert_strided": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, _IP, _IP, _IP, c_vp]),
    "toda_index_build": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp]),
    "toda_index_rows": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp]),
    "toda_index_release": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_vp]),
    "toda_points_select_workspace_bytes": (c_sz, [c_int]),
    "toda_points_select": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_int, c_int, ctypes.POINTER(ctypes.c_double), c_int, c_int,
                                   c_vp, c_vp, c_vp, c_sz, c_vp]),
    "toda_points_world_transform": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_int, c_int, _IP, _FP, c_vp, c_vp]),
    "toda_gt_sampling_pack_boxes": (c_int, [c_vp, c_int, c_vp, c_vp]),
    "toda_gt_sampling_workspace_bytes": (c_sz, [c_int, c_int, c_int]),
    "toda_gt_sampling": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_int, c_vp, _IP, c_vp, _IP, c_int, c_vp, c_int, c_vp, c_vp,
                                 c_int, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "toda_rotate_paste_workspace_bytes": (c_sz, [c_int] * 4),
    "toda_rotate_paste": (c_int, [c_vp, c_int, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_vp, _IP, c_vp, _IP, c_vp, c_vp, _IP,
                                  c_vp, ALLOC_FN, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "toda_voxelize_workspace_bytes": (c_sz, [c_i64, c_int, _IP, c_int, c_int]),
    "toda_voxelize_hard": (c_int, [c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp, c_int, _FP, _FP, _IP, c_int, c_int,
                                   c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "toda_voxelize_dynamic_workspace_bytes": (c_sz, [c_i64, c_int, _IP]),
    "toda_voxelize_dynamic": (c_int, [c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp, c_int, _FP, _FP, _IP, c_vp, c_vp, c_vp,
                                      c_vp, c_sz, c_vp]),
    "toda_mean_vfe_fwd": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "toda_mean_vfe_bwd": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "toda_rulebook_subm": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, _IP, c_vp, c_vp]),
    "toda_rulebook_sparse": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_vp,
                                     c_int, _IP, _IP, _IP, c_vp, c_vp, c_vp]),
    "toda_weight_repack": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "toda_spconv_fwd_workspace_bytes": (c_sz, [c_int] * 5),
    "toda_spconv_uses_tensor_cores": (c_int, [c_int] * 4),
    "toda_spconv_wgrad_uses_tensor_cores": (c_int, [c_int] * 4),
    "toda_parity_order_workspace_bytes": (c_sz, [c_int]),
    "toda_parity_order": (c_int, [c_vp, c_int, _IP, _IP, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "toda_table_tile_masks": (c_int, [c_vp, c_int, c_int, c_vp, c_vp]),
    "toda_tile_plan_capacity": (c_int, [c_int]),
    "toda_table_tile_plan": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "toda_spconv_fwd": (c_int, [c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_sz, c_vp]),
    "toda_weight_kmajor_bf16": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_vp]),
    "toda_layer_fwd": (c_int, [c_vp, c_vp]),
    "toda_layer_bwd": (c_int, [c_vp, c_vp]),
    "toda_layer_fwd_stats": (c_int, [c_vp, c_vp, c_vp]),
    "toda_layer_fwd_apply": (c_int, [c_vp, c_vp, c_vp]),
    "toda_layer_bwd_reduce": (c_int, [c_vp, c_vp, c_vp]),
    "toda_layer_bwd_finish": (c_int, [c_vp, c_vp, c_vp, c_vp]),
    "toda_spconv_wgrad_workspace_bytes": (c_sz, [c_int] * 6),
    "toda_spconv_wgrad": (c_int, [c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_sz, c_int,
                                  c_vp]),
    "toda_spconv_wgrad_row_splits": (c_int, [c_vp, c_int, c_int, c_int, c_int, _IP, _IP, c_vp, c_vp]),
    "toda_bn_workspace_bytes": (c_sz, [c_int]),
    "toda_bn_local_sums": (c_int, [c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "toda_bn_eval_coeffs": (c_int, [c_vp, c_vp, c_vp, c_vp, c_f32, c_int, c_vp, c_vp, c_vp]),
    "toda_bn_apply": (c_int, [c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_vp]),
    "toda_bn_apply_sums": (c_int, [c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                   c_vp, c_int, c_vp, c_vp, c_vp]),
    "toda_bn_bwd": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp,
                            c_vp, c_vp, c_sz, c_vp]),
    "toda_bn_bwd_reduce": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "toda_bn_bwd_finish": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp,
                                   c_vp, c_vp, c_sz, c_vp]),
    "toda_col_sum": (c_int, [c_vp, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "toda_bev_scatter_fwd": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "toda_bev_scatter_bwd": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "toda_gather_rows": (c_int, [c_vp, c_vp, c_int, c_int, c_vp, c_vp]),
}



class LayerFwdArgs(ctypes.Structure):
    """toda_layer_fwd_args (include/toda_b200.h)."""
    _fields_ = [("x", c_vp), ("x_bf16", c_vp), ("n_in", c_int), ("cin", c_int), ("nbr", c_vp), ("n_out", c_int), ("kvol", c_int),
                ("w", c_vp), ("w_bf16", c_vp), ("cout", c_int), ("bias", c_vp), ("tile_masks", c_vp),
                ("plan_lidx", c_vp), ("plan_rows", c_vp), ("plan_cnt", c_vp), ("plan_groups", c_int), ("plan_cap", c_int),
                ("precision", c_int), ("conv_ws", c_vp), ("conv_ws_bytes", c_sz),
                ("gamma", c_vp), ("beta", c_vp), ("eps", c_f32), ("momentum", c_f32), ("running_mean", c_vp), ("running_var", c_vp),
                ("training", c_int), ("residual", c_vp), ("relu", c_int),
                ("y", c_vp), ("sums", c_vp), ("stats", c_vp), ("a", c_vp), ("a_bf16", c_vp), ("bn_ws", c_vp), ("bn_ws_bytes", c_sz)]


class LayerBwdArgs(ctypes.Structure):
    """toda_layer_bwd_args (include/toda_b200.h)."""
    _fields_ = [("da", c_vp), ("a_mask", c_vp), ("y", c_vp), ("n_out", c_int), ("cout", c_int), ("gamma", c_vp), ("mean", c_vp),
                ("rstd", c_vp), ("relu", c_int), ("training", c_int), ("dy", c_vp), ("dy_bf16", c_vp), ("dres", c_vp), ("dgamma", c_vp),
                ("dbeta", c_vp), ("bn_ws", c_vp), ("bn_ws_bytes", c_sz),
                ("x", c_vp), ("x_bf16", c_vp), ("n_in", c_int), ("cin", c_int), ("kvol", c_int),
                ("need_dx", c_int), ("dgrad_nbr", c_vp), ("wt", c_vp), ("wt_bf16", c_vp), ("dgrad_out_rows", c_vp), ("dgrad_masks", c_vp),
                ("dplan_lidx", c_vp), ("dplan_rows", c_vp), ("dplan_cnt", c_vp), ("dplan_groups", c_int), ("dplan_cap", c_int),
                ("addend", c_vp), ("dx", c_vp),
                ("need_dw", c_int), ("nbr_fwd", c_vp), ("fwd_masks", c_vp), ("dw", c_vp), ("wgrad_ws", c_vp), ("wgrad_ws_bytes", c_sz),
                ("need_db", c_int), ("db", c_vp),
                ("precision", c_int), ("conv_ws", c_vp), ("conv_ws_bytes", c_sz)]


_lib = None


def lib():
    """The loaded shared library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  toda_b200 has no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().toda_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libtoda_b200 {what} failed (code {rc}): {msg}")


def ints(vals):
    return (ctypes.c_int * len(vals))(*[int(v) for v in vals])


def doubles(vals):
    return (ctypes.c_double * len(vals))(*[float(v) for v in vals])


def floats(vals):
    return (ctypes.c_float * len(vals))(*[float(v) for v in vals])
