"""ctypes binding of libgoliath_b200.so — the thin C-ABI extension (include/goliath_b200.h).

The product path has NO CPU fallback: if the CUDA library is missing, or a tensor is not on a CUDA
device, every op raises.  Build with `python -m goliath_b200.build` (nvcc, sm_100a).
"""
import ctypes
import os

import torch  # noqa: F401  (loads libcudart.so.12 first so the C library binds to the same runtime)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgoliath_b200.so")
_lib = None

_vp, _i, _f, _i64, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_int64, ctypes.c_size_t

# name -> (restype, argtypes); must list EVERY symbol include/goliath_b200.h declares (tests check it)
SIGNATURES = {
    "gb_version": (_i, []),
    "gb_launch_count": (ctypes.c_ulonglong, []),
    "gb_launch_count_reset": (None, []),
    "gb_sg_evaluate_fwd": (_i, [_vp] * 7 + [_i] * 4 + [_vp]),
    "gb_sg_evaluate_bwd": (_i, [_vp] * 10 + [_i] * 4 + [_vp]),
    "gb_project_gaussians_fwd": (_i, [_i, _vp, _vp, _f, _vp, _vp, _f, _f, _f, _f, _i, _i, _i, _f] + [_vp] * 7 + [_vp]),
    "gb_project_gaussians_bwd": (_i, [_i, _vp, _vp, _f, _vp, _vp, _f, _f] + [_vp] * 13 + [_vp]),
    "gb_cumsum_workspace_bytes": (_sz, [_i]),
    "gb_cumsum_i32": (_i, [_i, _vp, _vp, _vp, _vp]),
    "gb_map_gaussian_to_intersects": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "gb_sort_workspace_bytes": (_sz, [_i64]),
    "gb_sort_intersects": (_i, [_i64, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "gb_get_tile_bin_edges": (_i, [_i64, _vp, _vp, _vp]),
    "gb_rasterize_fwd": (_i, [_i, _i, _i, _i] + [_vp] * 10 + [_vp]),
    "gb_rasterize_bwd": (_i, [_i, _i, _i, _i] + [_vp] * 15 + [_vp]),
    "gb_pack_records": (_i, [_i64, _i] + [_vp] * 6 + [_vp]),
    "gb_tile_order": (_i, [_i, _vp, _vp, _vp]),
    "gb_pack_records_fused": (_i, [_i64] + [_vp] * 8 + [_vp]),
    "gb_pack_records_fused_dn": (_i, [_i64] + [_vp] * 9 + [_vp]),
    "gb_map_gaussian_to_intersects_dn": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _i64, _vp, _vp, _vp]),
    "gb_sort_intersects_dn": (_i, [_i64, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "gb_get_tile_bin_edges_dn": (_i, [_i64, _vp, _vp, _vp, _vp, _vp]),
    "gb_get_bin_sort_mode": (_i, []),
    "gb_set_bin_sort_mode": (None, [_i]),
    "gb_get_tile_sort_mode": (_i, []),
    "gb_set_tile_sort_mode": (None, [_i]),
    "gb_get_rank_sort_mode": (_i, []),
    "gb_set_rank_sort_mode": (None, [_i]),
    "gb_bin_tiles_supported": (_i, [_i]),
    "gb_bin_tiles_workspace_bytes": (_sz, [_i, _i, _i64]),
    "gb_bin_tiles_pack": (_i, [_i] + [_vp] * 7 + [_i, _i, _i, _i64] + [_vp, _vp, _i] + [_vp] * 5 + [_vp]),
    "gb_bin_tiles_pack_ev": (_i, [_i] + [_vp] * 7 + [_i, _i, _i, _i64] + [_vp, _vp, _i] + [_vp] * 5 + [_vp, _vp]),
    "gb_tile_schedule_ints": (_i, [_i]),
    "gb_tile_schedule": (_i, [_i, _vp, _vp, _vp]),
    "gb_rasterize_sched_fwd": (_i, [_i, _i, _i] + [_vp] * 7 + [_vp]),
    "gb_rasterize_sched_bwd": (_i, [_i, _i, _i] + [_vp] * 13 + [_vp]),
    "gb_records_widen": (_i, [_i64, _vp, _vp, _vp, _vp]),
    "gb_records_set_colors4": (_i, [_i64, _vp, _vp, _vp, _i, _i64, _vp, _vp]),
    "gb_rasterize_multi_fwd": (_i, [_i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "gb_rasterize_multi_bwd": (_i, [_i, _i, _vp, _vp, _vp, _i] + [_vp] * 9 + [_vp]),
    "gb_colors12_unpack": (_i, [_i64, _i, _vp, _vp, _vp]),
    "gb_records_set_colors": (_i, [_i64] + [_vp] * 5 + [_vp]),
    "gb_splat_grad_unpack": (_i, [_i] + [_vp] * 8 + [_vp]),
    "gb_get_blend_mode": (_i, []),
    "gb_set_blend_mode": (None, [_i]),
    "gb_rasterize_packed_fwd": (_i, [_i, _i, _i] + [_vp] * 7 + [_vp]),
    "gb_rasterize_packed_bwd": (_i, [_i, _i, _i] + [_vp] * 13 + [_vp]),
    "gb_rasterize_ranked_fwd": (_i, [_i, _i, _i] + [_vp] * 8 + [_vp]),
    "gb_rasterize_ranked_bwd": (_i, [_i, _i, _i] + [_vp] * 14 + [_vp]),
    "gb_bin_tiles_ranked": (_i, [_i] + [_vp] * 7 + [_i, _i, _i, _i64] + [_vp, _vp, _i] + [_vp] * 6 + [_vp, _vp]),
    "gb_compute_raydirs_fwd": (_i, [_i, _i, _i] + [_vp] * 5 + [_f] + [_vp] * 3 + [_vp]),
    "gb_compute_raydirs_bwd": (_i, []),
    "gb_mvp_aabb_workspace_bytes": (_sz, [_i, _i]),
    "gb_mvp_compute_aabb": (_i, [_i, _i] + [_vp] * 8 + [_vp]),
    "gb_get_raymarch_mode": (_i, []),
    "gb_set_raymarch_mode": (None, [_i]),
    "gb_mvp_raymarch_fwd": (_i, [_i] * 4 + [_vp, _vp, _f] + [_vp] * 5 + [_i] * 3 + [_vp] + [_i] * 3 + [_vp] * 4
                            + [_i, _f, _f, _i, _i, _vp]),
    "gb_deconv_tc_weight_bytes": (_sz, [_i, _i]),
    "gb_nchw_to_nhwc_split": (_i, [_i] * 5 + [_vp] * 3 + [_vp]),
    "gb_deconv4x4s2_tc_fwd": (_i, [_i] * 6 + [_vp] * 6 + [_f, _i, _vp, _vp, _i, _vp, _vp]),
    "gb_deconv4x4s2_wnub_fwd": (_i, [_i] * 5 + [_vp] * 4 + [_f, _i, _vp, _vp]),
    "gb_deconv4x4s2_wnub_bwd": (_i, [_i] * 5 + [_vp] * 5 + [_f, _i] + [_vp] * 4 + [_vp]),
    "gb_conv2d_wnub_fwd": (_i, [_i] * 6 + [_vp] * 4 + [_i, _f, _i, _vp, _vp]),
    "gb_conv2d_wnub_bwd": (_i, [_i] * 6 + [_vp] * 5 + [_f, _i, _i] + [_vp] * 4 + [_vp]),
    "gb_mvp_slab_to_prims_fwd": (_i, [_i] * 6 + [_vp] * 3 + [_f, _f, _i, _vp, _vp]),
    "gb_mvp_slab_to_prims_bwd": (_i, [_i] * 6 + [_vp] * 3 + [_f, _f, _i] + [_vp] * 3 + [_vp]),
    "gb_mvp_prim_transform_fwd": (_i, [_i, _i] + [_vp] * 3 + [_f, _i] + [_vp] * 3 + [_vp]),
    "gb_mvp_prim_transform_bwd": (_i, [_i, _i] + [_vp] * 3 + [_f, _i] + [_vp] * 4 + [_vp]),
    "gb_sg_shade_compose_fwd": (_i, [_vp] * 10 + [_i] * 4 + [_vp]),
    "gb_sg_shade_compose_bwd": (_i, [_vp] * 16 + [_i] * 4 + [_vp]),
    "gb_render_finish_fwd": (_i, [_i, _i] + [_vp] * 5 + [_vp]),
    "gb_render_finish_bwd": (_i, [_i, _i] + [_vp] * 4 + [_vp]),
    "gb_rgca_heads_fwd": (_i, [_i, _i] + [_vp] * 7 + [_f, _f] + [_vp] * 15 + [_vp]),
    "gb_rgca_heads_bwd": (_i, [_i, _i] + [_vp] * 7 + [_f, _f] + [_vp] * 20 + [_vp]),
    "gb_vert_normals_fwd": (_i, [_i, _i, _i, _vp, _vp, _f, _vp, _vp, _vp]),
    "gb_vert_normals_bwd": (_i, [_i, _i, _i, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp]),
    "gb_values_to_uv_fwd": (_i, [_i, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "gb_values_to_uv_bwd": (_i, [_i, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "gb_optim_chunk_elems": (_i, []),
    "gb_optim_row_bytes": (_i, []),
    "gb_grad_sanitize_sqnorm": (_i, [_vp, _vp, _i, _vp, _vp]),
    "gb_adam_step": (_i, [_vp, _vp, _i, _vp, _f, _f, _f, _f, _i, _i, _i, _vp]),
    "gb_post_render_fwd": (_i, [_i, _i, _i] + [_vp] * 8 + [_vp]),
    "gb_post_render_bwd": (_i, [_i, _i, _i] + [_vp] * 12 + [_vp]),
    "gb_ssim_l1_fwd": (_i, [_i, _i, _i] + [_vp] * 7 + [_vp]),
    "gb_ssim_l1_bwd": (_i, [_i, _i, _i] + [_vp] * 8 + [_f, _f, _vp, _vp]),
    "gb_envmap_spec_fwd": (_i, [_i, _i, _i] + [_vp] * 6 + [_f, _vp, _vp]),
    "gb_envmap_spec_bwd": (_i, [_i, _i, _i] + [_vp] * 6 + [_f, _vp, _vp, _vp, _vp]),
    "gb_mvp_raymarch_bwd": (_i, [_i] * 4 + [_vp, _vp, _f] + [_vp] * 5 + [_i] * 3 + [_vp] + [_i] * 3 + [_vp] * 8
                            + [_i, _f, _f, _i, _i, _vp]),
}


class GoliathB200Error(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GoliathB200Error(
                "libgoliath_b200.so is not built (%s). Run `python -m goliath_b200.build`; there is no CPU "
                "fallback." % LIB_PATH
            )
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(err, what):
    if err != 0:
        raise GoliathB200Error("%s failed: CUDA error %d" % (what, err))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr(device=None):
    return torch.cuda.current_stream(device).cuda_stream


def check_input(t, name, dtype=torch.float32):
    """Same contract as the reference's CHECK_INPUT (extensions/sgutils/utils.h): CUDA + contiguous."""
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor" % name)
    if not t.is_contiguous():
        raise RuntimeError("%s must be contiguous" % name)
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError("%s must have dtype %s (got %s)" % (name, dtype, t.dtype))
