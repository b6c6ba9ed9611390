"""CPU oracle for the goliath render hot path — TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import this package; nothing under ``goliath_b200/`` does (tests/test_layout.py enforces it).

numpy-in / numpy-out wrappers over ``liboracle.so`` (plain C, built by ``oracle/Makefile`` with
``-ffp-contract=off``).  Each C function cites the reference file:line it restates.

Parity status per path (also in DESIGN.md):
  * SG shade (sg_oracle.c)        — pinned on the GPU against recorded outputs of the reference kernels rebuilt
                                    into oracle/_ref (tests/golden/ref_kernels_sg.npz)
  * splat path (splat_oracle.c)   — PARITY UNPINNED: gsplat==0.1.11 is a third-party dependency absent from the
                                    reference checkout; restated from its published algorithm (SURVEY.md App. A)
  * raydirs / raymarch            — pinned on the GPU against recorded outputs of the reference kernels
                                    (tests/golden/ref_kernels_{mvp,raymarch}.npz) and against the reference's inline
                                    PyTorch raymarcher fixtures (tests/golden)
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force: bool = False) -> str:
    """Compile the C restatement (gcc, a second or two)."""
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("splat_oracle.c", "sg_oracle.c", "raymarch_oracle.c")]
    srcs = [s for s in srcs if os.path.exists(s)]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(
            ["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-Wall", "-o", so] + srcs + ["-lm"]
        )
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build())
        _LIB.orc_cumsum.restype = ctypes.c_int64
        _LIB.orc_num_threads.restype = ctypes.c_int
    return _LIB


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def set_num_threads(n):
    lib().orc_set_num_threads(int(n))


def num_threads():
    return int(lib().orc_num_threads())


# ----------------------------------------------------------------------------------------- splat path


def tile_bounds(H, W, bw):
    return (W + bw - 1) // bw, (H + bw - 1) // bw


def project_fwd(means3d, scales, glob_scale, quats, viewmat, fx, fy, cx, cy, H, W, block_width, clip_thresh=0.01):
    means3d, scales, quats = _f32(means3d), _f32(scales), _f32(quats)
    viewmat = _f32(np.asarray(viewmat).reshape(-1)[:12])
    G = means3d.shape[0]
    out = dict(
        cov3d=np.zeros((G, 6), np.float32), xys=np.zeros((G, 2), np.float32), depths=np.zeros(G, np.float32),
        radii=np.zeros(G, np.int32), conics=np.zeros((G, 3), np.float32), compensation=np.zeros(G, np.float32),
        num_tiles_hit=np.zeros(G, np.int32),
    )
    c = ctypes
    lib().orc_project_fwd(
        c.c_int(G), _p(means3d), _p(scales), c.c_float(glob_scale), _p(quats), _p(viewmat), c.c_float(fx),
        c.c_float(fy), c.c_float(cx), c.c_float(cy), c.c_int(H), c.c_int(W), c.c_int(block_width),
        c.c_float(clip_thresh), _p(out["cov3d"]), _p(out["xys"]), _p(out["depths"]), _p(out["radii"]),
        _p(out["conics"]), _p(out["compensation"]), _p(out["num_tiles_hit"]),
    )
    return out


def project_bwd(means3d, scales, glob_scale, quats, viewmat, fx, fy, cov3d, radii, conics, compensation,
                v_xy, v_depth, v_conic, v_compensation):
    means3d, scales, quats = _f32(means3d), _f32(scales), _f32(quats)
    viewmat = _f32(np.asarray(viewmat).reshape(-1)[:12])
    G = means3d.shape[0]
    out = dict(
        v_cov2d=np.zeros((G, 3), np.float32), v_cov3d=np.zeros((G, 6), np.float32),
        v_mean3d=np.zeros((G, 3), np.float32), v_scale=np.zeros((G, 3), np.float32),
        v_quat=np.zeros((G, 4), np.float32),
    )
    c = ctypes
    args = [_f32(cov3d), _i32(radii), _f32(conics), _f32(compensation), _f32(v_xy), _f32(v_depth), _f32(v_conic),
            _f32(v_compensation)]
    lib().orc_project_bwd(
        c.c_int(G), _p(means3d), _p(scales), c.c_float(glob_scale), _p(quats), _p(viewmat), c.c_float(fx),
        c.c_float(fy), *[_p(a) for a in args], _p(out["v_cov2d"]), _p(out["v_cov3d"]), _p(out["v_mean3d"]),
        _p(out["v_scale"]), _p(out["v_quat"]),
    )
    return out


def bin_and_sort(xys, depths, radii, num_tiles_hit, H, W, block_width):
    """cumsum -> map_gaussian_to_intersects -> stable sort -> tile bin edges (SURVEY.md App. A 'Binning')."""
    xys, depths, radii, nth = _f32(xys), _f32(depths), _i32(radii), _i32(num_tiles_hit)
    G = xys.shape[0]
    cum = np.zeros(G, np.int32)
    n = int(lib().orc_cumsum(ctypes.c_int(G), _p(nth), _p(cum)))
    isect = np.zeros(n, np.int64)
    gids = np.zeros(n, np.int32)
    lib().orc_map_to_intersects(ctypes.c_int(G), _p(xys), _p(depths), _p(radii), _p(cum), ctypes.c_int(H),
                                ctypes.c_int(W), ctypes.c_int(block_width), _p(isect), _p(gids))
    isect_s = np.zeros(n, np.int64)
    gids_s = np.zeros(n, np.int32)
    lib().orc_sort_intersects(ctypes.c_int64(n), _p(isect), _p(gids), _p(isect_s), _p(gids_s))
    tbx, tby = tile_bounds(H, W, block_width)
    bins = np.zeros((tbx * tby, 2), np.int32)
    lib().orc_tile_bin_edges(ctypes.c_int64(n), _p(isect_s), _p(bins))
    return dict(num_intersects=n, cum_tiles_hit=cum, isect_ids=isect, gaussian_ids=gids, isect_ids_sorted=isect_s,
                gaussian_ids_sorted=gids_s, tile_bins=bins)


def rasterize_fwd(H, W, block_width, gids_sorted, tile_bins, xys, conics, colors, opacities, background):
    colors = _f32(colors)
    C = colors.shape[1]
    assert C <= 8
    out_img = np.zeros((H, W, C), np.float32)
    final_Ts = np.zeros((H, W), np.float32)
    final_idx = np.zeros((H, W), np.int32)
    a = [_i32(gids_sorted), _i32(tile_bins), _f32(xys), _f32(conics), colors, _f32(np.asarray(opacities).reshape(-1)),
         _f32(background)]
    lib().orc_rasterize_fwd(ctypes.c_int(H), ctypes.c_int(W), ctypes.c_int(block_width), ctypes.c_int(C),
                            *[_p(x) for x in a], _p(out_img), _p(final_Ts), _p(final_idx))
    return out_img, final_Ts, final_idx


def rasterize_bwd(H, W, block_width, gids_sorted, tile_bins, xys, conics, colors, opacities, background, final_Ts,
                  final_idx, v_output, v_output_alpha):
    colors = _f32(colors)
    G, C = colors.shape
    v_xy = np.zeros((G, 2), np.float32)
    v_conic = np.zeros((G, 3), np.float32)
    v_colors = np.zeros((G, C), np.float32)
    v_opacity = np.zeros((G, 1), np.float32)
    a = [_i32(gids_sorted), _i32(tile_bins), _f32(xys), _f32(conics), colors, _f32(np.asarray(opacities).reshape(-1)),
         _f32(background), _f32(final_Ts), _i32(final_idx), _f32(v_output), _f32(v_output_alpha)]
    lib().orc_rasterize_bwd(ctypes.c_int(G), ctypes.c_int(H), ctypes.c_int(W), ctypes.c_int(block_width),
                            ctypes.c_int(C), *[_p(x) for x in a], _p(v_xy), _p(v_conic), _p(v_colors), _p(v_opacity))
    return v_xy, v_conic, v_colors, v_opacity


# ----------------------------------------------------------------------------------------- SG shade


def sg_fwd(lobe_dirs, lobe_sigmas, light_values, light_pts, prim_pts, n_lights, w_type=0):
    lobe_dirs = _f32(lobe_dirs)
    N, D = lobe_dirs.shape[:2]
    light_values = _f32(light_values)
    L = light_values.shape[1]
    out = np.zeros((N, D, 3), np.float32)
    a = [lobe_dirs, _f32(np.asarray(lobe_sigmas).reshape(N, D)), light_values, _f32(light_pts), _f32(prim_pts),
         _i32(n_lights)]
    lib().orc_sg_fwd(ctypes.c_int(N), ctypes.c_int(D), ctypes.c_int(L), *[_p(x) for x in a], _p(out),
                     ctypes.c_int(w_type))
    return out


def sg_bwd(lobe_dirs, lobe_sigmas, light_values, light_pts, prim_pts, n_lights, grad_integral, w_type=0,
           want_light_grad=True):
    lobe_dirs = _f32(lobe_dirs)
    N, D = lobe_dirs.shape[:2]
    light_values = _f32(light_values)
    L = light_values.shape[1]
    gd = np.zeros((N, D, 3), np.float32)
    gs = np.zeros((N, D), np.float32)
    gl = np.zeros((N, L, 3), np.float32) if want_light_grad else None
    a = [lobe_dirs, _f32(np.asarray(lobe_sigmas).reshape(N, D)), light_values, _f32(light_pts), _f32(prim_pts),
         _i32(n_lights), _f32(grad_integral)]
    lib().orc_sg_bwd(ctypes.c_int(N), ctypes.c_int(D), ctypes.c_int(L), *[_p(x) for x in a], _p(gd), _p(gs), _p(gl),
                     ctypes.c_int(w_type))
    return gd, gs, gl


# ----------------------------------------------------------------------------------------- MVP raymarch path


def raydirs_fwd(viewpos, viewrot, focal, princpt, pixelcoords, volradius, H=None, W=None):
    """compute_raydirs (extensions/utils/utils_kernel.cu:11-51). pixelcoords [N,H,W,2] or None (then H, W given)."""
    viewpos, viewrot, focal, princpt = _f32(viewpos), _f32(viewrot), _f32(focal), _f32(princpt)
    N = viewpos.shape[0]
    if pixelcoords is not None:
        pixelcoords = _f32(pixelcoords)
        H, W = pixelcoords.shape[1:3]
    raypos = np.zeros((N, H, W, 3), np.float32)
    raydir = np.zeros((N, H, W, 3), np.float32)
    tminmax = np.zeros((N, H, W, 2), np.float32)
    lib().orc_raydirs_fwd(ctypes.c_int(N), ctypes.c_int(H), ctypes.c_int(W), _p(viewpos), _p(viewrot), _p(focal),
                          _p(princpt), _p(pixelcoords), ctypes.c_float(volradius), _p(raypos), _p(raydir), _p(tminmax))
    return raypos, raydir, tminmax


def compute_aabb_fixedorder(primpos, primrot, primscale):
    primpos, primrot, primscale = _f32(primpos), _f32(primrot), _f32(primscale)
    N, K = primpos.shape[:2]
    aabb = np.zeros((N, 2 * K - 1, 2, 3), np.float32)
    lib().orc_compute_aabb_fixedorder(ctypes.c_int(N), ctypes.c_int(K), _p(primpos), _p(primrot), _p(primscale), _p(aabb))
    return aabb


def _rm_common(raypos, raydir, tminmax, primpos, primrot, primscale, template, warp):
    raypos, raydir, tminmax = _f32(raypos), _f32(raydir), _f32(tminmax)
    primpos, primrot, primscale, template = _f32(primpos), _f32(primrot), _f32(primscale), _f32(template)
    N, H, W = raypos.shape[:3]
    K = primpos.shape[1]
    TD, TH, TW = template.shape[2:5]
    assert template.shape[-1] == 4, "channels-last template [N,K,TD,TH,TW,4]"
    if warp is not None:
        warp = _f32(warp)
        WD, WH, WW = warp.shape[2:5]
    else:
        WD = WH = WW = 0
    aabb = compute_aabb_fixedorder(primpos, primrot, primscale)
    return raypos, raydir, tminmax, primpos, primrot, primscale, template, warp, aabb, (N, H, W, K, TD, TH, TW, WD, WH, WW)


def raymarch_fwd(raypos, raydir, stepsize, tminmax, primpos, primrot, primscale, template, warp=None, algo=0,
                 fadescale=8.0, fadeexp=8.0, blocksize=(8, 16), with_shadow=False):
    """mvpraymarch forward, usebvh='fixedorder' (extensions/mvpraymarch/mvpraymarch.py:91-220)."""
    (raypos, raydir, tminmax, primpos, primrot, primscale, template, warp, aabb,
     (N, H, W, K, TD, TH, TW, WD, WH, WW)) = _rm_common(raypos, raydir, tminmax, primpos, primrot, primscale, template, warp)
    rayrgba = np.zeros((N, H, W, 4), np.float32)
    raysat = np.full((N, H, W, 3), -1, np.float32)
    shadow = np.zeros((N, K, TD, TH, TW, 2), np.float32) if with_shadow else None
    c = ctypes
    lib().orc_raymarch_fwd(
        c.c_int(N), c.c_int(H), c.c_int(W), c.c_int(K), _p(raypos), _p(raydir), c.c_float(stepsize), _p(tminmax),
        _p(aabb), _p(primpos), _p(primrot), _p(primscale), c.c_int(TD), c.c_int(TH), c.c_int(TW), _p(template),
        c.c_int(WD), c.c_int(WH), c.c_int(WW), _p(warp), _p(rayrgba), _p(raysat), _p(shadow), c.c_int(algo),
        c.c_float(fadescale), c.c_float(fadeexp), c.c_int(blocksize[0]), c.c_int(blocksize[1]))
    return rayrgba, raysat, shadow


def raymarch_bwd(raypos, raydir, stepsize, tminmax, primpos, primrot, primscale, template, warp, raysat, grad_rayrgba,
                 algo=0, fadescale=8.0, fadeexp=8.0, blocksize=(8, 16)):
    (raypos, raydir, tminmax, primpos, primrot, primscale, template, warp, aabb,
     (N, H, W, K, TD, TH, TW, WD, WH, WW)) = _rm_common(raypos, raydir, tminmax, primpos, primrot, primscale, template, warp)
    g_pos, g_rot, g_scale = np.zeros_like(primpos), np.zeros_like(primrot), np.zeros_like(primscale)
    g_t = np.zeros_like(template)
    g_w = np.zeros_like(warp) if warp is not None else None
    c = ctypes
    lib().orc_raymarch_bwd(
        c.c_int(N), c.c_int(H), c.c_int(W), c.c_int(K), _p(raypos), _p(raydir), c.c_float(stepsize), _p(tminmax),
        _p(aabb), _p(primpos), _p(primrot), _p(primscale), c.c_int(TD), c.c_int(TH), c.c_int(TW), _p(template),
        c.c_int(WD), c.c_int(WH), c.c_int(WW), _p(warp), _p(_f32(raysat)), _p(_f32(grad_rayrgba)), _p(g_pos), _p(g_rot),
        _p(g_scale), _p(g_t), _p(g_w), c.c_int(algo), c.c_float(fadescale), c.c_float(fadeexp), c.c_int(blocksize[0]),
        c.c_int(blocksize[1]))
    return g_pos, g_rot, g_scale, g_t, g_w
