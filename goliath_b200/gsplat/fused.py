"""render_fused — project -> bin/sort -> pack -> one 4-channel blend, as a single autograd node (SURVEY.md §8f-1).

Equivalent, output for output, to the reference's call sequence in ca_code/utils/render_gsplat.py:41-106
(project_gaussians, rasterize rgb with opacity * compensation, rasterize depth-as-colour) — same kernels, same
arithmetic — but without the tensors that sequence materialises between the calls (`opacity * compensation[:, None]`,
`depths[:, None].expand(-1, 3)`, the second binning) and without their autograd glue in the backward."""
import os

import torch
from torch.autograd import Function

from .. import _lib
from .utils import _tile_bounds, _workspace, bin_and_sort_gaussians, compute_cumulative_intersects, key_bits

# sync-free mode: per-device overflow flag (int32 on the device, set by the bin-edges kernel when the intersection
# count exceeded the capacity of the buffers) — read it with check_overflow() at a point where a sync is acceptable
_OVERFLOW = {}

# binning of the sync-free path: "buckets" (csrc/splat_bin_tiles.cu) or "keysort" (csrc/splat_bin.cu, the gsplat-shaped
# pipeline: cumsum -> keys -> radix sort -> bin edges -> pack); identical outputs, the switch exists for A/B timing
BINNING = os.environ.get("GOLIATH_B200_BINNING", "buckets")
# sync-free path as two autograd nodes (projection | binning + blend), see render_fused_split; "0" keeps the single node
SPLIT = os.environ.get("GOLIATH_B200_RENDER_SPLIT", "1") != "0"
# records of the two-node path: "packed" (sorted 48-byte records materialised by the binning's gather, default) or "ranked"
# (the blend stages records by depth rank from a per-Gaussian table with 16-byte cp.async gathers: the binning loses its
# 31 us gather, but the forward goes from 74 to 132 us and the backward from 97 to 104 — measured, profiles/
# r02_bench_head_ranked.json; kept as an option because it holds 4x less memory per view for the backward)
RANKED = os.environ.get("GOLIATH_B200_RECORDS", "packed") == "ranked"


def _overflow_flag(dev):
    f = _OVERFLOW.get(dev.index)
    if f is None:
        f = torch.zeros(1, dtype=torch.int32, device=dev)
        _OVERFLOW[dev.index] = f
    return f


def check_overflow(device=None) -> bool:
    """True if any sync-free render on `device` since the last check dropped intersections (capacity too small).
    Synchronises; call it once per step / per epoch, not per render."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    f = _OVERFLOW.get(dev.index)
    if f is None:
        return False
    hit = bool(f.item())
    if hit:
        f.zero_()
    return hit


class _RenderFused(Function):
    @staticmethod
    def forward(ctx, means3d, scales, quats, opacity, colors, viewmat, background, glob_scale, fx, fy, cx, cy, img_height,
                img_width, clip_thresh, capacity):
        ins = [t.contiguous() for t in (means3d, scales, quats, opacity, colors, viewmat, background)]
        for t, n in zip(ins, ("means3d", "scales", "quats", "opacity", "colors", "viewmat", "background")):
            _lib.check_input(t, n)
        means3d, scales, quats, opacity, colors, viewmat, background = ins
        G = means3d.size(0)
        if G == 0:
            capacity = None  # nothing to bin: the exact path below returns the background (no device-side count to read)
        dev = means3d.device
        L = _lib.lib()
        f32 = dict(device=dev, dtype=torch.float32)
        i32 = dict(device=dev, dtype=torch.int32)
        cov3d, xys, depths = torch.empty(G, 6, **f32), torch.empty(G, 2, **f32), torch.empty(G, **f32)
        radii, conics, comp = torch.empty(G, **i32), torch.empty(G, 3, **f32), torch.empty(G, **f32)
        num_tiles_hit = torch.empty(G, **i32)
        H, W, BW = int(img_height), int(img_width), 16
        out4 = torch.empty(H, W, 4, **f32)
        final_Ts = torch.empty(H, W, **f32)
        final_idx = torch.empty(H, W, **i32)
        bg4 = torch.cat([background, background[:1]])
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            _lib.check(L.gb_project_gaussians_fwd(
                G, _lib.ptr(means3d), _lib.ptr(scales), float(glob_scale), _lib.ptr(quats), _lib.ptr(viewmat), float(fx),
                float(fy), float(cx), float(cy), H, W, BW, float(clip_thresh), _lib.ptr(cov3d), _lib.ptr(xys),
                _lib.ptr(depths), _lib.ptr(radii), _lib.ptr(conics), _lib.ptr(comp), _lib.ptr(num_tiles_hit), st),
                "project_gaussians_forward")
            tb = _tile_bounds(H, W, BW)
            T = tb[0] * tb[1]
            # blend modes 2 and 4: the tile order is an SM-affine schedule and the blend kernels draw their tiles from it
            sched = 1 if (capacity is not None and L.gb_get_blend_mode() in (2, 4)) else 0
            if capacity is not None:
                # ---- sync-free path: the count never visits the host; buffers hold `capacity` intersections
                cap = int(capacity)
                gids = torch.empty(cap, **i32)
                order = torch.empty(L.gb_tile_schedule_ints(T) if sched else T, **i32)
                records = torch.empty(cap, 12, **f32)
                if BINNING == "buckets" and L.gb_bin_tiles_supported(G):
                    # per-tile buckets, each sorted on chip by (depth key, id) (csrc/splat_bin_tiles.cu): same bins,
                    # ids and records as the key sort below, without a global sort of the intersection keys
                    bins = torch.empty(T, 2, **i32)
                    ws = _workspace(dev, L.gb_bin_tiles_workspace_bytes(G, T, cap))
                    _lib.check(L.gb_bin_tiles_pack(G, _lib.ptr(xys), _lib.ptr(depths), _lib.ptr(radii),
                                                   _lib.ptr(conics), _lib.ptr(colors), _lib.ptr(opacity),
                                                   _lib.ptr(comp), H, W, BW, cap, _lib.ptr(bins), _lib.ptr(order),
                                                   sched, _lib.ptr(gids), _lib.ptr(records), None,
                                                   _lib.ptr(_overflow_flag(dev)), _lib.ptr(ws), st), "bin_tiles_pack")
                else:
                    cum = torch.empty_like(num_tiles_hit)
                    ws = _workspace(dev, max(L.gb_cumsum_workspace_bytes(G), L.gb_sort_workspace_bytes(cap)))
                    _lib.check(L.gb_cumsum_i32(G, _lib.ptr(num_tiles_hit), _lib.ptr(cum), _lib.ptr(ws), st), "cumsum")
                    n_dev = cum.data_ptr() + 4 * (G - 1)
                    isect = torch.empty(cap, device=dev, dtype=torch.int64)
                    gids_u = torch.empty(cap, **i32)
                    isect_s = torch.empty(cap, device=dev, dtype=torch.int64)
                    bins = torch.zeros(T, 2, **i32)
                    _lib.check(L.gb_map_gaussian_to_intersects_dn(G, _lib.ptr(xys), _lib.ptr(depths), _lib.ptr(radii),
                                                                  _lib.ptr(cum), H, W, BW, cap, _lib.ptr(isect),
                                                                  _lib.ptr(gids_u), st), "map_dn")
                    _lib.check(L.gb_sort_intersects_dn(cap, n_dev, _lib.ptr(isect), _lib.ptr(gids_u),
                                                       _lib.ptr(isect_s), _lib.ptr(gids), key_bits(T), _lib.ptr(ws),
                                                       st), "sort_dn")
                    _lib.check(L.gb_get_tile_bin_edges_dn(cap, n_dev, _lib.ptr(isect_s), _lib.ptr(bins),
                                                          _lib.ptr(_overflow_flag(dev)), st), "edges_dn")
                    _lib.check((L.gb_tile_schedule if sched else L.gb_tile_order)(T, _lib.ptr(bins), _lib.ptr(order), st),
                               "tile_order")
                    _lib.check(L.gb_pack_records_fused_dn(cap, n_dev, _lib.ptr(gids), _lib.ptr(xys), _lib.ptr(conics),
                                                          _lib.ptr(colors), _lib.ptr(depths), _lib.ptr(opacity),
                                                          _lib.ptr(comp), _lib.ptr(records), st),
                               "pack_records_fused_dn")
                _lib.check((L.gb_rasterize_sched_fwd if sched else L.gb_rasterize_packed_fwd)(
                    H, W, 4, _lib.ptr(bins), _lib.ptr(order), _lib.ptr(records), _lib.ptr(bg4), _lib.ptr(out4),
                    _lib.ptr(final_Ts), _lib.ptr(final_idx), st), "rasterize_packed_forward")
                num_intersects = cap  # "some": the backward walks the bins, not the count
            else:
                num_intersects, cum = compute_cumulative_intersects(num_tiles_hit)
            if capacity is not None:
                pass
            elif num_intersects < 1:
                # reference behaviour with nothing to draw (gsplat 0.1.11 rasterize.py): background, final_Ts = 0
                out4.copy_(bg4.expand(H, W, 4))
                final_Ts.zero_()
                final_idx.zero_()
                gids = bins = order = records = torch.empty(0, **i32)
            else:
                _, _, _, gids, bins = bin_and_sort_gaussians(G, num_intersects, xys, depths, radii, cum, tb, BW)
                order = torch.empty(T, **i32)
                records = torch.empty(num_intersects, 12, **f32)
                _lib.check(L.gb_tile_order(T, _lib.ptr(bins), _lib.ptr(order), st), "tile_order")
                _lib.check(L.gb_pack_records_fused(num_intersects, _lib.ptr(gids), _lib.ptr(xys), _lib.ptr(conics),
                                                   _lib.ptr(colors), _lib.ptr(depths), _lib.ptr(opacity), _lib.ptr(comp),
                                                   _lib.ptr(records), st), "pack_records_fused")
                _lib.check(L.gb_rasterize_packed_fwd(H, W, 4, _lib.ptr(bins), _lib.ptr(order), _lib.ptr(records),
                                                     _lib.ptr(bg4), _lib.ptr(out4), _lib.ptr(final_Ts),
                                                     _lib.ptr(final_idx), st), "rasterize_packed_forward")
        ctx.save_for_backward(means3d, scales, quats, opacity, viewmat, bg4, cov3d, radii, conics, comp, gids, bins, order,
                              records, final_Ts, final_idx)
        ctx.meta = (G, H, W, num_intersects, float(glob_scale), float(fx), float(fy), sched)
        ctx.mark_non_differentiable(radii)
        ctx.set_materialize_grads(False)
        return out4, 1 - final_Ts, radii

    @staticmethod
    def backward(ctx, v_out4, v_alpha, _v_radii):
        (means3d, scales, quats, opacity, viewmat, bg4, cov3d, radii, conics, comp, gids, bins, order, records, final_Ts,
         final_idx) = ctx.saved_tensors
        G, H, W, num_intersects, glob_scale, fx, fy, sched = ctx.meta
        dev = means3d.device
        L = _lib.lib()
        f32 = dict(device=dev, dtype=torch.float32)
        v_out4 = torch.zeros(H, W, 4, **f32) if v_out4 is None else v_out4.contiguous()
        v_alpha = None if v_alpha is None else v_alpha.contiguous()  # NULL: no gradient through alpha (no zero fill)
        acc = torch.zeros(G * 10, **f32)  # the four atomically-accumulated gradient arrays, one fill
        v_xy, v_conic = acc[:2 * G].view(G, 2), acc[2 * G:5 * G].view(G, 3)
        v_col4, v_opeff = acc[5 * G:9 * G].view(G, 4), acc[9 * G:]
        v_colors, v_opacity = torch.empty(G, 3, **f32), torch.empty(G, 1, **f32)
        v_comp, v_depth = torch.empty(G, **f32), torch.empty(G, **f32)
        g_cov2d, g_cov3d = torch.empty(G, 3, **f32), torch.empty(G, 6, **f32)
        g_mean, g_scale, g_quat = torch.empty(G, 3, **f32), torch.empty(G, 3, **f32), torch.empty(G, 4, **f32)
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            if num_intersects >= 1:
                _lib.check((L.gb_rasterize_sched_bwd if sched else L.gb_rasterize_packed_bwd)(
                    H, W, 4, _lib.ptr(gids), _lib.ptr(bins), _lib.ptr(order), _lib.ptr(records), _lib.ptr(bg4),
                    _lib.ptr(final_Ts), _lib.ptr(final_idx), _lib.ptr(v_out4), _lib.ptr(v_alpha), _lib.ptr(v_xy),
                    _lib.ptr(v_conic), _lib.ptr(v_col4), _lib.ptr(v_opeff), st), "rasterize_packed_backward")
            _lib.check(L.gb_splat_grad_unpack(G, _lib.ptr(v_col4), _lib.ptr(v_opeff), _lib.ptr(opacity), _lib.ptr(comp),
                                              _lib.ptr(v_colors), _lib.ptr(v_opacity), _lib.ptr(v_comp), _lib.ptr(v_depth),
                                              st), "splat_grad_unpack")
            _lib.check(L.gb_project_gaussians_bwd(
                G, _lib.ptr(means3d), _lib.ptr(scales), glob_scale, _lib.ptr(quats), _lib.ptr(viewmat), fx, fy,
                _lib.ptr(cov3d), _lib.ptr(radii), _lib.ptr(conics), _lib.ptr(comp), _lib.ptr(v_xy), _lib.ptr(v_depth),
                _lib.ptr(v_conic), _lib.ptr(v_comp), _lib.ptr(g_cov2d), _lib.ptr(g_cov3d), _lib.ptr(g_mean),
                _lib.ptr(g_scale), _lib.ptr(g_quat), st), "project_gaussians_backward")
        return (g_mean, g_scale, g_quat, v_opacity, v_colors) + (None,) * 11


class _ProjectGeom(Function):
    """First half of the sync-free fused render: projection only (no dependence on the colours)."""

    @staticmethod
    def forward(ctx, means3d, scales, quats, viewmat, glob_scale, fx, fy, cx, cy, img_height, img_width, clip_thresh):
        ins = [t.contiguous() for t in (means3d, scales, quats, viewmat)]
        for t, n in zip(ins, ("means3d", "scales", "quats", "viewmat")):
            _lib.check_input(t, n)
        means3d, scales, quats, viewmat = ins
        G = means3d.size(0)
        dev = means3d.device
        f32 = dict(device=dev, dtype=torch.float32)
        i32 = dict(device=dev, dtype=torch.int32)
        cov3d, xys, depths = torch.empty(G, 6, **f32), torch.empty(G, 2, **f32), torch.empty(G, **f32)
        radii, conics, comp = torch.empty(G, **i32), torch.empty(G, 3, **f32), torch.empty(G, **f32)
        num_tiles_hit = torch.empty(G, **i32)
        H, W = int(img_height), int(img_width)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gb_project_gaussians_fwd(
                G, _lib.ptr(means3d), _lib.ptr(scales), float(glob_scale), _lib.ptr(quats), _lib.ptr(viewmat), float(fx),
                float(fy), float(cx), float(cy), H, W, 16, float(clip_thresh), _lib.ptr(cov3d), _lib.ptr(xys),
                _lib.ptr(depths), _lib.ptr(radii), _lib.ptr(conics), _lib.ptr(comp), _lib.ptr(num_tiles_hit),
                _lib.stream_ptr(dev)), "project_gaussians_forward")
        ctx.save_for_backward(means3d, scales, quats, viewmat, cov3d, radii, conics, comp)
        ctx.meta = (G, float(glob_scale), float(fx), float(fy))
        ctx.mark_non_differentiable(radii)
        ctx.set_materialize_grads(False)
        return xys, depths, conics, comp, radii

    @staticmethod
    def backward(ctx, v_xy, v_depth, v_conic, v_comp, _v_radii):
        means3d, scales, quats, viewmat, cov3d, radii, conics, comp = ctx.saved_tensors
        G, glob_scale, fx, fy = ctx.meta
        dev = means3d.device
        f32 = dict(device=dev, dtype=torch.float32)

        def z(t, shape):
            return torch.zeros(shape, **f32) if t is None else t.contiguous()

        v_xy, v_depth, v_conic, v_comp = z(v_xy, (G, 2)), z(v_depth, (G,)), z(v_conic, (G, 3)), z(v_comp, (G,))
        g_cov2d, g_cov3d = torch.empty(G, 3, **f32), torch.empty(G, 6, **f32)
        g_mean, g_scale, g_quat = torch.empty(G, 3, **f32), torch.empty(G, 3, **f32), torch.empty(G, 4, **f32)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gb_project_gaussians_bwd(
                G, _lib.ptr(means3d), _lib.ptr(scales), glob_scale, _lib.ptr(quats), _lib.ptr(viewmat), fx, fy,
                _lib.ptr(cov3d), _lib.ptr(radii), _lib.ptr(conics), _lib.ptr(comp), _lib.ptr(v_xy), _lib.ptr(v_depth),
                _lib.ptr(v_conic), _lib.ptr(v_comp), _lib.ptr(g_cov2d), _lib.ptr(g_cov3d), _lib.ptr(g_mean),
                _lib.ptr(g_scale), _lib.ptr(g_quat), _lib.stream_ptr(dev)), "project_gaussians_backward")
        return (g_mean, g_scale, g_quat) + (None,) * 9


class _BinBlend(Function):
    """Second half: bucket binning + record packing + the 4-channel blend.  `colors` may still be in flight on another
    stream: `colors_event` (torch.cuda.Event recorded after the kernel that writes them) is waited for inside
    gb_bin_tiles_pack_ev just before the record gather, the first reader."""

    @staticmethod
    def forward(ctx, xys, depths, conics, comp, radii, opacity, colors, background, img_height, img_width, capacity,
                colors_event):
        opacity, colors, background = opacity.contiguous(), colors.contiguous(), background.contiguous()
        for t, n in zip((opacity, colors, background), ("opacity", "colors", "background")):
            _lib.check_input(t, n)
        G = xys.size(0)
        dev = xys.device
        L = _lib.lib()
        f32 = dict(device=dev, dtype=torch.float32)
        i32 = dict(device=dev, dtype=torch.int32)
        H, W, BW = int(img_height), int(img_width), 16
        out4 = torch.empty(H, W, 4, **f32)
        final_Ts = torch.empty(H, W, **f32)
        final_idx = torch.empty(H, W, **i32)
        bg4 = torch.cat([background, background[:1]])
        tb = _tile_bounds(H, W, BW)
        T = tb[0] * tb[1]
        cap = int(capacity)
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            sched = 1 if L.gb_get_blend_mode() in (2, 4) else 0
            order = torch.empty(L.gb_tile_schedule_ints(T) if sched else T, **i32)
            bins = torch.empty(T, 2, **i32)
            ws = _workspace(dev, L.gb_bin_tiles_workspace_bytes(G, T, cap))
            ev = None
            if colors_event is not None:
                ev = colors_event.cuda_event
                colors.record_stream(torch.cuda.current_stream(dev))
            # rank-staged records (default with the mom blend, launch-order tiles): the blend gathers each stage from the
            # by-rank table, the sorted 48-byte records are never materialised (csrc/splat_blend_mom.cu, RANKED)
            ranked = RANKED and not sched and L.gb_get_blend_mode() == 3
            if ranked:
                gids = torch.empty(G, **i32)            # rank -> Gaussian id
                ranks = torch.empty(cap, **i32)         # per tile: depth ranks in blend order
                records = torch.empty(G, 12, **f32)     # one record per Gaussian, by rank
                _lib.check(L.gb_bin_tiles_ranked(G, _lib.ptr(xys), _lib.ptr(depths), _lib.ptr(radii), _lib.ptr(conics),
                                                 _lib.ptr(colors), _lib.ptr(opacity), _lib.ptr(comp), H, W, BW, cap,
                                                 _lib.ptr(bins), _lib.ptr(order), sched, _lib.ptr(ranks),
                                                 _lib.ptr(records), _lib.ptr(gids), None, _lib.ptr(_overflow_flag(dev)),
                                                 _lib.ptr(ws), ev, st), "bin_tiles_ranked")
                _lib.check(L.gb_rasterize_ranked_fwd(H, W, 4, _lib.ptr(bins), _lib.ptr(order), _lib.ptr(ranks),
                                                     _lib.ptr(records), _lib.ptr(bg4), _lib.ptr(out4), _lib.ptr(final_Ts),
                                                     _lib.ptr(final_idx), st), "rasterize_ranked_forward")
            else:
                gids = torch.empty(cap, **i32)
                ranks = gids  # unused
                records = torch.empty(cap, 12, **f32)
                _lib.check(L.gb_bin_tiles_pack_ev(G, _lib.ptr(xys), _lib.ptr(depths), _lib.ptr(radii), _lib.ptr(conics),
                                                  _lib.ptr(colors), _lib.ptr(opacity), _lib.ptr(comp), H, W, BW, cap,
                                                  _lib.ptr(bins), _lib.ptr(order), sched, _lib.ptr(gids),
                                                  _lib.ptr(records), None, _lib.ptr(_overflow_flag(dev)), _lib.ptr(ws), ev,
                                                  st), "bin_tiles_pack_ev")
                _lib.check((L.gb_rasterize_sched_fwd if sched else L.gb_rasterize_packed_fwd)(
                    H, W, 4, _lib.ptr(bins), _lib.ptr(order), _lib.ptr(records), _lib.ptr(bg4), _lib.ptr(out4),
                    _lib.ptr(final_Ts), _lib.ptr(final_idx), st), "rasterize_packed_forward")
        ctx.save_for_backward(opacity, comp, bg4, gids, bins, order, records, final_Ts, final_idx, ranks)
        ctx.meta = (G, H, W, sched, ranked)
        ctx.set_materialize_grads(False)
        return out4, 1 - final_Ts

    @staticmethod
    def backward(ctx, v_out4, v_alpha):
        opacity, comp, bg4, gids, bins, order, records, final_Ts, final_idx, ranks = ctx.saved_tensors
        G, H, W, sched, ranked = ctx.meta
        dev = opacity.device
        L = _lib.lib()
        f32 = dict(device=dev, dtype=torch.float32)
        v_out4 = torch.zeros(H, W, 4, **f32) if v_out4 is None else v_out4.contiguous()
        v_alpha = None if v_alpha is None else v_alpha.contiguous()
        acc = torch.zeros(G * 10, **f32)  # the four atomically-accumulated gradient arrays, one fill
        v_xy, v_conic = acc[:2 * G].view(G, 2), acc[2 * G:5 * G].view(G, 3)
        v_col4, v_opeff = acc[5 * G:9 * G].view(G, 4), acc[9 * G:]
        v_colors, v_opacity = torch.empty(G, 3, **f32), torch.empty(G, 1, **f32)
        v_comp, v_depth = torch.empty(G, **f32), torch.empty(G, **f32)
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            if ranked:
                _lib.check(L.gb_rasterize_ranked_bwd(
                    H, W, 4, _lib.ptr(gids), _lib.ptr(ranks), _lib.ptr(bins), _lib.ptr(order), _lib.ptr(records),
                    _lib.ptr(bg4), _lib.ptr(final_Ts), _lib.ptr(final_idx), _lib.ptr(v_out4), _lib.ptr(v_alpha),
                    _lib.ptr(v_xy), _lib.ptr(v_conic), _lib.ptr(v_col4), _lib.ptr(v_opeff), st), "rasterize_ranked_backward")
            else:
                _lib.check((L.gb_rasterize_sched_bwd if sched else L.gb_rasterize_packed_bwd)(
                    H, W, 4, _lib.ptr(gids), _lib.ptr(bins), _lib.ptr(order), _lib.ptr(records), _lib.ptr(bg4),
                    _lib.ptr(final_Ts), _lib.ptr(final_idx), _lib.ptr(v_out4), _lib.ptr(v_alpha), _lib.ptr(v_xy),
                    _lib.ptr(v_conic), _lib.ptr(v_col4), _lib.ptr(v_opeff), st), "rasterize_packed_backward")
            _lib.check(L.gb_splat_grad_unpack(G, _lib.ptr(v_col4), _lib.ptr(v_opeff), _lib.ptr(opacity), _lib.ptr(comp),
                                              _lib.ptr(v_colors), _lib.ptr(v_opacity), _lib.ptr(v_comp), _lib.ptr(v_depth),
                                              st), "splat_grad_unpack")
        return (v_xy, v_depth, v_conic, v_comp, None, v_opacity, v_colors) + (None,) * 5


def render_fused_split(means3d, scales, glob_scale, quats, viewmat, fx, fy, cx, cy, img_height, img_width, opacity, colors,
                       background, clip_thresh, capacity, colors_event=None):
    """render_fused(capacity=N) as TWO autograd nodes — projection | binning + blend — with the same kernels.  What the
    split buys: the projection, the depth ranks, the tile buckets and the per-tile sort do not read the colours, so a
    caller that runs its shade on a side stream (and passes the event recorded after it) gets them beside the shade
    forward; in the backward autograd finds the projection backward and the shade backward independent (both only need
    this node's gradients) and issues them on their own streams.  Requires the bucket binning and G >= 1."""
    xys, depths, conics, comp, radii = _ProjectGeom.apply(means3d, scales, quats, viewmat, glob_scale, fx, fy, cx, cy,
                                                          img_height, img_width, clip_thresh)
    out4, alpha = _BinBlend.apply(xys, depths, conics, comp, radii, opacity, colors, background, img_height, img_width,
                                  capacity, colors_event)
    return out4, alpha, radii


def render_fused(means3d, scales, glob_scale, quats, viewmat, fx, fy, cx, cy, img_height, img_width, opacity, colors,
                 background, clip_thresh=0.01, capacity=None, colors_event=None):
    """Returns (out4 [H,W,4] = rgb + depth, alpha [H,W], radii [G] i32).  block_width is 16.

    capacity=None keeps the reference's behaviour (one host sync to size the intersection buffers exactly).
    capacity=N runs sync-free: buffers hold N intersections, the count stays on the device, nothing blocks the host, and
    the call can be captured in a CUDA graph; if a view ever needs more than N intersections the excess is dropped and
    `check_overflow()` reports it (results of that call are then incomplete — re-run with a larger capacity).  With
    zero intersections the sync-free path returns alpha = 0, not the reference's alpha = 1 quirk."""
    if (capacity is not None and SPLIT and BINNING == "buckets" and means3d.size(0) > 0
            and _lib.lib().gb_bin_tiles_supported(means3d.size(0))):
        return render_fused_split(means3d, scales, glob_scale, quats, viewmat, fx, fy, cx, cy, img_height, img_width,
                                  opacity, colors, background, clip_thresh, capacity, colors_event)
    if colors_event is not None:  # single-node path: the colours must be complete before the first kernel
        torch.cuda.current_stream(means3d.device).wait_event(colors_event)
    return _RenderFused.apply(means3d, scales, quats, opacity, colors, viewmat, background, glob_scale, fx, fy, cx, cy,
                              img_height, img_width, clip_thresh, capacity)
