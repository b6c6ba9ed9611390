#!/usr/bin/env python
"""bench.py — rendered megapixels/s (fwd+bwd) of the RGCA shade+splat hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                     CPU restatement of the same path on the host cores

One "step" (default --config head) = one pass of the hot path over one view per rank of the BASELINE.json configs[1]
workload (300k Gaussians, 1 view 1024x667, L=32 point lights): SG specular shade + colour compose -> EWA projection ->
tile bin/sort -> alpha blend rgb + depth, forward AND backward (v_out = 1), through the reference-shaped Python surface
(goliath_b200.rgca_heads.shade_compose, goliath_b200.render.render_views).
`value` = views*H*W/1e6 / time with inputs resident in HBM; `e2e` = same through HOST buffers (H2D of the decoded
Gaussians from pinned memory + D2H of the rendered images inside the timed region; the gradients stay on the device
for the optimiser).  N>1: one view per rank (weak scaling), the frame owner (rank 0) broadcasts the decoded Gaussians
and gradients are all-reduced (goliath_b200.dist.FrameExchange), both inside the timed region.
--config olat | hand_mvp | mvp_full run BASELINE configs[2..4] with the same JSON schema.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, BW = 1024, 667, 16
NCOL = 19  # packed decoded Gaussian: pos3 quat4 scale3 opacity1 diff3 lobe3 sigma1 specvis1


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 200 for --config head, fewer for the heavier configs)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed warm-up steps (at least 3 are always run)")
    ap.add_argument("--config", default="head", choices=["head", "olat", "hand_mvp", "mvp_full"],
                    help="head = BASELINE configs[1] (the headline metric); olat = configs[2] (32 OLAT conditions x 16 views); "
                         "hand_mvp = configs[3] (4096 primitives, 8 cameras, decode + raymarch fwd+bwd); mvp_full = configs[4] "
                         "(256k primitives, 150 cameras)")
    ap.add_argument("--no-decoder", action="store_true", help="skip the `decoder` sub-object of the headline line")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gaussians", type=int, default=300_000)
    ap.add_argument("--lights", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager-sync", action="store_true", help="reference-like host path: exact buffers, one host sync per view")
    ap.add_argument("--no-graph", action="store_true", help="sync-free path without CUDA-graph capture")
    ap.add_argument("--mvp-density", type=float, default=2000.0, help="template alpha scale of the --ext-compare MVP scene")
    ap.add_argument("--decoder", action="store_true",
                    help="time the RGCA PrimDecoder forward at native size (1024^2 Gaussians): towers on tcgen05 vs SIMT, "
                         "fused heads kernel; prints its own JSON line")
    ap.add_argument("--decoder-library", action="store_true",
                    help="time the same decoder tower the reference's way (library conv_transpose2d + bias + LeakyReLU "
                         "passes, cuDNN); run under `timeout`: cuDNN may compile engines for minutes on a fresh box")
    ap.add_argument("--ext-compare", action="store_true",
                    help="time the reference's own extensions rebuilt for sm_100a (oracle/_ref) against ours: SG shade, "
                         "raydirs, MVP raymarch (BASELINE config 4 shape); prints its own JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (rendered images and the "
                         "gradients the step returns) as DIR/<name>.npy, at most 64 MB in all, for every --config of "
                         "--impl ours; one process only (--gpus 1): with more, each rank holds only its own views")
    a = ap.parse_args()
    if a.dump_outputs and (a.decoder or a.decoder_library or a.ext_compare or a.impl != "ours"):
        ap.error("--dump-outputs applies to the timed path of --impl ours (not --decoder / --decoder-library / "
                 "--ext-compare)")
    return a


FIELDS = (("primpos", 3), ("primqvec", 4), ("primscale", 3), ("opacity", 1), ("diff_color", 3), ("lobe_dirs", 3),
          ("sigma", 0), ("spec_vis", 1))  # width 0 = [G] vector


def packed_scene(G):
    """Flat fp32 buffer of G*19 floats holding the decoded Gaussians FIELD-MAJOR (each field contiguous, as the decoder
    heads kernel emits them), SURVEY.md §8d recipe, on the CPU.  One buffer = one H2D copy / one broadcast."""
    from goliath_b200 import synthetic

    sc = synthetic.head_gaussians(G)
    sh = synthetic.shade_inputs(G)
    g = torch.Generator().manual_seed(synthetic.SEED + 3)
    spec_vis = torch.sigmoid(torch.randn(G, 1, generator=g))
    parts = [sc["means3d"], sc["quats"], sc["scales"], sc["opacity"], sc["colors"], sh["lobe_dirs"][0],
             sh["lobe_sigmas"][0], spec_vis]
    return torch.cat([p.reshape(-1) for p in parts]).contiguous()


def unpack(flat, G=None):
    """Contiguous views (no copies) of the field-major buffer; works for torch tensors and numpy arrays."""
    G = flat.shape[0] // NCOL if G is None else G
    out, off = {}, 0
    for name, w in FIELDS:
        n = G * max(w, 1)
        v = flat[off:off + n]
        out[name] = v.reshape(G, w) if w else v
        off += n
    return out


# ------------------------------------------------------------------------------------------ GPU arm
# measured (profiles/r02_bench_head_shade_stream.json): the side stream costs 9 us per step on this workload — the shade is
# done before the latency-bound part of the binning starts, and the fork/join edges are not free; off by default
SHADE_STREAM = os.environ.get("GOLIATH_B200_SHADE_STREAM", "0") != "0"
HIGH_PRIO = os.environ.get("GOLIATH_B200_RENDER_PRIO", "0") != "0"


def _fused_mod():
    from goliath_b200.gsplat import fused
    return fused


def gpu_step(packed, cam, li, capacity=None):
    """forward + backward of shade + render for one view; returns (rgb, alpha, depth)."""
    from goliath_b200.render import render_views
    from goliath_b200.rgca_heads import shade_compose

    u = packed  # dict of leaf tensors (contiguous views of the flat buffer)
    # rgca.py:557-575: SG specular shade * spec_vis + clamped diffuse, clamped (one fused kernel each way).  Sync-free
    # path: the shade runs on a side stream beside the projection and the binning, which only need the colours at their
    # last kernel (render_views(color_event=...)); autograd runs its backward there too, beside the projection backward.
    ev = None
    if capacity is not None and SHADE_STREAM:
        from goliath_b200.render import shade_stream
        dev = u["primpos"].device
        main, side = torch.cuda.current_stream(dev), shade_stream(dev)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            color = shade_compose(u["lobe_dirs"][None], u["sigma"][None], li["light_intensity"], li["light_pos"],
                                  u["primpos"][None], li["n_lights"], u["diff_color"][None], u["spec_vis"][None])
            ev = torch.cuda.Event()
            ev.record(side)
    else:
        color = shade_compose(u["lobe_dirs"][None], u["sigma"][None], li["light_intensity"], li["light_pos"],
                              u["primpos"][None], li["n_lights"], u["diff_color"][None], u["spec_vis"][None])
    preds = dict(primpos=u["primpos"][None], primqvec=u["primqvec"][None], primscale=u["primscale"][None],
                 opacity=u["opacity"][None], color=color)
    rgb, alpha, depth = render_views(W, H, None, cam["Rt"], preds, intrinsics_host=[cam["intr"]], capacity=capacity,
                                     color_event=ev)
    torch.autograd.backward([rgb, depth], [_ones_like(rgb), _ones_like(depth)])  # v_out = 1 (SURVEY.md §8d)
    return rgb, alpha, depth


_ONES = {}


def _ones_like(t):
    key = (tuple(t.shape), t.device)
    o = _ONES.get(key)
    if o is None:
        o = _ONES[key] = torch.ones_like(t)
    return o


def sample_clocks_start(dev_index):
    f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
    q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    try:
        p = subprocess.Popen(["nvidia-smi", "-i", str(dev_index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                              "-lms", "100"], stdout=f, stderr=subprocess.DEVNULL)
    except OSError:
        return None, f.name
    return p, f.name


def sample_clocks_stop(p, path):
    out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    if p is not None:
        p.terminate()
        try:
            p.wait(timeout=5)
        except Exception:
            p.kill()
    try:
        rows = [r.strip().split(",") for r in open(path) if r.strip()]
        sm = [float(r[0]) for r in rows if r[0].strip().replace(".", "").isdigit()]
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(rows[0][1])
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for i, n in enumerate(names):
                if any(r[3 + i].strip().lower() == "active" for r in rows if len(r) >= 7):
                    out["reasons"].append(n)
            out["samples"] = len(sm)
    except Exception:
        pass
    finally:
        try:
            os.unlink(path)
        except OSError:
            pass
    return out


def kernel_roofline(dev, packed, cam, flush, sm_mhz=None):
    """Time the blend kernels alone through the C ABI (CUDA events on the launch stream, L2 flushed between
    launches) and report achieved ALGORITHMIC bytes/s (SURVEY.md §8d formulas) against the measured HBM peak."""
    from goliath_b200 import _lib
    from goliath_b200.gsplat import project_gaussians
    from goliath_b200.gsplat import utils as gu

    u = unpack(packed.detach())
    fx, fy, cx, cy = cam["intr"]
    xys, depths, radii, conics, comp, nth, cov3d = project_gaussians(
        u["primpos"].contiguous(), u["primscale"].contiguous(), 1.0, u["primqvec"].contiguous(), cam["Rt"][0], fx, fy,
        cx, cy, H, W, BW, 0.1)
    n, cum = gu.compute_cumulative_intersects(nth)
    tb = gu._tile_bounds(H, W, BW)
    _, _, _, gids, bins = gu.bin_and_sort_gaussians(xys.shape[0], n, xys, depths, radii, cum, tb, BW)
    C = 4  # the product path blends rgb + depth in one 4-channel pass (goliath_b200.render.render, fused=True)
    colors = torch.cat([u["diff_color"], depths[:, None]], 1).contiguous()
    opac = (u["opacity"] * comp[:, None]).contiguous()
    bg = torch.zeros(C, device=dev)
    out = torch.empty(H, W, C, device=dev)
    Ts = torch.empty(H, W, device=dev)
    fi = torch.empty(H, W, device=dev, dtype=torch.int32)
    G = xys.shape[0]
    v_out = torch.ones(H, W, C, device=dev)
    v_a = torch.zeros(H, W, device=dev)
    gx, gc, gcol, go = (torch.zeros(G, 2, device=dev), torch.zeros(G, 3, device=dev), torch.zeros(G, C, device=dev),
                        torch.zeros(G, 1, device=dev))
    L = _lib.lib()
    st = _lib.stream_ptr(dev)
    T_ = tb[0] * tb[1]
    rec = torch.empty(n, 12, device=dev)
    sched = 1 if L.gb_get_blend_mode() in (2, 4) else 0  # SM-affine schedule + the kernels that draw tiles from it
    order = torch.empty(L.gb_tile_schedule_ints(T_), dtype=torch.int32, device=dev)
    _lib.check((L.gb_tile_schedule if sched else L.gb_tile_order)(T_, bins.data_ptr(), order.data_ptr(), st), "order")
    ras_fwd = L.gb_rasterize_sched_fwd if sched else L.gb_rasterize_packed_fwd
    ras_bwd = L.gb_rasterize_sched_bwd if sched else L.gb_rasterize_packed_bwd

    def pack():
        _lib.check(L.gb_pack_records(n, C, gids.data_ptr(), xys.data_ptr(), conics.data_ptr(), colors.data_ptr(),
                                     opac.data_ptr(), rec.data_ptr(), st), "pack")

    def fwd():
        _lib.check(ras_fwd(H, W, C, bins.data_ptr(), order.data_ptr(), rec.data_ptr(), bg.data_ptr(),
                                             out.data_ptr(), Ts.data_ptr(), fi.data_ptr(), st), "fwd")

    def bwd():
        _lib.check(ras_bwd(H, W, C, gids.data_ptr(), bins.data_ptr(), order.data_ptr(),
                                             rec.data_ptr(), bg.data_ptr(), Ts.data_ptr(), fi.data_ptr(),
                                             v_out.data_ptr(), v_a.data_ptr(), gx.data_ptr(), gc.data_ptr(),
                                             gcol.data_ptr(), go.data_ptr(), st), "bwd")

    pack()
    # the product path (goliath_b200.gsplat.fused, blend mode 3): records staged by depth rank from the per-Gaussian
    # table, no sorted-record gather — time THOSE kernels and that binning when it is what the step runs
    from goliath_b200.gsplat import fused as _fused
    ranked = bool(_fused.RANKED and _fused.SPLIT and not sched and L.gb_get_blend_mode() == 3)
    cap_r = int(n) + 1024
    ranks_r = torch.empty(cap_r, dtype=torch.int32, device=dev)
    rbr_r = torch.empty(G, 12, device=dev)
    r2g_r = torch.empty(G, dtype=torch.int32, device=dev)
    bins_r = torch.empty(T_, 2, dtype=torch.int32, device=dev)
    order_r = torch.empty(T_, dtype=torch.int32, device=dev)
    ovf_r = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_r = torch.empty(L.gb_bin_tiles_workspace_bytes(G, T_, cap_r), dtype=torch.uint8, device=dev)
    col3_r, op1_r = u["diff_color"].contiguous(), u["opacity"].contiguous()

    def bin_ranked():
        _lib.check(L.gb_bin_tiles_ranked(G, xys.data_ptr(), depths.data_ptr(), radii.data_ptr(), conics.data_ptr(),
                                         col3_r.data_ptr(), op1_r.data_ptr(), comp.data_ptr(), H, W, BW, cap_r,
                                         bins_r.data_ptr(), order_r.data_ptr(), 0, ranks_r.data_ptr(), rbr_r.data_ptr(),
                                         r2g_r.data_ptr(), None, ovf_r.data_ptr(), ws_r.data_ptr(), None, st),
                   "bin_tiles_ranked")

    def fwd_ranked():
        _lib.check(L.gb_rasterize_ranked_fwd(H, W, C, bins_r.data_ptr(), order_r.data_ptr(), ranks_r.data_ptr(),
                                             rbr_r.data_ptr(), bg.data_ptr(), out.data_ptr(), Ts.data_ptr(), fi.data_ptr(),
                                             st), "ranked fwd")

    def bwd_ranked():
        _lib.check(L.gb_rasterize_ranked_bwd(H, W, C, r2g_r.data_ptr(), ranks_r.data_ptr(), bins_r.data_ptr(),
                                             order_r.data_ptr(), rbr_r.data_ptr(), bg.data_ptr(), Ts.data_ptr(),
                                             fi.data_ptr(), v_out.data_ptr(), v_a.data_ptr(), gx.data_ptr(), gc.data_ptr(),
                                             gcol.data_ptr(), go.data_ptr(), st), "ranked bwd")

    if ranked:
        bin_ranked()
        torch.cuda.synchronize()
        assert torch.equal(bins_r, bins) and torch.equal(r2g_r[ranks_r[:n].long()], gids) and int(ovf_r) == 0, \
            "ranked binning != key sort"
        # same colours as the packed records of this function (diffuse + depth)
        fwd_ranked()
    # the packed path's binning (sync-free): depth ranks + tile buckets + bitmap sort + record gather
    cap_b = int(n) + 1024
    col3, op1 = u["diff_color"].contiguous(), u["opacity"].contiguous()
    ws_b = torch.empty(L.gb_bin_tiles_workspace_bytes(G, T_, cap_b), dtype=torch.uint8, device=dev)
    bins_b = torch.empty(T_, 2, dtype=torch.int32, device=dev)
    order_b = torch.empty(L.gb_tile_schedule_ints(T_), dtype=torch.int32, device=dev)
    gids_b = torch.empty(cap_b, dtype=torch.int32, device=dev)
    rec_b = torch.empty(cap_b, 12, device=dev)
    ovf_b = torch.zeros(1, dtype=torch.int32, device=dev)

    def bin_tiles():
        _lib.check(L.gb_bin_tiles_pack(G, xys.data_ptr(), depths.data_ptr(), radii.data_ptr(), conics.data_ptr(),
                                       col3.data_ptr(), op1.data_ptr(), comp.data_ptr(), H, W, BW, cap_b,
                                       bins_b.data_ptr(), order_b.data_ptr(), sched, gids_b.data_ptr(), rec_b.data_ptr(), None,
                                       ovf_b.data_ptr(), ws_b.data_ptr(), st), "bin_tiles_pack")

    bin_tiles()
    torch.cuda.synchronize()
    assert torch.equal(bins_b, bins) and torch.equal(gids_b[:n], gids) and int(ovf_b) == 0, "bucket binning != key sort"

    def timeit(fn, reps=20):
        ts = []
        for _ in range(3):
            fn()
        for _ in range(reps):
            flush()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.mean(ts))

    t_p, t_f, t_b, t_bin = timeit(pack), timeit(fwd), timeit(bwd), timeit(bin_tiles)
    t_fr = t_br = t_binr = None
    if ranked:
        t_fr, t_br, t_binr = timeit(fwd_ranked), timeit(bwd_ranked), timeit(bin_ranked)
    P, T, I = H * W, tb[0] * tb[1], n
    # SURVEY.md §8d per-unit figures, with C = 4 colour channels (rgb + depth in one pass)
    bytes_f = I * (4 + 24 + 4 * C) + P * (4 * C + 4 + 4) + T * 8
    bytes_b = I * (4 + 24 + 4 * C) + I * (4 * (C + 6)) + P * (8 + 4 * C + 4)
    bytes_p = I * (4 + 24 + 4 * C) + I * 48
    # binning: keys/ranks of G Gaussians through 4 radix passes + bbox reads twice, one rank written and read per
    # intersection, sorted id written and read, record gather + write
    bytes_bin = G * (4 * 16 + 2 * 16) + I * (8 + 8) + I * (24 + 4 * C) + I * 48
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    which = "measured" if "hbm_gbs" in peaks else "fallback"
    mode = int(L.gb_get_blend_mode())
    list_fwd = os.environ.get("GOLIATH_B200_BLEND_FWD", "list") != "rounds"
    fwd_name = ("blend_fwd_packed_kernel<4>", "blend_fwd_pipe_kernel<4>", "blend_fwd_pipe_kernel<4>",
                "blend_fwd_ilp_kernel<4, %d, 0>" % list_fwd, "blend_fwd_ilp_kernel<4, %d, 0>" % list_fwd)[mode]
    bwd_name = ("blend_bwd_packed_kernel<4>", "blend_bwd_pipe_kernel<4>", "blend_bwd_pipe_kernel<4>",
                "blend_bwd_mom_kernel<4, 0>", "blend_bwd_mom_kernel<4, 0>")[mode]
    ks = {
        fwd_name: {"ms": t_f, "alg_bytes": bytes_f, "gbs": bytes_f / t_f / 1e6},
        bwd_name: {"ms": t_b, "alg_bytes": bytes_b, "gbs": bytes_b / t_b / 1e6},
        "pack_records_kernel<4>": {"ms": t_p, "alg_bytes": bytes_p, "gbs": bytes_p / t_p / 1e6},
        "bin_tiles_pack (rank sort, buckets, bitmap sort, record gather)": {
            "ms": t_bin, "alg_bytes": bytes_bin, "gbs": bytes_bin / t_bin / 1e6},
    }
    if ranked:  # what the step runs; the packed kernels above stay as the comparison
        # algorithmic bytes of the ranked formulation: 4 B rank + 48 B record per intersection read by the blend (the
        # record comes from the 14.4 MB per-Gaussian table), no 48 B write + read of sorted records in the binning
        bytes_binr = G * (4 * 16 + 2 * 16) + I * (8 + 8) + G * 48
        ks["blend_fwd_ilp_kernel<4, 1, 1>"] = {"ms": t_fr, "alg_bytes": bytes_f, "gbs": bytes_f / t_fr / 1e6}
        ks["blend_bwd_mom_kernel<4, 1>"] = {"ms": t_br, "alg_bytes": bytes_b, "gbs": bytes_b / t_br / 1e6}
        ks["bin_tiles_ranked (rank sort, buckets, bitmap sort; no record gather)"] = {
            "ms": t_binr, "alg_bytes": bytes_binr, "gbs": bytes_binr / t_binr / 1e6}
    in_step = (lambda k: k.endswith(", 1, 1>") or k.endswith("<4, 1>")) if ranked else (lambda k: True)
    dom = max((k for k in ks if k.startswith("blend") and in_step(k)), key=lambda k: ks[k]["ms"])
    # DRAM bytes and warp instructions per launch of the dominant kernel come from the committed `ncu --set full`
    # capture of the same scene (profiles/r02_traffic.json, written by scripts/ncu_summary.py traffic; neither is
    # measurable live).  The blend is not HBM-bound at this operating point (DESIGN.md section 4): the second figure is
    # the bound that does apply, warp instructions / (SMs x 4 schedulers x SM clock x the live duration).
    traffic, ncu_note, issue = None, None, None
    for fname in ("r02_traffic.json", "r01_traffic.json"):
        try:
            caps = json.load(open(os.path.join(ROOT, "profiles", fname)))["kernels"]
            cap = caps[dom]
        except Exception:
            continue
        traffic = cap["dram_bytes"]
        ncu_note = {k: cap[k] for k in ("issue_active_pct", "sm_cycles_active_over_elapsed", "top_stalls") if k in cap}
        ncu_note["capture"] = "profiles/" + fname
        if cap.get("warp_inst") and sm_mhz:
            sms = torch.cuda.get_device_properties(dev).multi_processor_count

            def slot_frac(k):
                return caps[k]["warp_inst"] / (sms * 4 * sm_mhz * 1e6 * ks[k]["ms"] * 1e-3)

            issue = {"warp_inst": int(cap["warp_inst"]), "sm_mhz": sm_mhz, "sms": sms, "frac": slot_frac(dom),
                     "kernels": {k: slot_frac(k) for k in ks if k in caps and caps[k].get("warp_inst")}}
        break
    roof = {"bound": "hbm", "kernel": dom, "achieved": ks[dom]["gbs"], "peak": peak, "unit": "GB/s",
            "frac": ks[dom]["gbs"] / peak, "traffic": traffic, "issue_slot": issue, "ncu": ncu_note, "peak_source": which, "intersections": int(I),
            "kernels": ks}
    return roof


# ------------------------------------------------------------------------------------------ RGCA workloads (configs 2, 3)
def _count_intersections(packed, Rts, intrs):
    """(tile, Gaussian) intersections summed over the given views (one host sync; reporting only)."""
    from goliath_b200.gsplat import project_gaussians

    u = unpack(packed.detach())
    total = 0
    for Rt, (fx, fy, cx, cy) in zip(Rts, intrs):
        nth = project_gaussians(u["primpos"].contiguous(), u["primscale"].contiguous(), 1.0, u["primqvec"].contiguous(), Rt,
                                fx, fy, cx, cy, H, W, BW, 0.1)[5]
        total += int(nth.sum().item())
    return total


class HeadWorkload:
    """BASELINE configs[1]: 300k Gaussians, ONE view 1024x667 per rank (weak scaling), L = 32 point lights."""
    key, scaling = "head", "weak"

    def __init__(self, args, rank, world, dev):
        from goliath_b200 import synthetic

        self.args, self.rank, self.world, self.dev = args, rank, world, dev
        self.G = args.gaussians
        self.li = {k: v.to(dev) for k, v in synthetic.lights(args.lights).items()}
        c = synthetic.ring_camera(rank % 16, img_h=H, img_w=W)
        self.cam = dict(Rt=c["viewmat"][None].to(dev), intr=(c["fx"], c["fy"], c["cx"], c["cy"]))
        self.cap = None if args.eager_sync else max(8 * self.G, 1 << 20)
        self.views_local, self.images_per_view = 1, 1
        self.mp_per_step = world * H * W / 1e6
        self.metric = "rendered megapixels/sec (fwd+bwd) RGCA head 300k Gaussians"
        self.workload = ("rgca_example.yml head: %d Gaussians, 1 view %dx%d per GPU, L=%d lights, shade+project+bin/sort+"
                         "blend(rgb)+blend(depth) fwd+bwd" % (self.G, H, W, args.lights))
        self.extra = {"views_per_gpu": 1, "lights": args.lights}

    def intersections(self, packed):
        return _count_intersections(packed, [self.cam["Rt"][0]], [self.cam["intr"]])

    def compute(self, packed, grad_out=None):
        """forward + backward of one view from the flat decoded buffer; returns ([rgb, alpha, depth], flat grad).
        grad_out: write the flat gradient there (the exchange's reduction buffer) instead of a new tensor."""
        leaves = {k: v.detach().requires_grad_() for k, v in unpack(packed).items()}
        rgb, alpha, depth = gpu_step(leaves, self.cam, self.li, capacity=self.cap)
        parts = [leaves[k].grad.reshape(-1) for k, _ in FIELDS]  # flat dL/d(decoded), same layout
        grad = torch.cat(parts) if grad_out is None else torch.cat(parts, out=grad_out)
        return [rgb, alpha, depth], grad


class OlatWorkload:
    """BASELINE configs[2]: 300k Gaussians x 32 OLAT lighting conditions x 16 views, views sharded over the ranks (strong
    scaling: the frame is fixed).  Per view: ONE projection + ONE tile binning, 32 x (L=1 shade -> blend) against the shared
    bins (goliath_b200.gsplat.olat), forward and backward; the decoded table is broadcast, its gradient all-reduced."""
    key, scaling = "olat", "strong"
    N_VIEWS, N_COND = 16, 32

    def __init__(self, args, rank, world, dev):
        from goliath_b200 import synthetic
        from goliath_b200.dist import views_of_rank

        self.args, self.rank, self.world, self.dev = args, rank, world, dev
        self.G = args.gaussians
        li = synthetic.lights(self.N_COND)
        self.lint = [li["light_intensity"][:, c:c + 1].contiguous().to(dev) for c in range(self.N_COND)]
        self.lpos = [li["light_pos"][:, c:c + 1].contiguous().to(dev) for c in range(self.N_COND)]
        self.one = torch.ones(1, dtype=torch.int32, device=dev)
        self.views = views_of_rank(rank, world, self.N_VIEWS)
        cams = [synthetic.ring_camera(v, img_h=H, img_w=W) for v in self.views]
        self.Rt = torch.stack([c["viewmat"] for c in cams]).to(dev) if cams else torch.zeros(0, 3, 4, device=dev)
        self.intr = [(c["fx"], c["fy"], c["cx"], c["cy"]) for c in cams]
        self.cap = max(8 * self.G, 1 << 20)
        self.views_local, self.images_per_view = len(self.views), self.N_COND
        self.mp_per_step = self.N_VIEWS * self.N_COND * H * W / 1e6
        self.metric = "rendered megapixels/sec (fwd+bwd) RGCA OLAT relighting 300k Gaussians x 32 lights x 16 views"
        self.workload = ("RGCA relighting: %d Gaussians x %d OLAT lighting conditions x %d views (%dx%d) sharded over the "
                         "ranks; per view one projection + one tile binning, %d x (L=1 shade + blend) fwd+bwd"
                         % (self.G, self.N_COND, self.N_VIEWS, H, W, self.N_COND))
        self.extra = {"views_total": self.N_VIEWS, "views_this_rank": len(self.views), "conditions": self.N_COND}

    def intersections(self, packed):
        return _count_intersections(packed, list(self.Rt), self.intr)

    def compute(self, packed, grad_out=None):
        from goliath_b200.gsplat.olat import render_views_shared
        from goliath_b200.rgca_heads import shade_compose

        u = {k: v.detach().requires_grad_() for k, v in unpack(packed).items()}
        V = len(self.views)
        cols = [shade_compose(u["lobe_dirs"][None], u["sigma"][None], self.lint[c], self.lpos[c], u["primpos"][None], self.one,
                              u["diff_color"][None], u["spec_vis"][None])[0] for c in range(self.N_COND)]
        colors = torch.stack(cols)                                             # [C,G,3]
        geom = {k: u[k][None].expand(V, *u[k].shape) for k in ("primpos", "primqvec", "primscale", "opacity")}
        rgb, alpha, depth = render_views_shared(W, H, self.Rt, geom, colors[None].expand(V, *colors.shape), self.intr,
                                                capacity=self.cap)
        torch.autograd.backward([rgb, depth], [torch.ones_like(rgb), torch.ones_like(depth)])
        parts = [u[k].grad.reshape(-1) for k, _ in FIELDS]
        grad = torch.cat(parts) if grad_out is None else torch.cat(parts, out=grad_out)
        return [rgb, alpha, depth], grad


DUMP_BYTES = 64_000_000


def _dump_one_process(args, world):
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one process (each rank holds only its own views): "
                         "run it with --gpus 1")


def dump_outputs(out_dir, arrays):
    """Write the named tensors a caller of the timed step receives as out_dir/<name>.npy (float32).  When they exceed
    DUMP_BYTES, each is replaced by a fixed, seeded sample of its flattened elements (<name>.npy), gathered on the device,
    and the sampled flat indices (<name>_index.npy), the budget shared in proportion to the sizes."""
    total = sum(t.numel() for t in arrays.values())
    budget = DUMP_BYTES - 2 * 128 * len(arrays)  # .npy headers
    keep = 1.0 if total * 4 <= budget else budget / (total * 12.0)  # 4 B value + 8 B index per sampled element
    os.makedirs(out_dir, exist_ok=True)
    for k, t in arrays.items():
        t = t.detach()
        if keep < 1.0:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), int(t.numel() * keep), replace=False))
            np.save(os.path.join(out_dir, k + "_index.npy"), idx.astype(np.int64))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, k + ".npy"), t.float().cpu().numpy())


def head_outputs(imgs, grad):
    """The images and the per-field gradient (dL/d decoded Gaussians) one step of run_ours returns, by name."""
    arrays = dict(zip(("rgb", "alpha", "depth"), imgs))
    arrays.update(("grad_" + k, v) for k, v in unpack(grad, grad.numel() // NCOL).items())
    return arrays


def _timeit_events(fn, reps, flush=None):
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return ts


def run_ours(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # The two 22.8 MB collectives of a step run UNDER the neighbouring renders; what they cost the step is the SMs
        # NCCL's CTAs take from the blend, not their own duration.  Measured at N = 4 (profiles/r02_nccl_ctas_n4.txt):
        # 8 CTAs lengthen them to 0.15 + 0.20 ms (still hidden under the 0.4 ms render) and shorten the step by 5 %.
        # At N = 2 the library default is better by 2 % (profiles/r02_exchange_n2.txt); at N = 8 a cap of 16 gives 11 107
        # MP/s, 8 gives 9 797 and 4 gives 7 390 (profiles/r02_nccl_ctas_n8.txt): two CTAs per peer from N = 4.
        if world >= 4:
            os.environ.setdefault("NCCL_MAX_CTAS", str(2 * world))
        dist.init_process_group("nccl", device_id=dev)
    from goliath_b200 import _lib
    from goliath_b200.dist import FrameExchange

    lib = _lib.lib()
    _dump_one_process(args, world)
    wl = (OlatWorkload if args.config == "olat" else HeadWorkload)(args, rank, world, dev)
    G = wl.G
    steps = args.steps if args.steps is not None else (200 if wl.key == "head" else 10)
    warmup = args.warmup if args.warmup is not None else (10 if wl.key == "head" else 3)
    warmup = max(3, warmup)
    host_packed = packed_scene(G).pin_memory()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def flush():
        flush_buf.fill_(1)  # > 126 MB L2

    resident = host_packed.to(dev)
    cap = wl.cap
    static_in = torch.empty_like(resident)                    # the graph's input buffer (field-major decoded Gaussians)
    state = {"graph": None, "outs": None}

    def capture(inp, grad_out=None):
        """Capture compute(inp) once (sync-free path), after side-stream warm-up as torch requires."""
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                wl.compute(inp, grad_out)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        from goliath_b200.render import render_stream
        # (optionally) captured on a high-priority stream: see SHADE_STREAM / HIGH_PRIO above
        with torch.cuda.graph(g, stream=render_stream(dev) if HIGH_PRIO else None):
            outs = wl.compute(inp, grad_out)
        return g, outs

    def build_graph():
        state["graph"], state["outs"] = capture(static_in)

    def run_step():
        if state["graph"] is not None:
            state["graph"].replay()
            return state["outs"]
        return wl.compute(static_in)

    # one eager step to count this library's launches per step, then capture
    static_in.copy_(resident)
    outs0, _ = wl.compute(static_in)
    torch.cuda.synchronize()
    lib.gb_launch_count_reset()
    wl.compute(static_in)
    torch.cuda.synchronize()
    launches_per_step = int(lib.gb_launch_count())
    host_out = [torch.empty(t.shape).pin_memory() for t in outs0]
    host_out2 = [torch.empty(t.shape).pin_memory() for t in outs0]
    d2h = sum(t.numel() * 4 for t in outs0)
    del outs0
    if cap is not None and not args.no_graph:
        build_graph()

    # ---------------------------------------------------------------- N = 1 paths
    def timed_single(e2e, n_steps, n_warm):
        """per-step event pairs; e2e: the table comes from pinned host memory and the images go back, serially."""
        def one():
            static_in.copy_(host_packed if e2e else resident, non_blocking=True)
            imgs, grad = run_step()
            if e2e:
                for dst, src_t in zip(host_out, imgs):
                    dst.copy_(src_t, non_blocking=True)
            return imgs, grad
        last = None
        for _ in range(n_warm):
            one()
        torch.cuda.synchronize()
        lib.gb_launch_count_reset()
        evs = []
        t0 = time.perf_counter()
        for _ in range(n_steps):
            flush()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            last = one()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        per_step = [a.elapsed_time(b) for a, b in evs]
        return sum(per_step), per_step, time.perf_counter() - t0, last

    # ---------------------------------------------------------------- N > 1: the exchange steps (goliath_b200.dist)
    def timed_exchange(e2e, n_steps, n_warm):
        """The frame owner (rank 0) broadcasts frame i+1's decoded table and every rank's gradient of frame i is
        all-reduced, both on FrameExchange's communication stream under the neighbouring renders.  e2e: the OWNER's table
        comes from pinned host memory (the other ranks receive it over NVLink and copy nothing in), every rank's images go
        back to its pinned host buffers on a copy stream."""
        ex = FrameExchange(resident.numel(), dev, owner=0)
        src = (host_packed if e2e else resident) if rank == 0 else None
        s_out = torch.cuda.Stream()
        main = torch.cuda.current_stream()
        # one captured graph per buffer parity: the step reads the exchange's input buffer and writes its flat gradient
        # into the exchange's reduction buffer, no device-to-device copy of either 22.8 MB table (GOLIATH_B200_EXCHANGE=copy
        # keeps the round-1 protocol: copy in, copy out)
        zero_copy = state["graph"] is not None and os.environ.get("GOLIATH_B200_EXCHANGE", "inplace") != "copy"
        pg = None
        if zero_copy:
            if "pgraphs" not in state:
                for k in range(2):
                    ex.inputs[k].copy_(resident)
                state["pgraphs"] = [capture(ex.inputs[k], ex.grads[k]) for k in range(2)]
                state["pgraphs_ex"] = ex
            else:  # graphs are bound to the first exchange's buffers: reuse it
                ex = state["pgraphs_ex"]
                ex.bytes_h2d = 0
            pg = state["pgraphs"]
        stage_out = [[torch.empty_like(t) for t in state["outs"][0]] for _ in range(2)] if e2e else None
        hosts = [host_out, host_out2]
        out_ready = [torch.cuda.Event() for _ in range(2)]
        out_free = [torch.cuda.Event() for _ in range(2)]

        def run(n, evs):
            ex.post_input(0, src)
            for i in range(n):
                k = i & 1
                flush()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                if zero_copy:
                    ex.wait_input(i)
                    if i + 1 < n:
                        ex.post_input(i + 1, src)
                    pg[k][0].replay()
                    imgs = pg[k][1][0]
                    ex.release_input(i)
                    ex.post_grad_inplace(i)
                else:
                    ex.take_input(i, static_in)
                    if i + 1 < n:
                        ex.post_input(i + 1, src)
                    imgs, grad = run_step()
                    ex.post_grad(i, grad)
                if e2e:
                    if i >= 2:
                        main.wait_event(out_free[k])
                    for dst, src_t in zip(stage_out[k], imgs):
                        dst.copy_(src_t, non_blocking=True)
                    out_ready[k].record(main)
                    with torch.cuda.stream(s_out):
                        s_out.wait_event(out_ready[k])
                        for dst, src_t in zip(hosts[k], stage_out[k]):
                            dst.copy_(src_t, non_blocking=True)
                        out_free[k].record(s_out)
                if i + 1 == n:
                    ex.finish()
                    main.wait_stream(s_out)
                b.record()
                evs.append((a, b))

        run(n_warm, [])
        torch.cuda.synchronize()
        dist.barrier()
        evs = []
        t0 = time.perf_counter()
        run(n_steps, evs)
        torch.cuda.synchronize()
        dist.barrier()
        wall = time.perf_counter() - t0
        per_step = [a.elapsed_time(b) for a, b in evs]
        return sum(per_step), per_step, wall, ex.bytes_h2d

    def timed_e2e_streamed_single(n_steps, n_warm):
        """N = 1, streamed: H2D of step i+1 and D2H of step i-1 on their own streams under step i's graph."""
        main = torch.cuda.current_stream()
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        stage_in = [torch.empty_like(resident) for _ in range(2)]
        stage_out = [[torch.empty_like(t) for t in state["outs"][0]] for _ in range(2)] if state["outs"] else None
        hosts = [host_out, host_out2]
        ev = lambda: [torch.cuda.Event() for _ in range(2)]
        in_ready, in_free, out_ready, out_free = ev(), ev(), ev(), ev()

        def h2d(i):
            k = i & 1
            with torch.cuda.stream(s_in):
                if i >= 2:
                    s_in.wait_event(in_free[k])
                stage_in[k].copy_(host_packed, non_blocking=True)
                in_ready[k].record(s_in)

        def run(n):
            h2d(0)
            for i in range(n):
                k = i & 1
                if i + 1 < n:
                    h2d(i + 1)
                flush()
                main.wait_event(in_ready[k])
                static_in.copy_(stage_in[k], non_blocking=True)
                in_free[k].record(main)
                imgs, _ = run_step()
                if stage_out is None:
                    for dst, src_t in zip(hosts[k], imgs):
                        dst.copy_(src_t, non_blocking=True)
                    continue
                if i >= 2:
                    main.wait_event(out_free[k])
                for dst, src_t in zip(stage_out[k], imgs):
                    dst.copy_(src_t, non_blocking=True)
                out_ready[k].record(main)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(out_ready[k])
                    for dst, src_t in zip(hosts[k], stage_out[k]):
                        dst.copy_(src_t, non_blocking=True)
                    out_free[k].record(s_out)
            main.wait_stream(s_out)

        run(n_warm)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run(n_steps)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def rank_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def rank_gather(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world == 1:
            return [float(x)]
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    proc = path = None
    if rank == 0:
        proc, path = sample_clocks_start(local)
    e2e_steps = max(min(steps, 20), steps // 4)
    collectives = None
    if world == 1:
        ms_total, per_step, wall, last = timed_single(False, steps, warmup)
        if args.dump_outputs:  # before the later phases reuse the graph's output buffers
            dump_outputs(args.dump_outputs, head_outputs(*last))
        del last
        ms_e2e_serial = timed_single(True, e2e_steps, 3)[0] * steps / e2e_steps
        ms_e2e = timed_e2e_streamed_single(steps, warmup)
        h2d_rank = host_packed.numel() * 4
    else:
        ms_total, per_step, wall, _ = timed_exchange(False, steps, warmup)
        ms_e2e, _, _, h2d_bytes = timed_exchange(True, steps, warmup)
        ms_e2e_serial = None
        h2d_rank = h2d_bytes // max(steps + warmup, 1)
        # the exchange steps alone (no render), on an idle machine: what has to be hidden under a step
        ex_t = resident.clone()
        torch.cuda.synchronize()
        dist.barrier()
        t_bc = float(np.median(_timeit_events(lambda: dist.broadcast(ex_t, src=0), 10)))
        t_ar = float(np.median(_timeit_events(lambda: dist.all_reduce(ex_t), 10)))
        collectives = {"broadcast_ms_alone": rank_max(t_bc), "allreduce_ms_alone": rank_max(t_ar),
                       "bytes": ex_t.numel() * 4}
    per_rank_isect = rank_gather(float(wl.intersections(resident)))
    own_ms = float(np.sum(per_step))
    ms_total = rank_max(ms_total)
    ms_e2e = rank_max(ms_e2e)
    per_rank_ms = rank_gather(own_ms / steps)
    h2d_per_rank = rank_gather(float(h2d_rank))
    # the render alone on this rank (no exchange, no copies): view heterogeneity vs collective cost
    torch.cuda.synchronize()
    render_only = float(np.mean(_timeit_events(lambda: run_step(), 10, flush)))
    per_rank_render = rank_gather(render_only)
    clocks = sample_clocks_stop(proc, path) if rank == 0 else None

    mp_per_step = wl.mp_per_step
    value = mp_per_step * steps / (ms_total / 1e3)
    e2e_v = mp_per_step * steps / (ms_e2e / 1e3)

    overflow = False
    if cap is not None:
        from goliath_b200.gsplat.fused import check_overflow
        overflow = check_overflow(dev)
    roof = cpu = dec = None
    if rank == 0 and wl.key == "head":
        roof = kernel_roofline(dev, resident, wl.cam, flush, (clocks or {}).get("sm_mhz"))
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline(args, steps=3, warmup=3)
            try:
                cpu["decoder_shade"] = cpu_decoder_shade(args.lights)
            except Exception as e:  # the headline line must not depend on this extra
                cpu["decoder_shade"] = {"error": str(e)[:200]}
            try:
                cpu["mesh_vae_decoder"] = cpu_mesh_vae_decoder()
            except Exception as e:
                cpu["mesh_vae_decoder"] = {"error": str(e)[:200]}
        if world == 1 and not args.no_decoder:
            try:
                dec = decoder_summary(args, dev)
            except Exception as e:
                dec = {"error": str(e)[:300]}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": wl.metric, "value": value, "unit": "MP/s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps,
        "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict({"workload": wl.workload, "name": wl.key, "gaussians": G, "block_width": BW,
                        "l2": "flushed between timed steps (256 MiB write)", "parallelism": "view-shard x%d" % world,
                        "nccl_max_ctas": None if world == 1 else os.environ.get("NCCL_MAX_CTAS"),
                        "exchange": None if world == 1 else os.environ.get("GOLIATH_B200_EXCHANGE", "inplace"),
                        "collectives": (None if world == 1 else "goliath_b200.dist.FrameExchange: NCCL broadcast of frame "
                                        "i+1's decoded table from its owner and all-reduce of frame i's gradient on a "
                                        "communication stream under the neighbouring renders; only the owner reads its source"),
                        "host_path": ("eager, exact buffers, 1 host sync/view" if cap is None else
                                      ("sync-free (capacity %d intersections)%s" % (cap, "" if args.no_graph else
                                                                                      ", step captured in a CUDA graph"))),
                        "binning": os.environ.get("GOLIATH_B200_BINNING", "buckets"),
                        "records": ("staged by depth rank from the per-Gaussian table (no sorted-record gather)"
                                    if (_fused_mod().RANKED and _fused_mod().SPLIT and int(lib.gb_get_blend_mode()) == 3)
                                    else "sorted 48-byte records materialised by the binning"),
                        "autograd_nodes": "projection | binning + blend" if _fused_mod().SPLIT else "one fused node",
                        "shade_stream": bool(SHADE_STREAM),
                        "rank_sort": ["cooperative LSD (one launch, varying key bits only)", "4 radix passes",
                                      "2048 key buckets + in-bucket ranking (cooperative LSD fallback)"][int(lib.gb_get_rank_sort_mode())],
                        "tile_sort": ["bitmap sort per tile + grid-wide record gather", "one kernel per tile"][int(lib.gb_get_tile_sort_mode())],
                        "blend": ["batch (CTA-synchronous)", "pipe (warp-decoupled)", "affine (warp-decoupled, SM-affine "
                                  "tile schedule)", "mom (exact cull, 4-hit ILP forward, transposed-reduction backward)",
                                  "mom-affine (mom over the SM-affine tile schedule)"][int(lib.gb_get_blend_mode())],
                        "intersection_overflow": overflow}, **wl.extra),
        "e2e": {"value": e2e_v, "unit": "MP/s", "h2d_bytes_per_step": int(sum(h2d_per_rank)), "d2h_bytes_per_step": d2h * world,
                "ms_per_step": ms_e2e / steps,
                "how": ("streamed: H2D of step i+1 and D2H of step i-1 on copy streams under step i's graph; rendered images "
                        "(not gradients: they stay on the device for the optimiser) go back to pinned host memory; the timed "
                        "region includes the per-step 256 MiB L2 flush" if world == 1 else
                        "owner-only H2D of the decoded table, NCCL broadcast, render, gradient all-reduce, D2H of every "
                        "rank's images, double-buffered on communication / copy streams; per-step event pairs, max over ranks"),
                "serial_ms_per_step": None if ms_e2e_serial is None else ms_e2e_serial / steps,
                "h2d_bytes_per_rank": [int(x) for x in h2d_per_rank]},
        "gpu_launches": launches_per_step * steps, "clocks": clocks, "roofline": roof,
        "per_rank": {"ms_per_step": per_rank_ms, "render_only_ms": per_rank_render,
                     "intersections": [int(x) for x in per_rank_isect], "collectives": collectives},
    }
    if dec is not None:
        line["decoder"] = dec
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ MVP workloads (configs 4, 5)
def _mvp_dist_setup():
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    return world, rank, local, dev


def _ref_ext(name):
    import importlib.util

    so = os.path.join(ROOT, "oracle", "_ref", name + ".so")
    if not os.path.exists(so):
        return None
    spec = importlib.util.spec_from_file_location(name, so)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _raymarch_kernels_alone(dev, raypos, raydir, tminmax, transf, template, step, reps=5):
    """forward / backward raymarch kernels alone through the extension-module API (ours and, when oracle/_ref holds it,
    the reference's mvpraymarchlib rebuilt for sm_100a) on the same tensors: the extension-level ratio of north_star."""
    from goliath_b200 import mvpraymarchlib
    from goliath_b200.mvpraymarch import _fixedorder_topology

    N, Hh, Ww = raypos.shape[:3]
    K = transf[0].shape[1]
    sid, ch, par = _fixedorder_topology(N, K, dev)
    aabb = torch.empty(N, 2 * K - 1, 2, 3, device=dev)
    rgba = torch.empty(N, Hh, Ww, 4, device=dev)
    sat = torch.empty(N, Hh, Ww, 3, device=dev)
    grgba = torch.ones(N, Hh, Ww, 4, device=dev)
    gp, gr, gsc = (torch.zeros_like(t) for t in transf)
    gt = torch.zeros_like(template)
    res = {}
    for tag, lib in (("ours", mvpraymarchlib), ("reference", _ref_ext("mvpraymarchlib"))):
        if lib is None:
            continue
        lib.compute_aabb(*transf, sid, ch, par, aabb, 0)

        def fwd():
            sat.fill_(-1.0)
            lib.raymarch_forward(raypos, raydir, step, tminmax, sid, ch, aabb, *transf, template, None, rgba, sat, None, None, 0,
                                 False, 512, True, True, 8.0, 8.0, 0, 0.99, 3, 8, 16)

        def bwd():
            lib.raymarch_backward(raypos, raydir, step, tminmax, sid, ch, aabb, transf[0], gp, transf[1], gr, transf[2], gsc,
                                  template, gt, None, None, rgba, grgba, sat, None, 0, False, 512, True, True, 8.0, 8.0, 0, 0.99,
                                  3, 8, 16)

        fwd(); bwd()
        res["raymarch_fwd_ms_" + tag] = float(np.median(_timeit_events(fwd, reps)))
        res["raymarch_bwd_ms_" + tag] = float(np.median(_timeit_events(bwd, reps)))
        res["alpha_mean_" + tag] = float(rgba[..., 3].mean())
    if "raymarch_fwd_ms_reference" in res:
        res["ours_over_reference_fwd_bwd"] = ((res["raymarch_fwd_ms_reference"] + res["raymarch_bwd_ms_reference"])
                                              / (res["raymarch_fwd_ms_ours"] + res["raymarch_bwd_ms_ours"]))
    return res


def _mvp_roofline(N, K, T, P, ms_fwd, ms_bwd):
    """SURVEY.md section 8d: raymarch fwd bytes = N*(K*TD*TH*TW*16 + K*60 + (2K-1)*24) + N*P*(32 + 16 + 12); the backward
    adds the template-gradient RMW (K*TD*TH*TW*16*2) and reads the forward's outputs.  L2/latency-bound by design: the
    HBM fraction is reported, it is not the target."""
    vox = K * T[0] * T[1] * T[2]
    b_f = N * (vox * 16 + K * 60 + (2 * K - 1) * 24) + N * P * (32 + 16 + 12)
    b_b = N * (vox * 16 * 3 + K * 60 * 2 + (2 * K - 1) * 24) + N * P * (32 + 16 + 12 + 16)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    ks = {"raymarch_fwd_kernel": {"ms": ms_fwd, "alg_bytes": b_f, "gbs": b_f / ms_fwd / 1e6},
          "raymarch_bwd_kernel": {"ms": ms_bwd, "alg_bytes": b_b, "gbs": b_b / ms_bwd / 1e6}}
    dom = max(ks, key=lambda k: ks[k]["ms"])
    return {"bound": "hbm", "kernel": dom, "achieved": ks[dom]["gbs"], "peak": peak, "unit": "GB/s",
            "frac": ks[dom]["gbs"] / peak, "traffic": None, "peak_source": "measured" if "hbm_gbs" in peaks else "fallback",
            "note": "the march is L2/latency-bound (SURVEY.md section 8d): HBM fraction reported, not the target",
            "kernels": ks}


def run_hand_mvp(args):
    """BASELINE configs[3]: hand_mvp_example.yml — 4096 volumetric primitives (64x64 UV grid, 8x16x16 voxels each), 8 cameras
    1024x667, one step = PoseEncoder -> TransDecoder + alpha / rgb slab decoders -> primitive transforms -> slab->primitive
    re-layout -> ray generation -> mvpraymarch, forward + backward (loss = sum of the rendered rgba), as
    ca_code/models/hand_mvp.py:205-268 runs it (mesh/LBS front end replaced by a synthetic base frame)."""
    import torch.distributed as dist

    world, rank, local, dev = _mvp_dist_setup()
    from goliath_b200 import _lib, synthetic
    from goliath_b200 import mvpraymarch as mvr
    from goliath_b200 import utils as gutils
    from goliath_b200.dist import views_of_rank
    from goliath_b200.hand_mvp import DeconvContentDecoder, PoseEncoder, TransDecoder, prim_transforms, slabs_to_primrgba

    lib = _lib.lib()
    steps = args.steps if args.steps is not None else 10
    warmup = max(3, args.warmup if args.warmup is not None else 3)
    NCAM, K, T = 8, 4096, (8, 16, 16)
    cams = views_of_rank(rank, world, NCAM)
    B = len(cams)
    torch.manual_seed(4096)
    s = synthetic.mvp_scene(N=NCAM, side=64, T=(1, 1, 1), img_h=H, img_w=W, density=1.0)  # geometry + cameras only
    sel = torch.tensor(cams, dtype=torch.long)
    posbase = s["primpos"][sel].to(dev).contiguous()
    rotbase = s["primrot"][sel].to(dev).contiguous()
    cam = {k: s[k][sel].to(dev).contiguous() for k in ("viewpos", "viewrot", "focal", "princpt")}
    penc = PoseEncoder(54, 64, 64).to(dev)
    tdec = TransDecoder(64).to(dev)
    adec, rdec = DeconvContentDecoder(8, 64, 1).to(dev), DeconvContentDecoder(8, 66, 3).to(dev)
    with torch.no_grad():  # random-init weights; output biases set so the volume is semi-transparent and coloured
        adec.texbranch[-1].bias.fill_(float(args.mvp_density))
        rdec.texbranch[-1].bias.fill_(2.0)
    named = [("%s.%s" % (mn, pn), p) for mn, m in (("penc", penc), ("tdec", tdec), ("adec", adec), ("rdec", rdec))
             for pn, p in m.named_parameters()]
    params = [p for _, p in named]
    _dump_one_process(args, world)
    kept = {}
    gen = torch.Generator().manual_seed(54)
    host_pose = torch.randn(NCAM, 60, generator=gen)[sel].contiguous().pin_memory()
    host_cond = torch.rand(NCAM, 2, 64, 64, generator=gen)[sel].contiguous().pin_memory()  # view_cos_uv, ambient occlusion
    pose_d, cond_d = host_pose.to(dev), host_cond.to(dev)
    step_sz = 1.0 / 2000.0
    host_img = torch.empty(B, H, W, 4).pin_memory()

    def forward(pose, cond):
        joint = penc(pose)
        primpos, primrot, primscale = prim_transforms(tdec.raw(joint), posbase, rotbase, prim_scale=56.0)
        alpha_raw = adec(joint).view(B, 8, 1, 1024, 1024)
        rgb_raw = rdec(torch.cat([joint, cond], 1)).view(B, 8, 3, 1024, 1024)
        tpl = slabs_to_primrgba(rgb_raw, alpha_raw, (16, 16, 8), valid_prims=None, raw=True)
        raypos, raydir, tminmax = gutils.compute_raydirs(cam["viewpos"], cam["viewrot"], cam["focal"], cam["princpt"], (W, H), 1.0)
        out = mvr.mvpraymarch(raypos, raydir, step_sz, tminmax, (primpos, primrot, primscale), tpl, None)
        return out, (raypos, raydir, tminmax, primpos, primrot, primscale, tpl)

    def step(e2e, keep=False):
        if e2e:
            pose_d.copy_(host_pose, non_blocking=True)
            cond_d.copy_(host_cond, non_blocking=True)
        out, _ = forward(pose_d, cond_d)
        out.backward(_ones_like(out))
        if world > 1:
            flat = torch.cat([p.grad.reshape(-1) for p in params])
            dist.all_reduce(flat)
        if e2e:
            host_img.copy_(out.detach(), non_blocking=True)
        if keep:  # --dump-outputs: the last timed step's rendered rgba and parameter gradients
            kept.update({"rgba": out.detach()}, **{"grad_" + n: p.grad for n, p in named if p.grad is not None})
        for p in params:
            p.grad = None

    def timed(e2e, n, w):
        for _ in range(w):
            step(e2e)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        lib.gb_launch_count_reset()
        evs = []
        for i in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); step(e2e, keep=bool(args.dump_outputs) and not e2e and i == n - 1); b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        launches = int(lib.gb_launch_count())
        if world > 1:
            dist.barrier()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches

    proc = path = None
    if rank == 0:
        proc, path = sample_clocks_start(local)
    ms_total, launches = timed(False, steps, warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: torch.cat(v) if isinstance(v, list) else v for k, v in kept.items()})
        kept.clear()
    ms_e2e, _ = timed(True, steps, 3)
    clocks = sample_clocks_stop(proc, path) if rank == 0 else None
    ext = roof = None
    if rank == 0:
        with torch.no_grad():
            out, (raypos, raydir, tminmax, primpos, primrot, primscale, tpl) = forward(pose_d, cond_d)
        ext = _raymarch_kernels_alone(dev, raypos, raydir, tminmax, (primpos.contiguous(), primrot.contiguous(),
                                                                     primscale.contiguous()), tpl.contiguous(), step_sz)
        roof = _mvp_roofline(B, K, T, H * W, ext["raymarch_fwd_ms_ours"], ext["raymarch_bwd_ms_ours"])
        ext["alpha_mean_rendered"] = float(out[..., 3].mean())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    mp = NCAM * H * W / 1e6
    line = {
        "metric": "rendered megapixels/sec (fwd+bwd) hand-MVP 4096 primitives, 8 cameras", "value": mp * steps / (ms_total / 1e3),
        "unit": "MP/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "hand_mvp_example.yml: 4096 volumetric primitives (8x16x16 voxels), 8 cameras %dx%d, decode "
                               "(PoseEncoder, TransDecoder, alpha/rgb slab decoders) + slab->primitive + raydirs + mvpraymarch "
                               "fwd+bwd, stepsize 1/2000" % (H, W),
                   "name": "hand_mvp", "cameras": NCAM, "cameras_this_rank": B, "primitives": K, "template": list(T),
                   "l2": "inputs regenerated every step (1.07 GB of templates per 8 cameras: larger than L2)",
                   "parallelism": "camera-shard x%d" % world, "alpha_bias": args.mvp_density},
        "e2e": {"value": mp * steps / (ms_e2e / 1e3), "unit": "MP/s", "h2d_bytes_per_step": NCAM * (60 + 2 * 64 * 64) * 4,
                "d2h_bytes_per_step": NCAM * H * W * 4 * 4, "ms_per_step": ms_e2e / steps,
                "how": "pose + conditioning maps from pinned host memory, rendered rgba images back to pinned host memory, "
                       "serial inside each step; parameter gradients stay on the device"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "reference_extension": ext,
    }
    print(json.dumps(line))


def run_mvp_full(args):
    """BASELINE configs[4]: full-body MVP — 262 144 primitives (512x512 UV grid, 8x8x8 voxels each: a 2.1 GB template), 150
    cameras of one frame sharded over the ranks (19/18 per GPU at N = 8), one train step = ray generation + raymarch
    forward + backward per camera against the shared template, template / transform gradients accumulated over the
    cameras and all-reduced.  The frame owner broadcasts the template (SURVEY.md section 8e)."""
    import torch.distributed as dist

    world, rank, local, dev = _mvp_dist_setup()
    from goliath_b200 import _lib, synthetic
    from goliath_b200 import mvpraymarch as mvr
    from goliath_b200 import utils as gutils
    from goliath_b200.dist import views_of_rank

    lib = _lib.lib()
    steps = args.steps if args.steps is not None else 3
    warmup = max(3, args.warmup if args.warmup is not None else 3)
    NCAM, SIDE, T = 150, 512, (8, 8, 8)
    K = SIDE * SIDE
    cams = views_of_rank(rank, world, NCAM)
    V = len(cams)
    s = synthetic.mvp_scene(N=1, side=SIDE, T=(1, 1, 1), img_h=H, img_w=W, density=1.0)  # geometry of the frame
    primpos = s["primpos"].to(dev).requires_grad_()
    primrot = s["primrot"].to(dev).requires_grad_()
    primscale = s["primscale"].to(dev).requires_grad_()
    views = [synthetic.ring_camera((v * 7) % 16, radius=2.5, img_h=H, img_w=W) for v in cams]
    yoff = [0.15 * ((v % 5) - 2) for v in cams]  # five rings of cameras at different heights
    viewpos = torch.stack([c["campos"] + torch.tensor([0.0, y, 0.0]) for c, y in zip(views, yoff)]).to(dev)
    viewrot = torch.stack([c["viewmat"][:, :3] for c in views]).to(dev).contiguous()
    focal = torch.full((V, 2), 1.6 * min(H, W), device=dev)
    princpt = torch.tensor([[W / 2.0, H / 2.0]] * V, device=dev)
    # template generated on the device (2.1 GB): softplus(1.5 N(0,1)), alpha channel shifted and scaled by the density
    gen = torch.Generator(device=dev).manual_seed(262144)
    tpl = torch.nn.functional.softplus(1.5 * torch.randn(1, K, *T, 4, device=dev, generator=gen))
    tpl[..., 3] = torch.nn.functional.softplus(tpl[..., 3] * 0 + 1.5 * torch.randn(1, K, *T, device=dev, generator=gen) - 1.0) \
        * float(args.mvp_density)
    host_tpl = tpl.cpu().pin_memory() if rank == 0 else None
    tpl.requires_grad_()
    step_sz = 1.0 / 2000.0
    host_img = torch.empty(max(V, 1), H, W, 4).pin_memory()
    _dump_one_process(args, world)
    kept = {}

    def step(e2e, keep=False):
        outs = []
        if e2e:
            if rank == 0:
                tpl.data.copy_(host_tpl, non_blocking=True)   # the frame owner's decoded template arrives from the host
        if world > 1:
            dist.broadcast(tpl.data, src=0)                   # ... and goes to the view shards
        for i in range(V):
            raypos, raydir, tminmax = gutils.compute_raydirs(viewpos[i:i + 1], viewrot[i:i + 1], focal[i:i + 1],
                                                             princpt[i:i + 1], (W, H), 1.0)
            out = mvr.mvpraymarch(raypos, raydir, step_sz, tminmax, (primpos, primrot, primscale), tpl, None)
            out.backward(_ones_like(out))
            if e2e:
                host_img[i].copy_(out.detach()[0], non_blocking=True)
            if keep:
                outs.append(out.detach())
        if world > 1:
            for t in (tpl, primpos, primrot, primscale):
                if t.grad is None:
                    t.grad = torch.zeros_like(t)
            dist.all_reduce(tpl.grad)
            small = torch.cat([primpos.grad.reshape(-1), primrot.grad.reshape(-1), primscale.grad.reshape(-1)])
            dist.all_reduce(small)
        if keep:  # --dump-outputs: the last timed step's rendered rgba of every camera and the accumulated gradients
            kept.update(rgba=outs, grad_template=tpl.grad, grad_primpos=primpos.grad, grad_primrot=primrot.grad,
                        grad_primscale=primscale.grad)
        for t in (tpl, primpos, primrot, primscale):
            t.grad = None

    def timed(e2e, n, w):
        for _ in range(w):
            step(e2e)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        lib.gb_launch_count_reset()
        evs = []
        for i in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); step(e2e, keep=bool(args.dump_outputs) and not e2e and i == n - 1); b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        launches = int(lib.gb_launch_count())
        if world > 1:
            dist.barrier()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches

    proc = path = None
    if rank == 0:
        proc, path = sample_clocks_start(local)
    ms_total, launches = timed(False, steps, warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: torch.cat(v) if isinstance(v, list) else v for k, v in kept.items()})
        kept.clear()
    ms_e2e, _ = timed(True, steps, 3)
    clocks = sample_clocks_stop(proc, path) if rank == 0 else None
    ext = roof = None
    if rank == 0 and V > 0:
        with torch.no_grad():
            raypos, raydir, tminmax = gutils.compute_raydirs(viewpos[:1], viewrot[:1], focal[:1], princpt[:1], (W, H), 1.0)
        ext = _raymarch_kernels_alone(dev, raypos, raydir, tminmax, (primpos.detach(), primrot.detach(), primscale.detach()),
                                      tpl.detach(), step_sz, reps=3)
        roof = _mvp_roofline(1, K, T, H * W, ext["raymarch_fwd_ms_ours"], ext["raymarch_bwd_ms_ours"])
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    mp = NCAM * H * W / 1e6
    tpl_bytes = K * T[0] * T[1] * T[2] * 16
    line = {
        "metric": "rendered megapixels/sec (fwd+bwd) full-body MVP 256k primitives, 150 cameras", "value": mp * steps / (ms_total / 1e3),
        "unit": "MP/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "full-body MVP: 262144 primitives (8x8x8 voxels, 2.1 GB template), 150 cameras %dx%d of one frame, "
                               "raydirs + mvpraymarch fwd+bwd per camera against the shared template, gradients accumulated "
                               "and all-reduced" % (H, W),
                   "name": "mvp_full", "cameras": NCAM, "cameras_this_rank": V, "primitives": K, "template": list(T),
                   "l2": "template (2.1 GB) larger than L2", "parallelism": "camera-shard x%d (19/18 per GPU at 8)" % world,
                   "collectives": None if world == 1 else "NCCL broadcast of the template, all-reduce of its gradient (2.1 GB each)",
                   "alpha_scale": args.mvp_density},
        "e2e": {"value": mp * steps / (ms_e2e / 1e3), "unit": "MP/s", "h2d_bytes_per_step": tpl_bytes,
                "d2h_bytes_per_step": NCAM * H * W * 4 * 4, "ms_per_step": ms_e2e / steps,
                "how": "the frame owner's template from pinned host memory (then broadcast), every camera's rgba image back to "
                       "pinned host memory; gradients stay on the device"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "reference_extension": ext,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ CPU arm (oracle port)
def cpu_step(orc, P, cam, li):
    u = {k: np.ascontiguousarray(v) for k, v in unpack(P).items()}
    fx, fy, cx, cy = cam["intr"]
    V = cam["Rt"]
    nrm = u["lobe_dirs"] / np.linalg.norm(u["lobe_dirs"], axis=-1, keepdims=True)
    spec = orc.sg_fwd(nrm[None], u["sigma"][None], li["light_intensity"], li["light_pos"], u["primpos"][None],
                      li["n_lights"], 0)[0]
    color = np.maximum(np.maximum(u["diff_color"], 0) + spec * u["spec_vis"], 0).astype(np.float32)
    p = orc.project_fwd(u["primpos"], u["primscale"], 1.0, u["primqvec"], V, fx, fy, cx, cy, H, W, BW, 0.1)
    b = orc.bin_and_sort(p["xys"], p["depths"], p["radii"], p["num_tiles_hit"], H, W, BW)
    opac = (u["opacity"][:, 0] * p["compensation"]).astype(np.float32)
    z3 = np.zeros(3, np.float32)
    o1, T1, f1 = orc.rasterize_fwd(H, W, BW, b["gaussian_ids_sorted"], b["tile_bins"], p["xys"], p["conics"], color,
                                   opac, z3)
    dcol = np.repeat(p["depths"][:, None], 3, 1)
    o2, T2, f2 = orc.rasterize_fwd(H, W, BW, b["gaussian_ids_sorted"], b["tile_bins"], p["xys"], p["conics"], dcol,
                                   opac, z3)
    ones = np.ones((H, W, 3), np.float32)
    za = np.zeros((H, W), np.float32)
    inv_a = (1.0 / np.clip(1 - T2, 0.05, 1.0)).astype(np.float32)
    wd = np.zeros((H, W, 3), np.float32)
    wd[..., 0] = inv_a
    g1 = orc.rasterize_bwd(H, W, BW, b["gaussian_ids_sorted"], b["tile_bins"], p["xys"], p["conics"], color, opac, z3,
                           T1, f1, ones, za)
    g2 = orc.rasterize_bwd(H, W, BW, b["gaussian_ids_sorted"], b["tile_bins"], p["xys"], p["conics"], dcol, opac, z3,
                           T2, f2, wd, za)
    v_op = (g1[3] + g2[3])[:, 0]
    orc.project_bwd(u["primpos"], u["primscale"], 1.0, u["primqvec"], V, fx, fy, p["cov3d"], p["radii"], p["conics"],
                    p["compensation"], g1[0] + g2[0], g2[2].sum(1), g1[1] + g2[1], v_op * u["opacity"][:, 0])
    orc.sg_bwd(nrm[None], u["sigma"][None], li["light_intensity"], li["light_pos"], u["primpos"][None], li["n_lights"],
               (g1[2] * u["spec_vis"])[None], 0, want_light_grad=False)
    return b["num_intersects"]


def cpu_baseline(args, steps, warmup):
    import oracle
    from goliath_b200 import synthetic

    oracle.lib()
    cores = os.cpu_count() or 1
    oracle.set_num_threads(cores)
    P = packed_scene(args.gaussians).numpy()
    li = {k: v.numpy() for k, v in synthetic.lights(args.lights).items()}
    c = synthetic.ring_camera(0, img_h=H, img_w=W)
    cam = dict(Rt=c["viewmat"].numpy(), intr=(c["fx"], c["fy"], c["cx"], c["cy"]))
    for _ in range(warmup):
        cpu_step(oracle, P, cam, li)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_step(oracle, P, cam, li)
    dt = (time.perf_counter() - t0) / steps
    return {"value": H * W / 1e6 / dt, "unit": "MP/s", "cores": oracle.num_threads(), "kind": "port",
            "sample": "%d full step(s) of the same workload (1 view %dx%d, %d Gaussians, L=%d) through the C oracle "
                      "(oracle/*.c, OpenMP)" % (steps, H, W, args.gaussians, args.lights),
            "s_per_step": dt}


def cpu_decoder_shade(lights=32, slab=1024):
    """north_star's second CPU number: the reference's decoder + shade path as it runs without a GPU — PyTorch on the host
    cores (7-layer untied-bias deconv towers via conv_transpose2d, the head math of rgca.py:506-546 via the torch
    restatement oracle/heads_oracle.py, SG shade via the C oracle since the reference has no CPU kernel for it) —
    one frame at native size (slab^2 Gaussians), random weights of the real shapes.  Bounded: one frame, a few seconds."""
    import oracle
    from oracle import heads_oracle
    from goliath_b200 import synthetic

    th = torch
    th.set_num_threads(os.cpu_count() or 1)
    gen = th.Generator().manual_seed(3)
    plan = [256, 256, 128, 128, 64, 32, 16]

    def tower(cin0, cout_last):
        n_layers = int(round(np.log2(slab / 8)))  # 7 at the native 1024
        ws, bs, size, chans = [], [], 8, [cin0] + plan[1:n_layers] + [cout_last]
        for a_, b_ in zip(chans[:-1], chans[1:]):
            size *= 2
            ws.append(th.randn(a_, b_, 4, 4, generator=gen) * 0.05)
            bs.append(th.zeros(b_, size, size))
        return ws, bs

    def run_tower(x, ws, bs):
        h = x
        for i, (w_, b_) in enumerate(zip(ws, bs)):
            h = th.nn.functional.conv_transpose2d(h, w_, None, 2, 1) + b_[None]
            if i + 1 < len(ws):
                h = th.nn.functional.leaky_relu(h, 0.2)
        return h

    t1, t2 = tower(256, 125), tower(264, 4)
    x = th.randn(1, 256, 8, 8, generator=gen)
    xv = th.randn(1, 264, 8, 8, generator=gen)
    G = slab * slab
    shell = synthetic.head_gaussians(G)["means3d"]
    postex = shell.t().reshape(1, 3, slab, slab).contiguous()
    tn = th.nn.functional.normalize(shell, dim=1).t().reshape(1, 3, slab, slab).contiguous()
    albedo = th.rand(1, G, 3, generator=gen)
    light_sh = th.randn(1, 3, 81, generator=gen)
    campos = th.tensor([[0.0, 0.0, 1000.0]])
    li = {k: v.numpy() for k, v in synthetic.lights(lights).items()}
    oracle.lib()
    oracle.set_num_threads(os.cpu_count() or 1)
    t0 = time.perf_counter()
    with th.no_grad():
        f1, f2 = run_tower(x, *t1), run_tower(xv, *t2)
        t_dec = time.perf_counter() - t0
        heads = heads_oracle.gaussian_heads(f1, f2, postex, tn, albedo, light_sh, campos)
        t_heads = time.perf_counter() - t0 - t_dec
        spec = oracle.sg_fwd(np.ascontiguousarray(heads["ref_dirs"].numpy()), np.ascontiguousarray(heads["sigma"].numpy()),
                             li["light_intensity"], li["light_pos"], np.ascontiguousarray(heads["primpos"].numpy()),
                             li["n_lights"], 0)
        heads_oracle.compose_color(heads["diff_color"], th.from_numpy(spec) * heads["spec_vis"])
    dt = time.perf_counter() - t0
    return {"s_per_frame": dt, "decoder_s": t_dec, "heads_s": t_heads, "shade_s": dt - t_dec - t_heads, "gaussians": G,
            "lights": lights, "cores": os.cpu_count() or 1, "torch_threads": th.get_num_threads(),
            "gaussians_decoded_shaded_per_s": G / dt,
            "what": "PyTorch CPU decoder towers + head math (oracle restatement of rgca.py:506-546) + C-oracle SG shade, "
                    "1 frame, native size, random weights"}


def cpu_mesh_vae_decoder(frames=3):
    """BASELINE.json configs[0] / SURVEY.md §8 row R9: the reference's body decoder (mesh_vae.ConvDecoder, 58.7 M
    parameters, mesh_vae_example.yml) forward for one frame on the host cores — pure PyTorch, the case the reference
    itself can run without a GPU.  Timed on the restatement oracle/mesh_vae_oracle.py, which is pinned to the reference
    class by tests/golden/mesh_vae_ref.npz (identical outputs on identical weights).  Bounded: 1 warm-up + `frames`."""
    from oracle import mesh_vae_oracle as mo

    th = torch
    th.set_num_threads(os.cpu_count() or 1)
    dec = mo.seeded_fill(mo.ConvDecoder(mo.synthetic_masks(), mo.identity_resample, mo.uv_vertex_gather()))
    pose, embs, face = mo.seeded_inputs()
    ts = []
    with th.no_grad():
        dec(pose, embs, face)
        for _ in range(frames):
            t0 = time.perf_counter()
            dec(pose, embs, face)
            ts.append(time.perf_counter() - t0)
    return {"s_per_frame": float(np.median(ts)), "frames": frames, "params_M": sum(p.numel() for p in dec.parameters()) / 1e6,
            "cores": os.cpu_count() or 1, "torch_threads": th.get_num_threads(),
            "what": "mesh_vae.ConvDecoder forward, 1 frame, uv 1024 (mesh_vae_example.yml), PyTorch CPU, random weights; "
                    "seam sampler / from_uv replaced by bilinear gathers of the same shapes"}


def run_reference(args):
    """Reference arm: the reference has no CPU rasteriser (gsplat is a CUDA-only third-party dependency, absent), so the
    CPU implementation of the path is the oracle port, timed with all host threads.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    # honours --steps / --warmup (same counts as our arm asks for); one CPU step of this workload takes ~1 s on the
    # host cores of a B200 box, so the default (no flags) is a bounded 5 + 3
    steps = 5 if args.steps is None else max(1, args.steps)
    warmup = 3 if args.warmup is None else max(0, args.warmup)
    cpu = cpu_baseline(args, steps=steps, warmup=warmup)
    line = {
        "impl": "reference", "metric": "rendered megapixels/sec (fwd+bwd) RGCA head 300k Gaussians",
        "value": cpu["value"], "unit": "MP/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": cpu["s_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "rgca_example.yml head: %d Gaussians, 1 view %dx%d, L=%d lights, shade+project+bin/sort+"
                               "blend(rgb)+blend(depth) fwd+bwd" % (args.gaussians, H, W, args.lights),
                   "gaussians": args.gaussians, "lights": args.lights, "block_width": BW},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ decoder (rows R1 + R2)
def decoder_summary(args, dev):
    """The `decoder` sub-object of the headline line (rows R1 + R2 where the driver can see them): big tower on the tensor
    cores (graph replay), last layer alone, heads, training fwd+bwd of the big tower, decode+shade+render frame."""
    r = run_decoder(args, quick=True, dev=dev)["decoder"]
    keep = ("tower_vnocond_ms_tc_graph", "tower_vnocond_ms_simt", "last_layer_ms_simt", "last_layer_alg_GBs_simt",
            "last_layer_ms_tc16", "heads_ms", "heads_alg_GBs", "full_decoder_ms_tc_graph", "tower_vnocond_fwd_bwd_ms_simt",
            "frame_decode_shade_render_fwd_ms_graph", "frame_MP_per_s_fwd_graph", "tc_vs_simt_rel_err")
    out = {k: r[k] for k in keep if k in r}
    out["what"] = ("RGCA PrimDecoder at native size (1024^2 Gaussians, 162.8 M parameters, random init), B = 1; ms per call, "
                   "CUDA events, L2 flushed; last_layer = 16->125 @1024^2 on 1.07 GB of mandatory traffic")
    return out


def run_decoder(args, quick=False, dev=None):
    """Inference forward of the RGCA PrimDecoder at native size (B=1, 1024x1024 Gaussians, 162.8 M parameters,
    random init): the two 7-layer towers on the tensor cores (tcgen05 + TMA) and on the SIMT kernels, then the fused heads
    kernel and the SG shade.  Reports ms per part and the last layer's achieved HBM bandwidth on its mandatory bytes
    (SURVEY.md §8d: 2*Cout*H*W*4 + Cin*(H/2)*(W/2)*4)."""
    from goliath_b200 import nn as gnn
    from goliath_b200 import synthetic
    from goliath_b200.rgca import PrimDecoder
    from goliath_b200.rgca_heads import gaussian_heads, shade_and_compose

    if dev is None:
        dev = torch.device("cuda", 0)
        torch.cuda.set_device(dev)
    S = 1024

    class Geo:
        def __init__(self, pos, nml): self.pos, self.nml = pos, nml
        def to_uv(self, x): return x
        def vn(self, g): return self.nml

    gen = torch.Generator().manual_seed(1)
    shell = synthetic.head_gaussians(S * S)["means3d"]  # SURVEY.md §8d ellipsoid shell, as the posed-mesh UV map
    pos = shell.t().reshape(1, 3, S, S).contiguous().to(dev)
    nml = torch.nn.functional.normalize(shell, dim=1).t().reshape(1, 3, S, S).contiguous().to(dev)
    dec = PrimDecoder(256, Geo(pos, nml), 255 * torch.rand(3, S, S, generator=gen), slabsize=S).to(dev)
    dec.eval()  # inference timings: no training-mode random back light (rgca.py:590-618)
    with torch.no_grad():
        for n_, p in dec.named_parameters():
            if n_.endswith("bias"):
                p.normal_(0, 0.05)
    embs = torch.randn(1, 256, generator=gen).to(dev)
    campos = torch.tensor([[0.0, 0.0, 1000.0]], device=dev)
    li = {k: v.to(dev) for k, v in synthetic.lights(args.lights).items()}
    light_sh = torch.randn(1, 3, 81, generator=gen).to(dev)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timeit(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            flush_buf.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    res = {}
    with torch.no_grad():
        x = dec.encmod(embs).view(-1, 256, 8, 8)
        view = dec.viewmod(torch.nn.functional.normalize(campos, dim=1))[:, :, None, None].expand(-1, -1, 8, 8)
        xv = torch.cat([x, view], 1).contiguous()
        res["tower_vnocond_ms_tc"] = timeit(lambda: gnn.tower_forward_tc(dec.vnocond_mod, x))
        res["tower_vnocond_ms_simt"] = timeit(lambda: dec.vnocond_mod(x))
        res["tower_vcond_ms_tc"] = timeit(lambda: gnn.tower_forward_tc(dec.vcond_mod, xv))
        res["tower_vcond_ms_simt"] = timeit(lambda: dec.vcond_mod(xv))
        f1, f2 = gnn.tower_forward_tc(dec.vnocond_mod, x), gnn.tower_forward_tc(dec.vcond_mod, xv)
        g1 = dec.vnocond_mod(x)
        res["tc_vs_simt_rel_err"] = float((f1 - g1).norm() / g1.norm())
        tn = torch.nn.functional.normalize(nml, dim=1)
        res["heads_ms"] = timeit(lambda: gaussian_heads(f1, f2, pos, tn, dec.albedo, light_sh, campos))
        heads = gaussian_heads(f1, f2, pos, tn, dec.albedo, light_sh, campos)
        res["shade_compose_ms"] = timeit(lambda: shade_and_compose(heads, li["light_intensity"], li["light_pos"], li["n_lights"]))
        res["full_decoder_ms_tc"] = timeit(lambda: dec(embs, pos, campos, li["light_intensity"], li["light_pos"], light_sh, li["n_lights"]))
        # last layer alone (16 -> 125 @ 1024^2): mandatory traffic = output + untied bias + input
        last = dec.vnocond_mod[12]
        h5 = torch.randn(1, 16, 512, 512, device=dev)
        seq = torch.nn.Sequential(last)
        res["last_layer_ms_tc"] = timeit(lambda: gnn.tower_forward_tc(seq, h5))
        res["last_layer_ms_simt"] = timeit(lambda: last(h5))
        bytes_last = 2 * 125 * S * S * 4 + 16 * 512 * 512 * 4
        res["last_layer_alg_GBs_tc"] = bytes_last / res["last_layer_ms_tc"] / 1e6
        res["last_layer_alg_GBs_simt"] = bytes_last / res["last_layer_ms_simt"] / 1e6
        heads_bytes = S * S * (129 * 4 + 36 + 130)
        res["heads_alg_GBs"] = heads_bytes / res["heads_ms"] / 1e6
        # (iii) of SURVEY.md §8d: decode + shade + render of one frame/view at native G = 1024^2, inference
        from goliath_b200.gsplat.fused import check_overflow
        from goliath_b200.render import render_views
        cam = synthetic.ring_camera(0, img_h=H, img_w=W)
        Rt = cam["viewmat"][None].to(dev)
        intr = [(cam["fx"], cam["fy"], cam["cx"], cam["cy"])]
        cap = 16 << 20

        def frame():
            preds = dec(embs, pos, campos, li["light_intensity"], li["light_pos"], light_sh, li["n_lights"])
            return render_views(W, H, None, Rt, preds, intrinsics_host=intr, capacity=cap)

        res["frame_decode_shade_render_fwd_ms"] = timeit(frame)
        # the same pieces replayed from CUDA graphs (frozen parameters, static shapes): launch latency removed
        from goliath_b200.graph import Graphed
        g_tower = Graphed(lambda: gnn.tower_forward_tc(dec.vnocond_mod, x))
        res["tower_vnocond_ms_tc_graph"] = timeit(g_tower)
        g_dec = Graphed(lambda: dec(embs, pos, campos, li["light_intensity"], li["light_pos"], light_sh, li["n_lights"]))
        res["full_decoder_ms_tc_graph"] = timeit(g_dec)
        g_frame = Graphed(frame)
        res["frame_decode_shade_render_fwd_ms_graph"] = timeit(g_frame)
        res["frame_MP_per_s_fwd_graph"] = H * W / 1e6 / (res["frame_decode_shade_render_fwd_ms_graph"] * 1e-3)
        res["frame_intersection_overflow_graph"] = bool(check_overflow(dev))
        # last layer on the tensor cores (pair-phase epilogue), for comparison with the FFMA2 kernel
        gnn.TC_MIN_CIN = 16
        for m_ in dec.vnocond_mod:
            if hasattr(m_, "_tc_cache"):
                del m_._tc_cache
        res["last_layer_ms_tc16"] = timeit(lambda: gnn.tower_forward_tc(seq, h5))
        f1b = gnn.tower_forward_tc(dec.vnocond_mod, x)
        res["tc16_vs_simt_rel_err"] = float((f1b - g1).norm() / g1.norm())
        g_tower16 = Graphed(lambda: gnn.tower_forward_tc(dec.vnocond_mod, x))
        res["tower_vnocond_ms_tc16_graph"] = timeit(g_tower16)
        gnn.TC_MIN_CIN = 32
        for m_ in dec.vnocond_mod:
            if hasattr(m_, "_tc_cache"):
                del m_._tc_cache
        res["frame_intersection_overflow"] = bool(check_overflow(dev))
        res["frame_MP_per_s_fwd"] = H * W / 1e6 / (res["frame_decode_shade_render_fwd_ms"] * 1e-3)
    # training direction: forward + backward of the big tower through the autograd layers (SIMT kernels, no cuDNN)
    x_t = x.detach().clone().requires_grad_()

    def tower_train():
        out = dec.vnocond_mod(x_t)
        out.backward(torch.ones_like(out))
        for p_ in dec.vnocond_mod.parameters():
            p_.grad = None

    res["tower_vnocond_fwd_bwd_ms_simt"] = timeit(tower_train, reps=3, warm=1)
    out = {"decoder": res, "config": {"slabsize": S, "params_M": sum(p.numel() for p in dec.parameters()) / 1e6,
                                      "lights": args.lights}}
    if quick:
        return out
    print(json.dumps(out))
    return out


def run_decoder_library(args):
    """The reference's own way of running a decoder tower (ca_code/nn/layers.py:380-396): library transposed
    convolution (cuDNN, TF32 allowed as by torch's default) + a bias-add pass + a LeakyReLU pass per layer, same weights
    layout and sizes as `--decoder`.  Separate flag and process because the first cuDNN call may spend minutes in
    engine compilation on a fresh box: run it under `timeout`."""
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    plan = [256, 256, 128, 128, 64, 32, 16, 125]
    gen = torch.Generator().manual_seed(1)
    ws, bs = [], []
    size = 8
    for cin, cout in zip(plan[:-1], plan[1:]):
        size *= 2
        ws.append((torch.randn(cin, cout, 4, 4, generator=gen) * 0.05).to(dev))
        bs.append((torch.randn(cout, size, size, generator=gen) * 0.05).to(dev))
    x = torch.randn(1, 256, 8, 8, generator=gen).to(dev)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def tower(inp):
        h = inp
        for i, (w, b) in enumerate(zip(ws, bs)):
            h = torch.nn.functional.conv_transpose2d(h, w, None, 2, 1) + b[None]
            if i + 1 < len(ws):
                h = torch.nn.functional.leaky_relu(h, 0.2)
        return h

    def timeit(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            flush_buf.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    res = {"tf32_allowed": bool(torch.backends.cudnn.allow_tf32)}
    with torch.no_grad():
        res["tower_vnocond_ms_library"] = timeit(lambda: tower(x))
        h5 = torch.randn(1, 16, 512, 512, device=dev)
        res["last_layer_ms_library"] = timeit(lambda: torch.nn.functional.conv_transpose2d(h5, ws[-1], None, 2, 1) + bs[-1][None])
    # forward + backward (data, weight and untied-bias gradients), the training pass the SIMT backward of --decoder is
    # compared with
    for t in ws + bs:
        t.requires_grad_(True)
    xg = x.clone().requires_grad_(True)

    def fwd_bwd():
        out = tower(xg)
        out.backward(torch.ones_like(out))
        for t in ws + bs + [xg]:
            t.grad = None

    res["tower_vnocond_fwd_bwd_ms_library"] = timeit(fwd_bwd)
    h5g = h5.clone().requires_grad_(True)

    def last_fwd_bwd():
        out = torch.nn.functional.conv_transpose2d(h5g, ws[-1], None, 2, 1) + bs[-1][None]
        out.backward(torch.ones_like(out))
        ws[-1].grad = bs[-1].grad = h5g.grad = None

    res["last_layer_fwd_bwd_ms_library"] = timeit(last_fwd_bwd)
    # the same with TF32 disallowed: cuDNN's fp32 kernels, the precision class of this repo's SIMT backward (the TF32
    # numbers above are the precision class of the 3xTF32 tcgen05 forward only up to the 3x split)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            res["tower_vnocond_ms_library_fp32"] = timeit(lambda: tower(x))
        res["tower_vnocond_fwd_bwd_ms_library_fp32"] = timeit(fwd_bwd)
        res["last_layer_fwd_bwd_ms_library_fp32"] = timeit(last_fwd_bwd)
    finally:
        torch.backends.cudnn.allow_tf32 = True
    print(json.dumps({"decoder_library": res}))


# ------------------------------------------------------------------------------------------ extension-level comparison
def run_ext_compare(args):
    """Reference arm at the EXTENSION level (SURVEY.md §8d): the reference's sgutilslib / utilslib / mvpraymarchlib
    rebuilt for sm_100a by oracle/build_ref.py versus ours, same tensors, CUDA-event timing, L2 flushed between reps.
    gsplat cannot be compared: it is absent from the reference tree and from this image."""
    import importlib.util

    from goliath_b200 import mvpraymarchlib, sgutilslib, synthetic, utilslib
    from goliath_b200.mvpraymarch import _fixedorder_topology

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def ref_mod(name):
        so = os.path.join(ROOT, "oracle", "_ref", name + ".so")
        if not os.path.exists(so):
            return None
        spec = importlib.util.spec_from_file_location(name, so)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        return m

    def timeit(fn, reps=10, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            flush_buf.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    res = {}
    # --- SG shade, G = 300k, L = 32
    G, L = args.gaussians, args.lights
    sh = synthetic.shade_inputs(G)
    li = synthetic.lights(L)
    sc = synthetic.head_gaussians(G)
    a = [torch.nn.functional.normalize(sh["lobe_dirs"], dim=-1).to(dev).contiguous(), sh["lobe_sigmas"].to(dev),
         li["light_intensity"].to(dev), li["light_pos"].to(dev), sc["means3d"][None].to(dev).contiguous(), li["n_lights"].to(dev)]
    out = torch.empty(1, G, 3, device=dev)
    g = torch.ones(1, G, 3, device=dev)
    gd, gs = torch.zeros(1, G, 3, device=dev), torch.zeros(1, G, device=dev)
    for tag, lib in (("ours", sgutilslib), ("reference", ref_mod("sgutilslib"))):
        if lib is None:
            continue
        res["sg_fwd_ms_" + tag] = timeit(lambda: lib.evaluate_gaussian_fwd(*a, out, 0))
        res["sg_bwd_ms_" + tag] = timeit(lambda: lib.evaluate_gaussian_bwd(*a, g, gd, gs, None, 0))
    # --- MVP: BASELINE config 4 shape (4096 primitives of 8x16x16 voxels, 1024x667 rays, dt = 1/2000), N views
    N = 2
    s = synthetic.mvp_scene(N=N, side=64, T=(8, 16, 16), img_h=H, img_w=W, density=args.mvp_density)
    t = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in s.items()}
    raypos, raydir, tmm = (torch.empty(N, H, W, 3, device=dev), torch.empty(N, H, W, 3, device=dev),
                           torch.empty(N, H, W, 2, device=dev))
    for tag, lib in (("ours", utilslib), ("reference", ref_mod("utilslib"))):
        if lib is None:
            continue
        res["raydirs_ms_" + tag] = timeit(lambda: lib.compute_raydirs_forward(t["viewpos"], t["viewrot"], t["focal"], t["princpt"],
                                                                               None, W, H, 1.0, raypos, raydir, tmm))
    K = t["primpos"].shape[1]
    sid, ch, par = _fixedorder_topology(N, K, dev)
    aabb = torch.empty(N, 2 * K - 1, 2, 3, device=dev)
    step = 1.0 / 2000.0
    rgba = torch.empty(N, H, W, 4, device=dev)
    sat = torch.empty(N, H, W, 3, device=dev)
    grgba = torch.ones(N, H, W, 4, device=dev)
    gp, gr, gsc = torch.zeros_like(t["primpos"]), torch.zeros_like(t["primrot"]), torch.zeros_like(t["primscale"])
    gt = torch.zeros_like(t["template"])
    for tag, lib in (("ours", mvpraymarchlib), ("reference", ref_mod("mvpraymarchlib"))):
        if lib is None:
            continue
        res["aabb_ms_" + tag] = timeit(lambda: lib.compute_aabb(t["primpos"], t["primrot"], t["primscale"], sid, ch, par, aabb, 0))

        def fwd():
            sat.fill_(-1.0)
            lib.raymarch_forward(raypos, raydir, step, tmm, sid, ch, aabb, t["primpos"], t["primrot"], t["primscale"],
                                 t["template"], None, rgba, sat, None, None, 0, False, 512, True, True, 8.0, 8.0, 0, 0.99, 3, 8, 16)

        def bwd():
            lib.raymarch_backward(raypos, raydir, step, tmm, sid, ch, aabb, t["primpos"], gp, t["primrot"], gr,
                                  t["primscale"], gsc, t["template"], gt, None, None, rgba, grgba, sat, None, 0, False, 512,
                                  True, True, 8.0, 8.0, 0, 0.99, 3, 8, 16)

        res["raymarch_fwd_ms_" + tag] = timeit(fwd, reps=5, warm=1)
        res["raymarch_bwd_ms_" + tag] = timeit(bwd, reps=5, warm=1)
        res["raymarch_alpha_mean_" + tag] = float(rgba[..., 3].mean())
    mp = N * H * W / 1e6
    for tag in ("ours", "reference"):
        if "raymarch_fwd_ms_" + tag in res:
            res["raymarch_mp_per_s_fwd_bwd_" + tag] = mp / ((res["raymarch_fwd_ms_" + tag] + res["raymarch_bwd_ms_" + tag]) / 1e3)
    print(json.dumps({"ext_compare": res, "config": {"sg": {"G": G, "L": L}, "mvp": {"N": N, "K": K, "template": [8, 16, 16],
                      "rays": [H, W], "stepsize": step, "algo": 0, "density": args.mvp_density}}}))


if __name__ == "__main__":
    a = parse()
    if a.decoder_library:
        run_decoder_library(a)
    elif a.decoder:
        run_decoder(a)
    elif a.ext_compare:
        run_ext_compare(a)
    elif a.impl == "reference":
        run_reference(a)
    elif a.config == "hand_mvp":
        run_hand_mvp(a)
    elif a.config == "mvp_full":
        run_mvp_full(a)
    else:
        run_ours(a)
