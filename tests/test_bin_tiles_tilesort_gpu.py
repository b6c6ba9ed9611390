"""gb_bin_tiles_pack under both orderings — the per-tile (depth key, id) sort (`tile`, default) and depth ranks + per-tile
rank ordering (`rank`) — against the key sort: tile_bins, sorted Gaussian ids and the 48-byte records (compared as
int32) bit for bit.  Besides the scenes of test_bin_tiles_matches_key_sort: a tile longer than the per-tile sort holds
in shared memory, all-equal depths, equal depths across many ids in one tile, capacity overflow, workspace reuse, late
colours, and the 1 048 576-Gaussian bench scene."""
import numpy as np
import pytest
import torch

from util import small_scene, t2n

pytestmark = pytest.mark.gpu

MODES = {"tile": 0, "rank": 1}
PAIR_CAP = 6144  # pairs of one tile sorted in shared memory (kPairCap, csrc/splat_bin_tiles.cu)

SCENES = {
    # name: (kwargs of small_scene, block_width, scale multiplier) — the 13 scenes of test_bin_tiles_matches_key_sort
    "dense96": (dict(G=3000, img_h=96, img_w=80), 16, 12.0),
    "ragged": (dict(G=2500, img_h=70, img_w=93, seed=11, cam=3), 16, 15.0),
    "bw8": (dict(G=1500, img_h=64, img_w=48, seed=5), 8, 10.0),
    "ties": (dict(G=4000, img_h=96, img_w=80, depth_quant=True), 16, 8.0),
    "tiny_prims": (dict(G=5000, img_h=128, img_w=96, seed=9), 16, 1.0),
    "one_cta": (dict(G=4096, img_h=96, img_w=80, seed=3), 16, 10.0),
    "two_ctas": (dict(G=4097, img_h=96, img_w=80, seed=4, depth_quant=True), 16, 10.0),
    "big": (dict(G=150_000, img_h=512, img_w=384, seed=13), 16, 6.0),
    "many_tiles": (dict(G=30_000, img_h=768, img_w=1024, seed=17), 8, 2.0),
    "too_many_tiles": (dict(G=20_000, img_h=600, img_w=640, seed=19), 4, 1.5),
    "sixteen_per_thread": (dict(G=400_000, img_h=256, img_w=192, seed=23), 16, 1.5),
    "flat_depth": (dict(G=6000, img_h=96, img_w=80, seed=31, cam=0), 16, 10.0),
    "wide_depth": (dict(G=9000, img_h=96, img_w=80, seed=37, cam=0), 16, 10.0),
}


@pytest.fixture
def lib():
    from goliath_b200 import _lib

    L = _lib.lib()
    before = L.gb_get_bin_sort_mode()
    yield L
    L.gb_set_bin_sort_mode(before)


def _bin(L, mode, G, xys, depths, radii, conics, colors, opacity, comp, H, W, bw, cap, ws=None, colors_event=None):
    from goliath_b200 import _lib

    dev = xys.device
    T = -(-W // bw) * -(-H // bw)
    if ws is None:
        ws = torch.empty(L.gb_bin_tiles_workspace_bytes(G, T, cap), dtype=torch.uint8, device=dev)
    out = dict(bins=torch.full((T, 2), -7, dtype=torch.int32, device=dev),
               order=torch.full((T,), -7, dtype=torch.int32, device=dev),
               gids=torch.full((max(cap, 1),), -7, dtype=torch.int32, device=dev),
               rec=torch.full((max(cap, 1), 12), float("nan"), device=dev),
               n=torch.zeros(1, dtype=torch.int32, device=dev), ovf=torch.zeros(1, dtype=torch.int32, device=dev))
    L.gb_set_bin_sort_mode(MODES[mode])
    assert L.gb_get_bin_sort_mode() == MODES[mode]
    args = (G, xys.data_ptr(), depths.data_ptr(), radii.data_ptr(), conics.data_ptr(), colors.data_ptr(),
            opacity.data_ptr(), comp.data_ptr(), H, W, bw, cap, out["bins"].data_ptr(), out["order"].data_ptr(), 0,
            out["gids"].data_ptr(), out["rec"].data_ptr(), out["n"].data_ptr(), out["ovf"].data_ptr(), ws.data_ptr())
    st = _lib.stream_ptr(dev)
    if colors_event is None:
        _lib.check(L.gb_bin_tiles_pack(*args, st), "bin_tiles_pack")
    else:
        _lib.check(L.gb_bin_tiles_pack_ev(*args, colors_event.cuda_event, st), "bin_tiles_pack_ev")
    torch.cuda.synchronize()
    out["T"] = T
    return out


def _pack_ref(L, gids_ref, xys, conics, colors, depths, opacity, comp):
    from goliath_b200 import _lib

    n = gids_ref.numel()
    rec = torch.empty(n, 12, device=xys.device)
    _lib.check(L.gb_pack_records_fused(n, gids_ref.data_ptr(), xys.data_ptr(), conics.data_ptr(), colors.data_ptr(),
                                       depths.data_ptr(), opacity.data_ptr(), comp.data_ptr(), rec.data_ptr(),
                                       _lib.stream_ptr(xys.device)), "pack")
    return rec


def _numpy_key_sort(xys, depths, radii, H, W, bw):
    """The key sort's tile lists in numpy: same tile rectangle arithmetic (float32, round to nearest, truncation),
    each tile ordered by (depth bits, id)."""
    f = np.float32
    tbx, tby = -(-W // bw), -(-H // bw)
    tcx, tcy = xys[:, 0] / f(bw), xys[:, 1] / f(bw)
    tr = radii.astype(f) / f(bw)
    x0 = np.clip(np.trunc(tcx - tr).astype(np.int64), 0, tbx)
    x1 = np.clip(np.trunc((tcx + tr) + f(1)).astype(np.int64), 0, tbx)
    y0 = np.clip(np.trunc(tcy - tr).astype(np.int64), 0, tby)
    y1 = np.clip(np.trunc((tcy + tr) + f(1)).astype(np.int64), 0, tby)
    w, h = x1 - x0, y1 - y0
    cnt = np.where(radii > 0, w * h, 0)
    gid = np.repeat(np.arange(len(radii)), cnt)
    k = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    tile = (y0[gid] + k // w[gid]) * tbx + x0[gid] + k % w[gid]
    key = depths.view(np.uint32)[gid]
    o = np.lexsort((gid, key, tile))
    counts = np.bincount(tile, minlength=tbx * tby)
    ends = np.cumsum(counts)
    bins = np.stack([ends - counts, ends], 1)
    bins[counts == 0] = 0
    return gid[o].astype(np.int32), bins.astype(np.int32)


def _synthetic(cuda, G, H, W, seed, hot=0, flat=False, tie_levels=0):
    """Projected inputs drawn directly: `hot` Gaussians inside tile 0 only (radius 2, centres 4..12 px), the rest spread
    over the image with radii 1..24.  flat: one depth for all; tie_levels > 0: depths from that many values."""
    rng = np.random.default_rng(seed)
    xy = np.stack([rng.uniform(0, W, G), rng.uniform(0, H, G)], 1).astype(np.float32)
    radii = rng.integers(1, 25, G).astype(np.int32)
    radii[rng.random(G) < 0.05] = 0  # culled
    if hot:
        xy[:hot] = rng.uniform(4.0, 12.0, (hot, 2)).astype(np.float32)
        radii[:hot] = 2
    depths = rng.uniform(0.5, 3.0, G).astype(np.float32)
    if tie_levels:
        depths = (1.0 + rng.integers(0, tie_levels, G) / 64.0).astype(np.float32)
    if flat:
        depths[:] = np.float32(1.25)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    t = dict(xys=d(xy), depths=d(depths), radii=d(radii), conics=d(rng.uniform(0.01, 1, (G, 3)).astype(np.float32)),
             colors=d(rng.uniform(0, 1, (G, 3)).astype(np.float32)),
             opacity=d(rng.uniform(0.1, 1, (G, 1)).astype(np.float32)), comp=d(rng.uniform(0.5, 1, G).astype(np.float32)))
    gids_ref, bins_ref = _numpy_key_sort(xy, depths, radii, H, W, 16)
    return t, gids_ref, bins_ref


def _check_exact(L, out, t, gids_ref, bins_ref):
    n = len(gids_ref)
    assert int(out["n"]) == n and int(out["ovf"]) == 0
    assert sorted(t2n(out["order"]).tolist()) == list(range(out["T"]))
    assert np.array_equal(t2n(out["bins"]), bins_ref)
    assert np.array_equal(t2n(out["gids"][:n]), gids_ref)
    g = torch.from_numpy(gids_ref).to(out["gids"].device)
    rec_ref = _pack_ref(L, g, t["xys"], t["conics"], t["colors"], t["depths"], t["opacity"], t["comp"])
    assert torch.equal(out["rec"][:n].view(torch.int32), rec_ref.view(torch.int32))
    assert bool((out["gids"][n:] == -7).all())


def _run_synthetic(L, cuda, mode, G, H, W, seed, **kw):
    t, gids_ref, bins_ref = _synthetic(cuda, G, H, W, seed, **kw)
    n = len(gids_ref)
    out = _bin(L, mode, G, t["xys"], t["depths"], t["radii"], t["conics"], t["colors"], t["opacity"], t["comp"], H, W,
               16, n + 99)
    _check_exact(L, out, t, gids_ref, bins_ref)
    return out, t, gids_ref, bins_ref


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("case", list(SCENES))
def test_both_orderings_match_key_sort(lib, cuda, case, mode):
    from goliath_b200.gsplat import project_gaussians
    from goliath_b200.gsplat import utils as gu

    kw, bw, mult = SCENES[case]
    s = small_scene(**kw)
    if case == "flat_depth":
        s["means3d"][:, 2] = 0.0
    if case == "wide_depth":
        rng = np.random.default_rng(37)
        s["means3d"][:, 2] = (1000.0 - np.exp2(rng.uniform(-2.0, 10.0, size=len(s["means3d"])))).astype(np.float32)
        s["means3d"][:, :2] *= 0.05
    d = lambda a: torch.from_numpy(a).to(cuda)
    H, W = s["img_h"], s["img_w"]
    xys, depths, radii, conics, comp, nth, _ = project_gaussians(d(s["means3d"]), d(s["scales"]) * mult, 1.0,
                                                                 d(s["quats"]), d(s["viewmat"]), s["fx"], s["fy"],
                                                                 s["cx"], s["cy"], H, W, bw, 0.1)
    colors, opacity = d(s["colors"]).contiguous(), d(s["opacity"]).contiguous()
    G = xys.shape[0]
    n, cum = gu.compute_cumulative_intersects(nth)
    _, _, _, gids_ref, bins_ref = gu.bin_and_sort_gaussians(G, n, xys, depths, radii, cum, gu._tile_bounds(H, W, bw), bw)
    rec_ref = _pack_ref(lib, gids_ref, xys, conics, colors, depths, opacity, comp)
    out = _bin(lib, mode, G, xys, depths, radii, conics, colors, opacity, comp, H, W, bw, n + 77)
    assert int(out["n"]) == n and int(out["ovf"]) == 0
    assert torch.equal(out["bins"], bins_ref)
    assert torch.equal(out["gids"][:n], gids_ref)
    assert torch.equal(out["rec"][:n].view(torch.int32), rec_ref.view(torch.int32))


@pytest.mark.parametrize("mode", list(MODES))
def test_tile_longer_than_shared_memory(lib, cuda, mode):
    """20 000 Gaussians in tile 0 alone (plus 30 000 spread out): the per-tile sort of tile 0 runs out of shared
    memory, in the tile's own record slots."""
    out, *_ = _run_synthetic(lib, cuda, mode, 50_000, 256, 320, seed=5, hot=20_000)
    b = t2n(out["bins"])
    assert (b[:, 1] - b[:, 0]).max() > PAIR_CAP


@pytest.mark.parametrize("mode", list(MODES))
def test_all_equal_depths(lib, cuda, mode):
    """One depth for every Gaussian: each tile is ordered by id alone (with a hot tile, in and out of shared memory)."""
    _run_synthetic(lib, cuda, mode, 30_000, 200, 240, seed=6, flat=True, hot=8000)


@pytest.mark.parametrize("mode", list(MODES))
def test_equal_depths_across_many_ids_in_one_tile(lib, cuda, mode):
    """Depths from 3 values: thousands of ids share a depth inside the same tile, so the tie order (ascending id) decides
    almost every position."""
    _run_synthetic(lib, cuda, mode, 12_000, 128, 128, seed=8, tie_levels=3, hot=5000)


@pytest.mark.parametrize("mode", list(MODES))
def test_capacity_overflow(lib, cuda, mode):
    """cap < n: *overflow is set, bins are clamped to the capacity and every surviving bucket — including the hot tile
    that straddles the capacity — is a depth-ordered subset of its tile's list."""
    t, gids_ref, bins_ref = _synthetic(cuda, 50_000, 256, 320, seed=9, hot=20_000)
    n = len(gids_ref)
    for cap in (n - 1, 15_000, n // 3):
        out = _bin(lib, mode, 50_000, t["xys"], t["depths"], t["radii"], t["conics"], t["colors"], t["opacity"],
                   t["comp"], 256, 320, 16, cap)
        assert int(out["n"]) == n and int(out["ovf"]) == 1
        b = t2n(out["bins"]).astype(np.int64)
        br = np.minimum(bins_ref.astype(np.int64), cap)
        br[br[:, 1] <= br[:, 0]] = 0
        assert np.array_equal(b, br)
        g = t2n(out["gids"])
        for tile in np.nonzero(b[:, 1] > b[:, 0])[0]:
            mine = g[b[tile, 0]:b[tile, 1]]
            pos = {v: i for i, v in enumerate(gids_ref[bins_ref[tile, 0]:bins_ref[tile, 1]].tolist())}
            idx = [pos[v] for v in mine.tolist()]
            assert idx == sorted(idx) and len(set(idx)) == len(idx)


def test_workspace_reuse_across_scenes_and_modes(lib, cuda):
    """One workspace, four calls — two scenes, both orderings, alternating: nothing stale leaks between calls."""
    G, H, W = 40_000, 256, 320
    scenes = [_synthetic(cuda, G, H, W, seed=s, hot=h) for s, h in ((11, 9000), (12, 0))]
    cap = max(len(s[1]) for s in scenes) + 5
    ws = torch.empty(lib.gb_bin_tiles_workspace_bytes(G, -(-W // 16) * -(-H // 16), cap), dtype=torch.uint8, device=cuda)
    for mode in ("tile", "rank", "tile"):
        for t, gids_ref, bins_ref in scenes:
            out = _bin(lib, mode, G, t["xys"], t["depths"], t["radii"], t["conics"], t["colors"], t["opacity"], t["comp"],
                       H, W, 16, cap, ws=ws)
            n = len(gids_ref)
            assert np.array_equal(t2n(out["bins"]), bins_ref)
            assert np.array_equal(t2n(out["gids"][:n]), gids_ref)


@pytest.mark.parametrize("mode", list(MODES))
def test_late_colours(lib, cuda, mode):
    """gb_bin_tiles_pack_ev with the colours written on another stream: same records as with the colours at hand."""
    t, gids_ref, bins_ref = _synthetic(cuda, 30_000, 200, 240, seed=13, hot=7000)
    final = t["colors"].clone()
    t["colors"].zero_()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    ev = torch.cuda.Event()
    with torch.cuda.stream(side):
        torch.cuda._sleep(2_000_000)  # the binning starts long before the colours exist
        t["colors"].copy_(final)
        ev.record(side)
    out = _bin(lib, mode, 30_000, t["xys"], t["depths"], t["radii"], t["conics"], t["colors"], t["opacity"], t["comp"],
               200, 240, 16, len(gids_ref) + 3, colors_event=ev)
    _check_exact(lib, out, t, gids_ref, bins_ref)


def test_tile_sort_bit_exact_at_native_size(lib, cuda):
    """The bench scene at 1 048 576 Gaussians, 1024x667: the per-tile sort against the key sort, records included."""
    import bench
    from goliath_b200 import synthetic
    from goliath_b200.gsplat import project_gaussians
    from goliath_b200.gsplat import utils as gu

    G = 1_048_576
    u = bench.unpack(bench.packed_scene(G).to(cuda))
    c = synthetic.ring_camera(2, img_h=bench.H, img_w=bench.W)
    H, W, BW = bench.H, bench.W, 16
    xys, depths, radii, conics, comp, nth, _ = project_gaussians(
        u["primpos"].contiguous(), u["primscale"].contiguous(), 1.0, u["primqvec"].contiguous(), c["viewmat"].to(cuda),
        c["fx"], c["fy"], c["cx"], c["cy"], H, W, BW, 0.1)
    col3, op1 = u["diff_color"].contiguous(), u["opacity"].contiguous()
    n, cum = gu.compute_cumulative_intersects(nth)
    _, _, _, gids_ref, bins_ref = gu.bin_and_sort_gaussians(G, n, xys, depths, radii, cum, gu._tile_bounds(H, W, BW), BW)
    rec_ref = _pack_ref(lib, gids_ref, xys, conics, col3, depths, op1, comp)
    out = _bin(lib, "tile", G, xys, depths, radii, conics, col3, op1, comp, H, W, BW, n + 4096)
    assert int(out["n"]) == n and int(out["ovf"]) == 0
    assert torch.equal(out["bins"], bins_ref)
    assert torch.equal(out["gids"][:n], gids_ref)
    assert torch.equal(out["rec"][:n].view(torch.int32), rec_ref.view(torch.int32))
