"""GPU parity of the MVP raymarch path (csrc/raydirs.cu, csrc/mvp_raymarch.cu) through the reference-shaped Python
surface (goliath_b200.utils.compute_raydirs, goliath_b200.mvpraymarch.mvpraymarch) against
  * the CPU oracle (oracle/raymarch_oracle.c),
  * the reference's PyTorch-oracle fixtures (tests/golden/raymarch_pytorch_ref.npz),
  * the outputs of the reference's own kernels rebuilt for sm_100a (utilslib, mvpraymarchlib) on the same inputs
    (tests/golden/ref_kernels_{mvp,raymarch}.npz, written by tests/golden/make_ref_kernels_golden.py)."""
import os

import numpy as np
import pytest
import torch

from util import (MARCH_KEYS, MARCH_SCENE, MARCH_STEP, assert_close, load_ref_golden, march_grad, march_inputs,
                  mvp_scene, raydirs_pixels, ref_pair, t2n)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "raymarch_pytorch_ref.npz")


@pytest.fixture(params=["legacy", "queue"], autouse=True)
def raymarch_mode(request):
    """march formulation: per-primitive kernels (default) or the lane-compacted sampling queue, forward and backward"""
    from goliath_b200 import _lib

    L = _lib.lib()
    before = L.gb_get_raymarch_mode()
    L.gb_set_raymarch_mode({"legacy": 0, "queue": 3}[request.param])
    yield request.param
    L.gb_set_raymarch_mode(before)


def _rays(t):
    from goliath_b200.utils import compute_raydirs

    return compute_raydirs(t["viewpos"], t["viewrot"], t["focal"], t["princpt"], (t["img_w"], t["img_h"]), t["volradius"])


def test_raydirs_vs_oracle_and_reference(orc, cuda):
    s, t = mvp_scene(cuda, N=3, img_h=37, img_w=45)
    raypos, raydir, tminmax = _rays(t)
    n = lambda x: x.numpy()
    o = orc.raydirs_fwd(n(s["viewpos"]), n(s["viewrot"]), n(s["focal"]), n(s["princpt"]), None, 1.0, H=37, W=45)
    assert_close(t2n(raypos), o[0], rtol=1e-6, what="raypos")
    assert_close(t2n(raydir), o[1], rtol=1e-6, what="raydir")
    assert_close(t2n(tminmax), o[2], rtol=1e-5, what="tminmax")
    # explicit pixel coordinates
    from goliath_b200.utils import compute_raydirs
    pix = raydirs_pixels(3, 37, 45)
    ref = load_ref_golden("mvp", "raydirs_", [s["viewpos"], s["viewrot"], s["focal"], s["princpt"], pix])
    pix = pix.to(cuda)
    r2 = compute_raydirs(t["viewpos"], t["viewrot"], t["focal"], t["princpt"], pix, 1.0)
    o2 = orc.raydirs_fwd(n(s["viewpos"]), n(s["viewrot"]), n(s["focal"]), n(s["princpt"]), t2n(pix), 1.0)
    assert_close(t2n(r2[1]), o2[1], rtol=1e-6, what="raydir(pix)")
    for a, name in zip(r2, ("raypos", "raydir", "tminmax")):
        assert np.array_equal(t2n(a), ref[name]), "%s not bit-identical to the reference kernel" % name


def test_compute_aabb_vs_oracle_and_reference(orc, cuda):
    from goliath_b200.mvpraymarch import build_accel

    for side in (4, 5, 8):  # K = 16, 25 (not a power of two), 64
        s, t = mvp_scene(cuda, N=2, side=side)
        sid, ch, aabb = build_accel((t["primpos"], t["primrot"], t["primscale"]), 0, fixedorder=True)
        o = orc.compute_aabb_fixedorder(s["primpos"].numpy(), s["primrot"].numpy(), s["primscale"].numpy())
        assert_close(t2n(aabb), o, rtol=1e-5, what="nodeaabb K=%d" % (side * side))
        K = side * side
        assert np.array_equal(t2n(sid), np.tile(np.arange(K, dtype=np.int32), (2, 1)))
    ref = load_ref_golden("mvp", "aabb_", [s["primpos"], s["primrot"], s["primscale"]])
    assert np.array_equal(t2n(aabb), ref["nodeaabb"]), "nodeaabb not bit-identical to the reference kernel"


@pytest.mark.parametrize("algo", [0, 1])
@pytest.mark.parametrize("cfg", [dict(N=2, side=8, img_h=64, img_w=48), dict(N=1, side=5, img_h=45, img_w=37, density=400.0)])
def test_raymarch_vs_oracle(orc, cuda, algo, cfg):
    """forward + backward against the CPU oracle; the second config is dense enough to saturate rays and has K=25."""
    from goliath_b200.mvpraymarch import mvpraymarch

    s, t, raypos, raydir, tminmax = march_inputs(cuda, algo, **cfg)
    step = 0.02
    pp, pr, ps = t["primpos"].requires_grad_(), t["primrot"].requires_grad_(), t["primscale"].requires_grad_()
    tpl = t["template"].requires_grad_()
    warp = t["warp"].requires_grad_() if algo == 1 else None
    out = mvpraymarch(raypos, raydir, step, tminmax, (pp, pr, ps), tpl, warp, algo=algo, fadescale=8.0, fadeexp=8.0)
    n = lambda x: x.detach().cpu().numpy()
    warp_n = n(warp) if algo == 1 else None
    o_rgba, o_sat, _ = orc.raymarch_fwd(n(raypos), n(raydir), step, n(tminmax), n(pp), n(pr), n(ps), n(tpl), warp_n,
                                        algo=algo)
    assert (o_rgba[..., 3] > 0.05).mean() > 0.05, "scene must hit primitives"
    if cfg.get("density", 0) > 100:
        assert (o_sat[..., 0] > -1).mean() > 0.02, "dense config must saturate some rays"
    assert_close(t2n(out), o_rgba, rtol=2e-4, atol=2e-5, frac=0.999, what="rayrgba")
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(5)).to(cuda)
    out.backward(g)
    gp, gr, gs, gt, gw = orc.raymarch_bwd(n(raypos), n(raydir), step, n(tminmax), n(pp), n(pr), n(ps), n(tpl), warp_n,
                                          o_sat, n(g), algo=algo)
    tol = dict(rtol=1e-3, frac=0.995)
    assert_close(t2n(tpl.grad), gt, atol=1e-4 * np.abs(gt).max(), what="grad_template", **tol)
    assert_close(t2n(pp.grad), gp, atol=2e-3 * np.abs(gp).max(), what="grad_primpos", **tol)
    assert_close(t2n(pr.grad), gr, atol=2e-3 * np.abs(gr).max(), what="grad_primrot", **tol)
    assert_close(t2n(ps.grad), gs, atol=2e-3 * np.abs(gs).max(), what="grad_primscale", **tol)
    if algo == 1:
        assert_close(t2n(warp.grad), gw, atol=2e-3 * np.abs(gw).max(), what="grad_warp", **tol)


@pytest.mark.parametrize("tag,algo", [("n", 0), ("w", 1)])
def test_raymarch_vs_reference_pytorch_fixture(cuda, tag, algo):
    from goliath_b200.mvpraymarch import mvpraymarch

    gold = np.load(GOLD)
    g = lambda k: torch.from_numpy(gold[tag + "_" + k]).to(cuda).contiguous()
    tpl = g("template").requires_grad_()
    pp, pr, ps = g("primpos").requires_grad_(), g("primrot").requires_grad_(), g("primscale").requires_grad_()
    warp = g("warp") if algo == 1 else None
    out = mvpraymarch(g("raypos"), g("raydir"), float(gold[tag + "_stepsize"]), g("tminmax"), (pp, pr, ps), tpl, warp,
                      algo=algo, fadescale=float(gold["fadescale"]), fadeexp=float(gold["fadeexp"]))
    assert_close(t2n(out), gold[tag + "_rayrgba"], rtol=1e-4, atol=1e-6, what="rayrgba vs reference PyTorch oracle")
    out.sum().backward()
    assert_close(t2n(tpl.grad), gold[tag + "_g_template"], rtol=5e-4, what="grad_template vs reference autograd")
    if algo == 0:
        assert_close(t2n(pp.grad), gold[tag + "_g_primpos"], rtol=2e-3, what="grad_primpos vs reference autograd")
        assert_close(t2n(pr.grad), gold[tag + "_g_primrot"], rtol=2e-3, what="grad_primrot vs reference autograd")
        assert_close(t2n(ps.grad), gold[tag + "_g_primscale"], rtol=2e-3, what="grad_primscale vs reference autograd")


@pytest.mark.parametrize("algo", [0, 1])
def test_raymarch_vs_reference_kernels(cuda, algo):
    """Same tensors as the reference's mvpraymarchlib (rebuilt, -use_fast_math) was run on, through ours; the backward
    of both reads the reference's forward outputs.  The template / warp gradients are a fixed sample.  The fixture's
    input digest covers the seeded scene and output gradient, not the rays: they come from our compute_raydirs, which
    test_raydirs_vs_oracle_and_reference pins bit for bit to the reference kernel."""
    from goliath_b200 import mvpraymarchlib as ours
    from goliath_b200.mvpraymarch import build_accel

    s, t, raypos, raydir, tminmax = march_inputs(cuda, algo, **MARCH_SCENE)
    N, H, W = raypos.shape[:3]
    g = march_grad((N, H, W))
    ref = load_ref_golden("raymarch", "algo%d_" % algo, [s[k] for k in MARCH_KEYS if k in s] + [g])
    sid, ch, aabb = build_accel((t["primpos"], t["primrot"], t["primscale"]), algo, fixedorder=True)
    warp = t["warp"] if algo == 1 else None
    step = MARCH_STEP
    rgba = torch.empty(N, H, W, 4, device=cuda)
    sat = torch.full((N, H, W, 3), -1.0, device=cuda)
    ours.raymarch_forward(raypos, raydir, step, tminmax, sid, ch, aabb, t["primpos"], t["primrot"], t["primscale"],
                          t["template"], warp, rgba, sat, None, None, algo, False, 512, True, True, 8.0, 8.0, 0, 0.99, 3,
                          8, 16)
    torch.cuda.synchronize()
    r_rgba, r_sat = ref["rayrgba"], ref["raysat"]
    assert (r_rgba[..., 3] > 0.05).mean() > 0.05
    same = (t2n(rgba) == r_rgba).mean()
    assert_close(t2n(rgba), r_rgba, rtol=1e-5, atol=1e-6, frac=0.9999, what="rayrgba vs reference kernel")
    assert same > 0.99, "only %.4f of rayrgba values bit-identical to the reference kernel" % same
    assert_close(t2n(sat), r_sat, rtol=1e-5, atol=1e-6, frac=0.9999, what="raysat vs reference kernel")
    gp, gr, gs = torch.zeros_like(t["primpos"]), torch.zeros_like(t["primrot"]), torch.zeros_like(t["primscale"])
    gt = torch.zeros_like(t["template"])
    gw = torch.zeros_like(warp) if warp is not None else None
    ours.raymarch_backward(raypos, raydir, step, tminmax, sid, ch, aabb, t["primpos"], gp, t["primrot"], gr,
                           t["primscale"], gs, t["template"], gt, warp, gw, torch.from_numpy(r_rgba).to(cuda), g.to(cuda),
                           torch.from_numpy(r_sat).to(cuda), None, algo, False, 512, True, True, 8.0, 8.0, 0, 0.99, 3, 8,
                           16)
    torch.cuda.synchronize()
    for name, t in zip(("grad_primpos", "grad_primrot", "grad_primscale", "grad_template", "grad_warp"),
                       (gp, gr, gs, gt, gw)):
        if t is None:
            continue
        x, y, absmax = ref_pair(ref, name, t)
        assert_close(x, y, rtol=1e-4, atol=1e-5 * absmax, frac=0.9995, what=name + " vs reference kernel")


def test_shadow_splat_vs_oracle(orc, cuda):
    from goliath_b200.mvpraymarch import mvpraymarch

    s, t, raypos, raydir, tminmax = march_inputs(cuda, 0, N=1, side=6, img_h=40, img_w=33)
    with torch.no_grad():
        out, shadow = mvpraymarch(raypos, raydir, 0.02, tminmax, (t["primpos"], t["primrot"], t["primscale"]), t["template"],
                                  None, with_shadow=True)
    n = lambda x: x.detach().cpu().numpy()
    o_rgba, _, o_sh = orc.raymarch_fwd(n(raypos), n(raydir), 0.02, n(tminmax), n(t["primpos"]), n(t["primrot"]),
                                       n(t["primscale"]), n(t["template"]), None, with_shadow=True)
    o_shadow = o_sh[..., 0:1] / (o_sh[..., 1:] + 1e-5)
    assert_close(t2n(out), o_rgba, rtol=2e-4, atol=2e-5, frac=0.999, what="rayrgba")
    assert (o_sh[..., 1] > 0).mean() > 0.01
    assert_close(t2n(shadow), o_shadow, rtol=1e-3, atol=1e-3, frac=0.999, what="shadow")


def test_raymarch_argument_errors(cuda):
    from goliath_b200 import mvpraymarchlib

    z = torch.zeros(1, 4, 4, 3)
    with pytest.raises(RuntimeError):
        mvpraymarchlib.raymarch_forward(z, z, 0.1, z[..., :2], None, None, z, z, z, z, z, None, z, None, None, None, 0,
                                        False, 512, True, True, 8.0, 8.0, 0, 0.99, 3, 8, 16)
