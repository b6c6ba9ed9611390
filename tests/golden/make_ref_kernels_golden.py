"""Generate tests/golden/ref_kernels_{sg,mvp,raymarch}.npz: outputs of the REFERENCE's own CUDA kernels (sgutilslib,
utilslib, mvpraymarchlib rebuilt for sm_100a into oracle/_ref/ by oracle/build_ref.py) on the inputs that
tests/test_sg_gpu.py and tests/test_raymarch_gpu.py build, so that those tests compare our kernels against the
reference without the reference being present.

Needs a CUDA device and oracle/_ref/*.so; the .npz files are committed.
Usage: python tests/golden/make_ref_kernels_golden.py [OUT_DIR]   (default: tests/golden)

Each file holds an `inputs_sha256` of the seeded CPU inputs; the tests recompute it and refuse to compare against
outputs recorded for other inputs.  The raymarch rays are not in it: they come from our compute_raydirs on the GPU,
which tests/test_raymarch_gpu.py pins bit for bit to the reference's raydirs kernel.  Arrays larger than the per-file budget are stored as a fixed, seeded sample
(`*_idx` = flat indices into the full array, `*_absmax` = max |x| of the full array, which the tolerances use).
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import util  # noqa: E402


def ref_lib(name):
    so = os.path.join(ROOT, "oracle", "_ref", name + ".so")
    if not os.path.exists(so):
        sys.exit("oracle/_ref/%s.so is missing: build it with oracle/build_ref.py first" % name)
    spec = importlib.util.spec_from_file_location(name, so)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def t2n(t):
    return t.detach().cpu().numpy()


def sampled(d, key, full, n):
    idx = util.sample_index(full.size, n)
    d[key] = full.reshape(-1)[idx]
    d[key + "_idx"] = idx
    d[key + "_absmax"] = np.float32(np.abs(full).max())


def make_sg(dev):
    ref = ref_lib("sgutilslib")
    out = {}
    for w_type in (0, 1, 2, 3):
        a, g = util.sg_inputs(w_type)
        out["w%d_inputs_sha256" % w_type] = util.sha256(a + [g])
        a = [t.to(dev).contiguous() for t in a]
        g = g.to(dev).contiguous()
        N, D, L = util.SG_SHAPE
        o = torch.empty(N, D, 3, device=dev)
        ref.evaluate_gaussian_fwd(*a, o, w_type)
        gd, gs, gl = torch.zeros(N, D, 3, device=dev), torch.zeros(N, D, device=dev), torch.zeros(N, L, 3, device=dev)
        ref.evaluate_gaussian_bwd(*a, g, gd, gs, gl, w_type)
        torch.cuda.synchronize()
        p = "w%d_" % w_type
        sampled(out, p + "integral", t2n(o), util.SG_SAMPLE)
        sampled(out, p + "grad_dirs", t2n(gd), util.SG_SAMPLE)
        sampled(out, p + "grad_sigmas", t2n(gs), util.SG_SAMPLE // 3)
        out[p + "grad_light_values"] = t2n(gl)
    return out


def make_mvp(dev):
    from goliath_b200.mvpraymarch import _fixedorder_topology, build_accel

    ut, mv = ref_lib("utilslib"), ref_lib("mvpraymarchlib")
    out = {}
    # test_raydirs_vs_oracle_and_reference: explicit pixel coordinates
    s, t = util.mvp_scene(dev, N=3, img_h=37, img_w=45)
    pix = util.raydirs_pixels(3, 37, 45)
    out["raydirs_inputs_sha256"] = util.sha256([s["viewpos"], s["viewrot"], s["focal"], s["princpt"], pix])
    pix = pix.to(dev)
    rr = [torch.empty(3, 37, 45, k, device=dev) for k in (3, 3, 2)]
    ut.compute_raydirs_forward(t["viewpos"], t["viewrot"], t["focal"], t["princpt"], pix, 45, 37, 1.0, *rr)
    torch.cuda.synchronize()
    for name, x in zip(("raypos", "raydir", "tminmax"), rr):
        out["raydirs_" + name] = t2n(x)
    # test_compute_aabb_vs_oracle_and_reference: K = 64
    s, t = util.mvp_scene(dev, N=2, side=8)
    out["aabb_inputs_sha256"] = util.sha256([s["primpos"], s["primrot"], s["primscale"]])
    sid, ch, par = _fixedorder_topology(2, 64, dev)
    _, _, aabb = build_accel((t["primpos"], t["primrot"], t["primscale"]), 0, fixedorder=True)
    ra = torch.empty_like(aabb)
    mv.compute_aabb(t["primpos"], t["primrot"], t["primscale"], sid, ch, par, ra, 0)
    torch.cuda.synchronize()
    out["aabb_nodeaabb"] = t2n(ra)
    return out


def make_raymarch(dev):
    from goliath_b200.mvpraymarch import build_accel

    mv = ref_lib("mvpraymarchlib")
    out = {}
    for algo in (0, 1):
        s, t, raypos, raydir, tminmax = util.march_inputs(dev, algo, **util.MARCH_SCENE)
        g = util.march_grad(raypos.shape[:3])
        p = "algo%d_" % algo
        out[p + "inputs_sha256"] = util.sha256([s[k] for k in util.MARCH_KEYS if k in s] + [g])
        N, H, W = raypos.shape[:3]
        sid, ch, aabb = build_accel((t["primpos"], t["primrot"], t["primscale"]), algo, fixedorder=True)
        warp = t["warp"] if algo == 1 else None
        rgba = torch.empty(N, H, W, 4, device=dev)
        sat = torch.full((N, H, W, 3), -1.0, device=dev)
        mv.raymarch_forward(raypos, raydir, util.MARCH_STEP, tminmax, sid, ch, aabb, t["primpos"], t["primrot"],
                            t["primscale"], t["template"], warp, rgba, sat, None, None, algo, False, 512, True, True, 8.0,
                            8.0, 0, 0.99, 3, 8, 16)
        torch.cuda.synchronize()
        g = g.to(dev)
        gp, gr, gs = torch.zeros_like(t["primpos"]), torch.zeros_like(t["primrot"]), torch.zeros_like(t["primscale"])
        gt = torch.zeros_like(t["template"])
        gw = torch.zeros_like(warp) if warp is not None else None
        mv.raymarch_backward(raypos, raydir, util.MARCH_STEP, tminmax, sid, ch, aabb, t["primpos"], gp, t["primrot"],
                             gr, t["primscale"], gs, t["template"], gt, warp, gw, rgba, g, sat, None, algo, False, 512,
                             True, True, 8.0, 8.0, 0, 0.99, 3, 8, 16)
        torch.cuda.synchronize()
        out[p + "rayrgba"], out[p + "raysat"] = t2n(rgba), t2n(sat)
        for name, x in zip(("grad_primpos", "grad_primrot", "grad_primscale"), (gp, gr, gs)):
            out[p + name] = t2n(x)
        sampled(out, p + "grad_template", t2n(gt), util.MARCH_SAMPLE)
        if gw is not None:
            sampled(out, p + "grad_warp", t2n(gw), util.MARCH_SAMPLE)
    return out


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(out_dir, exist_ok=True)
    dev = torch.device("cuda:0")
    for name, fn in (("sg", make_sg), ("mvp", make_mvp), ("raymarch", make_raymarch)):
        path = os.path.join(out_dir, "ref_kernels_%s.npz" % name)
        np.savez_compressed(path, **fn(dev))
        print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
