"""Shared helpers for the parity tests."""
import numpy as np
import torch

from goliath_b200 import synthetic


def small_scene(G=3000, img_h=96, img_w=80, seed=7, cam=1, spread=1.0, depth_quant=False):
    """A small RGCA-like scene that projects to a few hundred pixels; returns numpy inputs."""
    sc = synthetic.head_gaussians(G, seed=seed)
    c = synthetic.ring_camera(cam, img_h=img_h, img_w=img_w)
    # shrink the focal length so the 100 mm head fills the small image
    f = 0.35 * min(img_h, img_w) / 120.0 * 1000.0 * spread
    c.update(fx=f, fy=f)
    d = {k: v.numpy() for k, v in sc.items()}
    if depth_quant:  # force exact depth ties between different Gaussians (sort stability case)
        d["means3d"] = np.round(d["means3d"] / 8.0).astype(np.float32) * 8.0
    d.update(viewmat=c["viewmat"].numpy(), fx=c["fx"], fy=c["fy"], cx=c["cx"], cy=c["cy"], img_h=img_h, img_w=img_w)
    return d


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def assert_close(a, b, rtol=1e-4, atol=None, frac=1.0, what=""):
    """Element-wise |a-b| <= atol + rtol*|b| for at least `frac` of the elements, and norm-wise rel err <= rtol.
    atol defaults to rtol * 1e-2 * max|b| (fp32 cancellation noise scales with the summands, not the result)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if atol is None:
        atol = rtol * 1e-2 * (np.abs(b).max() if b.size else 0.0)
    ok = np.abs(a - b) <= atol + rtol * np.abs(b)
    got = ok.mean() if ok.size else 1.0
    assert got >= frac, "%s: only %.6f of elements within tol (need %.6f); max abs diff %.3e" % (
        what, got, frac, np.abs(a - b).max())
    r = rel_err(a, b)
    assert r <= rtol, "%s: norm-wise relative error %.3e > %.1e" % (what, r, rtol)


def t2n(t):
    return t.detach().cpu().numpy()


# ------------------------------------------------------------------ reference-kernel fixtures (tests/golden/ref_kernels_*.npz)
# The inputs below are what tests/golden/make_ref_kernels_golden.py fed to the reference's own kernels; the tests that
# compare against those recorded outputs build the same inputs here.
SG_SHAPE = (2, 20000, 32)        # N, D, L
SG_SAMPLE = 12000                # stored elements of each [N, D, 3] output (grad_sigmas: a third as many)
MARCH_SCENE = dict(N=2, side=12, T=(4, 8, 8), img_h=96, img_w=72, density=150.0)
MARCH_STEP = 0.01
MARCH_SAMPLE = 20000             # stored elements of the template / warp gradients
MARCH_KEYS = ("primpos", "primrot", "primscale", "template", "warp", "viewpos", "viewrot", "focal", "princpt")


def sha256(arrays):
    """Digest of the shapes, dtypes and bytes of a list of tensors / arrays."""
    import hashlib

    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a.detach().cpu().numpy() if torch.is_tensor(a) else a)
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def sample_index(size, n):
    """Fixed, seeded, sorted sample of n flat indices out of size (all of them when n >= size)."""
    if n >= size:
        return np.arange(size, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(size, n, replace=False)).astype(np.int64)


def load_ref_golden(name, key_prefix, inputs):
    """The recorded reference outputs of tests/golden/ref_kernels_<name>.npz whose keys start with key_prefix, after
    checking that they were recorded for these inputs."""
    import os

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels_%s.npz" % name)
    z = np.load(path)
    want = str(z[key_prefix + "inputs_sha256"])
    assert sha256(inputs) == want, "inputs differ from those the reference outputs in %s were recorded for" % path
    return {k[len(key_prefix):]: z[k] for k in z.files if k.startswith(key_prefix)}


def ref_pair(ref, name, ours):
    """(ours, the recorded reference values, max |reference| over the full array) for the entry `name` of a
    load_ref_golden() dict; a sampled entry selects the same elements of ours."""
    x, y = t2n(ours), ref[name]
    if name + "_idx" in ref:
        return x.reshape(-1)[ref[name + "_idx"]], y, float(ref[name + "_absmax"])
    return x, y, float(np.abs(y).max())


def sg_inputs(w_type):
    """[dirs, sigmas, light values, light positions, primitive positions, n_lights] and the output gradient."""
    from test_oracle_sg import make

    N, D, L = SG_SHAPE
    dirs, sig, lv, lp, pp, nl = make(N=N, D=D, L=L, seed=123)
    if w_type >= 2:
        sig = sig * 0 + 0.3
    g = torch.randn(N, D, 3, generator=torch.Generator().manual_seed(3))
    return [dirs, sig, lv, lp, pp, nl], g


def mvp_scene(dev, **kw):
    s = synthetic.mvp_scene(**kw)
    t = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in s.items()}
    return s, t


def raydirs_pixels(N, H, W):
    px, py = torch.meshgrid(torch.arange(float(W)), torch.arange(float(H)), indexing="xy")
    return (torch.stack([px, py], -1)[None].repeat(N, 1, 1, 1) + 0.5).contiguous()


def march_inputs(dev, algo, **kw):
    """Scene and rays (from our compute_raydirs) of a raymarch test."""
    from goliath_b200.utils import compute_raydirs

    s, t = mvp_scene(dev, with_warp=(algo == 1), **kw)
    raypos, raydir, tminmax = compute_raydirs(t["viewpos"], t["viewrot"], t["focal"], t["princpt"], (t["img_w"], t["img_h"]),
                                              t["volradius"])
    return s, t, raypos, raydir, tminmax


def march_grad(shape):
    N, H, W = shape
    return torch.randn(N, H, W, 4, generator=torch.Generator().manual_seed(11))
