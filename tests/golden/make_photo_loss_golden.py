"""Generate tests/golden/photo_loss_ref.npz with the REFERENCE's own modules (imported from /root/reference, build
container only): CalV5 (ca_code/nn/color_cal.py), the background composite line of rgca.AutoEncoder.forward
(ca_code/models/rgca.py:226-230, restated: `rgb + (1 - alpha) * bg`), LearnableBlur (ca_code/nn/dof_cal.py) and the
losses rgb_l1 / rgb_ssim (ca_code/loss/__init__.py) at the weights of config/rgca_example.yml (10, 0.2).
Stores inputs, every intermediate, the loss and autograd gradients (rendered rgb, calibration rows, blur weights).

Usage: python tests/golden/make_photo_loss_golden.py"""
import os
import sys

import numpy as np
import torch as th

sys.path.insert(0, "/root/reference")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "photo_loss_ref.npz")


def main():
    # packages the reference imports at module level but this path never touches (absent from the image): stubbed on the
    # harness side, the reference files are not modified
    import types
    from unittest.mock import MagicMock
    for name in ("addict", "pytorch3d", "pytorch3d.renderer", "pytorch3d.renderer.mesh", "pytorch3d.renderer.mesh.rasterize_meshes",
                 "pytorch3d.structures", "pytorch3d.io", "drtk", "omegaconf", "lpips", "torchvision.models"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = MagicMock() if name != "addict" else types.SimpleNamespace(Dict=dict)
    from ca_code.nn.color_cal import CalV5
    from ca_code.nn.dof_cal import LearnableBlur
    import ca_code.loss as L

    th.manual_seed(226)
    B, H, W = 4, 45, 56                      # not multiples of the 32-pixel tiles; image wider than tall
    cams = ["400870", "400871", "410001", "400872"]     # identity, colour, GREY ("41..."), colour
    cal = CalV5(cameras=cams, identity_camera="400870").double().eval()   # eval: no lr-scale gradient hook (color_cal.py:239-240)
    with th.no_grad():
        cal.holder.params.data[:, :3] += 0.2 * th.randn(4, 3, dtype=th.float64)
        cal.holder.params.data[:, 3:] += 5.0 * th.randn(4, 3, dtype=th.float64)
    blur = LearnableBlur(cams).double()
    with th.no_grad():
        blur.weights_raw.data += th.randn(4, 3, dtype=th.float64)
    frame_cams = ["400871", "400870", "410001", "400872"]
    rgb = (255.0 * th.rand(B, 3, H, W, dtype=th.float64)).requires_grad_()
    alpha = th.rand(B, 1, H, W, dtype=th.float64)
    bg = 255.0 * th.rand(B, 3, H, W, dtype=th.float64)
    image = 255.0 * th.rand(B, 3, H, W, dtype=th.float64)
    image[:, :, :20] = rgb.detach()[:, :, :20] + 3.0 * th.randn(B, 3, 20, W, dtype=th.float64)  # a region where SSIM is high
    mask = (th.rand(B, 1, H, W, dtype=th.float64) > 0.3).double() * th.rand(B, 1, H, W, dtype=th.float64)

    idx = cal.name_to_idx(frame_cams)
    x1 = cal(rgb, idx)
    x2 = x1 + (1.0 - alpha) * bg
    x3 = blur(x2, frame_cams)
    preds, targets = {"rgb": x3}, {"image": image, "image_weight": mask}
    l1 = L.rgb_l1(preds, targets, src_key="rgb", tgt_key="image", mask_key="image_weight")
    ss = L.rgb_ssim(preds, targets, src_key="rgb", tgt_key="image", mask_key="image_weight")
    loss = 10.0 * l1 + 0.2 * ss
    params = cal.holder.params
    g_rgb, g_params, g_blur_raw, g_x3 = th.autograd.grad(loss, [rgb, params, blur.weights_raw, x3])
    # per-frame rows as the fused kernels take them
    rows = params.detach()[idx].clone()
    ident = idx == cal.identity_idx       # CalV5 passes the identity camera's image through untouched (color_cal.py:218-221):
    rows[ident, :3], rows[ident, 3:] = 1.0, 0.0   # the fused kernel's rows for such a frame are w = 1, b = 0
    bw = th.softmax(blur.weights_raw.detach()[blur.name_to_idx(frame_cams)], dim=-1)
    # gradient w.r.t. the per-frame softmax-ed weights: recompute through a leaf at that point
    bw_leaf = bw.clone().requires_grad_()
    from torchvision.transforms.functional import gaussian_blur
    x2d = x2.detach()
    x3b = (bw_leaf[:, 0].reshape(B, 1, 1, 1) * x2d + bw_leaf[:, 1].reshape(B, 1, 1, 1) * gaussian_blur(x2d, [3, 3])
           + bw_leaf[:, 2].reshape(B, 1, 1, 1) * gaussian_blur(x2d, [7, 7]))
    assert th.allclose(x3b, x3.detach(), atol=1e-9)
    (g_bw,) = th.autograd.grad((x3b * g_x3).sum(), [bw_leaf])
    g_rows = g_params[idx].clone()   # (the reference's lr-scale hook is training policy, not part of the function; rows are distinct)
    assert float(g_rows[ident].abs().max()) == 0.0   # the identity camera's parameters receive no gradient upstream
    d = dict(rgb=rgb, alpha=alpha, bg=bg, image=image, mask=mask, cal_w=rows[:, :3], cal_b=rows[:, 3:],
             grey=th.tensor([int(c.startswith("41")) for c in frame_cams]), blur_w=bw, x1=x1, x2=x2, pred=x3, l1=l1, ssim_loss=ss,
             loss=loss, g_rgb=g_rgb, g_cal_w=g_rows[:, :3], g_cal_b=g_rows[:, 3:], g_blur_w=g_bw, g_pred=g_x3)
    np.savez_compressed(OUT, **{k: (v.detach().numpy().astype(np.float32) if v.dim() == 4 else v.detach().numpy())
                                for k, v in d.items()})
    print("loss %.6f l1 %.6f ssim-loss %.6f; wrote %s (%d bytes)" % (float(loss), float(l1), float(ss), OUT, os.path.getsize(OUT)))


if __name__ == "__main__":
    main()
