"""GPU parity of the SG shade kernels (csrc/sg_shade.cu) through the reference-shaped Python surface
(goliath_b200.sgutils.evaluate_gaussian) against the CPU oracle, and against the outputs of the reference's own
sgutilslib rebuilt for sm_100a (tests/golden/ref_kernels_sg.npz, written by tests/golden/make_ref_kernels_golden.py)."""
import numpy as np
import pytest
import torch

from test_oracle_sg import make
from util import SG_SHAPE, assert_close, load_ref_golden, ref_pair, sg_inputs, t2n

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("w_type", [0, 1, 2, 3])
@pytest.mark.parametrize("shape", [(2, 257, 5), (1, 5000, 32), (3, 130, 300)])
def test_sg_vs_oracle(orc, cuda, w_type, shape):
    from goliath_b200.sgutils import evaluate_gaussian

    N, D, L = shape
    dirs, sig, lv, lp, pp, nl = make(N=min(N, 2), D=D, L=L, seed=D)
    if N > 2:
        dirs, sig, lv, lp, pp = (t.repeat(2, *([1] * (t.dim() - 1)))[:N].contiguous() for t in (dirs, sig, lv, lp, pp))
        nl = torch.tensor([L, L - 1, 1], dtype=torch.int32)
    if w_type >= 2:
        sig = sig * 0 + 0.3
    c = lambda t: t.to(cuda)
    dd, ss, ll = c(dirs).requires_grad_(), c(sig).requires_grad_(), c(lv).requires_grad_()
    out = evaluate_gaussian(dd, ss, ll, c(lp), c(pp), c(nl), w_type=w_type, normalize_lobe_dirs=False)
    ref = orc.sg_fwd(dirs.numpy(), sig.numpy(), lv.numpy(), lp.numpy(), pp.numpy(), nl.numpy(), w_type)
    # both sides are fp32 evaluations of an ill-conditioned formula (acos near 1, / sigma^2): compare to 1e-4 of the
    # output scale element-wise and 1e-4 norm-wise... narrow lobes amplify 1-ulp cosine differences, hence atol
    assert_close(t2n(out), ref, rtol=1e-3, atol=1e-4 * float(np.abs(ref).max()), frac=0.999, what="integral")
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(2))
    out.backward(c(g))
    gd, gs, gl = orc.sg_bwd(dirs.numpy(), sig.numpy(), lv.numpy(), lp.numpy(), pp.numpy(), nl.numpy(), g.numpy(), w_type)
    assert_close(t2n(ll.grad), gl, rtol=1e-3, atol=1e-4 * float(np.abs(gl).max()), what="grad_light_values")
    assert_close(t2n(ss.grad), gs, rtol=2e-3, atol=1e-4 * float(np.abs(gs).max()), frac=0.999, what="grad_sigmas")
    assert_close(t2n(dd.grad), gd, rtol=2e-3, atol=1e-4 * float(np.abs(gd).max()), frac=0.999, what="grad_dirs")


@pytest.mark.parametrize("w_type", [0, 1, 2, 3])
def test_sg_vs_reference_kernels(cuda, w_type):
    """Same inputs as the reference's sg.cu (rebuilt, -use_fast_math) was run on, through ours; the reference's
    outputs are a fixed sample of its [N, D] results (its full light-value gradient)."""
    from goliath_b200 import sgutilslib as ours

    a, g = sg_inputs(w_type)
    ref = load_ref_golden("sg", "w%d_" % w_type, a + [g])
    N, D, L = SG_SHAPE
    c = lambda t: t.to(cuda).contiguous()
    a, g = [c(t) for t in a], c(g)
    o_our = torch.empty(N, D, 3, device=cuda)
    ours.evaluate_gaussian_fwd(*a, o_our, w_type)
    torch.cuda.synchronize()
    o, r, absmax = ref_pair(ref, "integral", o_our)
    assert_close(o, r, rtol=1e-3, atol=1e-4 * absmax, frac=0.999, what="integral vs ref")
    # same formula, same operation order, same -use_fast_math flag: the forward is bit-identical to sg.cu
    assert (o.view(np.uint32) == r.view(np.uint32)).mean() >= 0.9999, "forward not bit-identical to the reference kernel"
    gd, gs, gl = torch.zeros(N, D, 3, device=cuda), torch.zeros(N, D, device=cuda), torch.zeros(N, L, 3, device=cuda)
    ours.evaluate_gaussian_bwd(*a, g, gd, gs, gl, w_type)
    torch.cuda.synchronize()
    for name, t in zip(("grad_dirs", "grad_sigmas", "grad_light_values"), (gd, gs, gl)):
        x, y, absmax = ref_pair(ref, name, t)
        assert_close(x, y, rtol=2e-3, atol=1e-4 * absmax, frac=0.999, what=name + " vs ref")
        if name != "grad_light_values":  # that one is an atomics-order sum in both implementations
            assert (x.view(np.uint32) == y.view(np.uint32)).mean() >= 0.9999, name + " not bit-identical to the reference kernel"


def test_sg_errors_like_reference(cuda):
    from goliath_b200 import sgutilslib

    t = torch.zeros(1, 4, 3)
    with pytest.raises(RuntimeError):
        sgutilslib.evaluate_gaussian_fwd(t, t[..., 0], t, t, t, torch.ones(1, dtype=torch.int32), t.clone(), 0)
    tc = t.to(cuda)
    with pytest.raises(RuntimeError):  # non-contiguous
        sgutilslib.evaluate_gaussian_fwd(tc.transpose(1, 2).transpose(1, 2)[:, ::2], tc[..., 0], tc, tc, tc,
                                         torch.ones(1, dtype=torch.int32, device=cuda), tc.clone(), 0)


@pytest.mark.parametrize("w_type", [0, 2])
def test_shade_compose_matches_unfused_chain(cuda, w_type):
    """rgca_heads.shade_compose (normalise + SG + spec_vis + both clamps in one kernel each way) against the
    reference's op-by-op chain rgca.py:557-575 built from evaluate_gaussian and torch ops; negative light values and
    negative diffuse exercise both clamp masks."""
    from goliath_b200.rgca_heads import shade_compose
    from goliath_b200.sgutils import evaluate_gaussian

    gen = torch.Generator().manual_seed(41 + w_type)
    N, D, L = 2, 3001, 9
    mk = lambda *s: torch.randn(*s, generator=gen)
    base = dict(ref_dirs=mk(N, D, 3) * 3.0, sigma=(0.1 * torch.exp(0.5 * mk(N, D))).clamp(min=0.01),
                lint=mk(N, L, 3) * 0.7 + 0.3, diff=mk(N, D, 3) * 0.5, vis=torch.sigmoid(mk(N, D, 1)))
    lpos = (mk(N, L, 3) * 900.0).to(cuda)
    ppos = (mk(N, D, 3) * 100.0).to(cuda)
    nl = torch.tensor([L, L - 2], dtype=torch.int32, device=cuda)
    w_c, w_s = mk(N, D, 3).to(cuda), mk(N, D, 3).to(cuda)
    outs = []
    for fused in (False, True):
        lv = {k: v.clone().to(cuda).requires_grad_() for k, v in base.items()}
        if fused:
            color, spec = shade_compose(lv["ref_dirs"], lv["sigma"], lv["lint"], lpos, ppos, nl, lv["diff"], lv["vis"],
                                        w_type=w_type, return_spec=True)
        else:
            spec = evaluate_gaussian(lv["ref_dirs"], lv["sigma"], lv["lint"], lpos, ppos, nl, w_type=w_type) * lv["vis"]
            color = (lv["diff"].clamp(min=0.0) + spec).clamp(min=0.0)
        ((color * w_c).sum() + (spec * w_s).sum()).backward()
        outs.append((t2n(color), t2n(spec), {k: t2n(v.grad) for k, v in lv.items()}))
    (c0, s0, g0), (c1, s1, g1) = outs
    assert (c0 < 1e-12).mean() > 0.01, "the outer clamp must be active somewhere in this case"
    # the in-kernel normalisation differs from F.normalize in the last bit of the direction; sharp lobes (sigma -> 0.01)
    # amplify that, hence the absolute tolerance relative to the largest value
    assert_close(c1, c0, rtol=1e-4, atol=1e-5 * np.abs(c0).max(), what="color")
    assert_close(s1, s0, rtol=1e-4, atol=1e-5 * np.abs(s0).max(), what="spec_color")
    for k in g0:
        assert_close(g1[k], g0[k], rtol=2e-4, atol=2e-5 * np.abs(g0[k]).max(), frac=0.9995, what="grad " + k)
