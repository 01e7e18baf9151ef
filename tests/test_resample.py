"""F1 (SURVEY.md 8f): the fused sigmoid + bilinear(align_corners=True) resample in front of the path.

CPU part: the oracle restatement (oracle/resample_oracle.py) against the reference's own
implementation of this step -- PyTorch on CPU -- and against the committed golden vectors.
GPU part (-m gpu): tl_resample_forward / tl_resample_backward through the C ABI against the oracle,
the golden vectors and torch on the GPU, and the fused call-site function against the two-step form."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import resample_oracle as ro

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "resample_small.npz")
FWD_TOL = 2e-6   # absolute, values in [0, 1] (sigmoid) / O(10) (plain): fp32 rounding of the 4-tap blend
BWD_TOL = 1e-5   # relative to the largest gradient entry (atomics: summation order is not fixed)


def _cases():
    z = np.load(GOLD)
    k = 0
    while f"x{k}" in z:
        for sig in (0, 1):
            yield k, sig, z[f"x{k}"], z[f"g{k}"], z[f"y{k}_{sig}"], z[f"gx{k}_{sig}"]
        k += 1


def test_oracle_matches_golden_vectors():
    n = 0
    for k, sig, x, g, y, gx in _cases():
        got = ro.resample(x, y.shape[-1], bool(sig))
        assert np.abs(got - y).max() <= FWD_TOL * max(1.0, np.abs(y).max()), (k, sig)
        gb = ro.resample_backward(g, x, bool(sig))
        assert np.abs(gb - gx).max() <= BWD_TOL * np.abs(gx).max(), (k, sig)
        n += 1
    assert n >= 8


@pytest.mark.parametrize("shape,S", [((1, 2, 9, 13), 5), ((2, 1, 40, 40), 50), ((1, 1, 7, 7), 1), ((1, 3, 2, 2), 6)])
def test_oracle_matches_pytorch_cpu(shape, S):
    rng = np.random.default_rng(sum(shape) + S)
    x = (2.0 * rng.standard_normal(shape)).astype(np.float32)
    for sig in (False, True):
        t = torch.from_numpy(x).clone().requires_grad_(True)
        y = F.interpolate(torch.sigmoid(t) if sig else t, size=(S, S), mode="bilinear", align_corners=True)
        g = rng.standard_normal(y.shape).astype(np.float32)
        y.backward(torch.from_numpy(g))
        assert np.abs(ro.resample(x, S, sig) - y.detach().numpy()).max() <= FWD_TOL * max(1.0, float(y.abs().max()))
        assert np.abs(ro.resample_backward(g, x, sig) - t.grad.numpy()).max() <= BWD_TOL * float(t.grad.abs().max())


def test_identity_size_is_exact():
    x = np.random.default_rng(1).standard_normal((2, 8, 8)).astype(np.float32)
    assert np.array_equal(ro.resample(x, 8, False), x)


# ------------------------------------------------------------------ GPU, through the C ABI

@pytest.mark.gpu
def test_gpu_resample_matches_golden_and_oracle():
    import dilabhelmholtzoct_b200 as tlb
    for k, sig, x, g, y, gx in _cases():
        t = torch.from_numpy(x).cuda().requires_grad_(True)
        out = tlb.resample(t, y.shape[-1], sigmoid=bool(sig))
        out.backward(torch.from_numpy(g).cuda())
        assert np.abs(out.detach().cpu().numpy() - y).max() <= FWD_TOL * max(1.0, np.abs(y).max()), (k, sig)
        assert np.abs(out.detach().cpu().numpy() - ro.resample(x, y.shape[-1], bool(sig))).max() <= FWD_TOL * max(1.0, np.abs(y).max())
        assert np.abs(t.grad.cpu().numpy() - gx).max() <= BWD_TOL * np.abs(gx).max(), (k, sig)


@pytest.mark.gpu
def test_gpu_resample_callsite_shape_against_torch_gpu():
    """496x512 -> 50x50 (the reference call site's sizes), against torch.sigmoid + F.interpolate on the GPU."""
    import dilabhelmholtzoct_b200 as tlb
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = 3.0 * torch.randn((4, 14, 496, 512), device="cuda", generator=gen)
    g = torch.randn((4, 14, 50, 50), device="cuda", generator=gen)
    for sig in (False, True):
        a = x.clone().requires_grad_(True)
        b = x.clone().requires_grad_(True)
        ya = tlb.resample(a, 50, sigmoid=sig)
        yb = F.interpolate(torch.sigmoid(b) if sig else b, size=(50, 50), mode="bilinear", align_corners=True)
        ya.backward(g)
        yb.backward(g)
        assert float((ya - yb).abs().max()) <= FWD_TOL * max(1.0, float(yb.abs().max()))
        assert float((a.grad - b.grad).abs().max()) <= BWD_TOL * float(b.grad.abs().max())
        assert int((a.grad != 0).sum()) == int((b.grad != 0).sum())


@pytest.mark.gpu
def test_gpu_fused_callsite_equals_two_step_form():
    """topo_loss_from_logits(masks, gt, ...) == topo_loss(resample(sigmoid), resample(gt), ...) exactly, and
    agrees with the reference's two-step form on torch's own resample within the north-star tolerance."""
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(2, 96, 96, seed=77, device="cuda", n_classes=5)
    logits = torch.logit(pred.clamp(1e-4, 1 - 1e-4))
    a = logits.clone().requires_grad_(True)
    la = tlb.topo_loss_from_logits(a, truth, 0.1, feat_d=1, interp=50)
    la.backward()
    b = logits.clone().requires_grad_(True)
    lb = tlb.topo_loss(tlb.resample(b, 50, sigmoid=True), tlb.resample(truth, 50), 0.1, feat_d=1)
    lb.backward()
    assert float(la) == float(lb)
    assert torch.equal(a.grad, b.grad)
    c = logits.clone().requires_grad_(True)
    lc = tlb.topo_loss(torch.sigmoid(c), truth, 0.1, feat_d=1, interp=50)   # torch's sigmoid + F.interpolate
    lc.backward()
    assert abs(float(la) - float(lc)) <= 1e-5 * abs(float(lc))
    assert float((a.grad - c.grad).abs().max()) <= 1e-4 * float(c.grad.abs().max())
    # interp = 0: the fused form is the plain sigmoid
    d = logits.clone().requires_grad_(True)
    ld = tlb.topo_loss_from_logits(d, truth, 0.1, feat_d=1)
    e = logits.clone().requires_grad_(True)
    le = tlb.topo_loss(torch.sigmoid(e), truth, 0.1, feat_d=1)
    ld.backward(); le.backward()
    assert abs(float(ld) - float(le)) <= 1e-5 * abs(float(le))
    assert float((d.grad - e.grad).abs().max()) <= 1e-4 * float(e.grad.abs().max())


# ------------------------------------------------------------------ F3: SAM post-processing chain

def _torch_chain(x, T, rh, rw, oh, ow):
    m = F.interpolate(x, (T, T), mode="bilinear", align_corners=False)
    m = m[..., :rh, :rw]
    return F.interpolate(m, (oh, ow), mode="bilinear", align_corners=False)


@pytest.mark.parametrize("Hs,T,rh,rw,oh,ow", [(16, 64, 62, 64, 31, 32), (8, 32, 32, 20, 50, 33), (12, 24, 24, 24, 7, 9)])
def test_postprocess_oracle_matches_pytorch_cpu(Hs, T, rh, rw, oh, ow):
    rng = np.random.default_rng(Hs + T + oh)
    x = (2.0 * rng.standard_normal((2, 3, Hs, Hs))).astype(np.float32)
    want = _torch_chain(torch.from_numpy(x), T, rh, rw, oh, ow).numpy()
    got = ro.postprocess(x, T, rh, rw, oh, ow)
    assert np.abs(got - want).max() <= FWD_TOL * max(1.0, np.abs(want).max())


@pytest.mark.gpu
@pytest.mark.parametrize("Hs,T,rh,rw,oh,ow,n", [(256, 1024, 992, 1024, 496, 512, 6), (64, 256, 256, 200, 300, 123, 4),
                                               (32, 64, 64, 64, 700, 650, 2), (16, 64, 62, 64, 31, 32, 5)])
def test_gpu_postprocess_matches_torch_and_oracle(Hs, T, rh, rw, oh, ow, n):
    """Forward against the oracle and torch's two-step chain on the GPU; backward against torch autograd
    (the third case up-samples, so the backward takes the scatter kernel; every tile's source window still fits
    in shared memory.  tests/test_fused_ops_edges.py reaches the global-atomic fallback and the other paths.)"""
    import dilabhelmholtzoct_b200 as tlb
    gen = torch.Generator(device="cuda").manual_seed(Hs + oh)
    x = 3.0 * torch.randn((n, Hs, Hs), device="cuda", generator=gen)
    g = torch.randn((n, oh, ow), device="cuda", generator=gen)
    a = x.clone().requires_grad_(True)
    b = x.clone().requires_grad_(True)
    ya = tlb.postprocess_masks(a, (rh, rw), (oh, ow), padded_size=T)
    yb = _torch_chain(b[None], T, rh, rw, oh, ow)[0]
    ya.backward(g)
    yb.backward(g)
    scale = max(1.0, float(yb.abs().max()))
    assert float((ya - yb).abs().max()) <= FWD_TOL * scale
    assert np.abs(ya.detach().cpu().numpy() - ro.postprocess(x.cpu().numpy(), T, rh, rw, oh, ow)).max() <= FWD_TOL * scale
    assert float((a.grad - b.grad).abs().max()) <= BWD_TOL * float(b.grad.abs().max())
