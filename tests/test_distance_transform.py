"""Exact Euclidean distance transform (``distance_transform_edt``, ``tl_edt``) and the Hausdorff distance-transform loss
(``hausdorff_dt_loss``, ``tl_hausdorff_dt_*``).

The transform is pinned bit for bit against ``scipy.ndimage.distance_transform_edt``.  The loss is pinned against a
float64 numpy / scipy restatement of its definition (``ref_cost``), which the CPU tests check on hand-derived cases.
"""
import ctypes
import math
import os
import re

import numpy as np
import pytest
import scipy.ndimage as ndi
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["tl_edt_workspace_bytes", "tl_edt", "tl_hausdorff_dt_workspace_bytes", "tl_hausdorff_dt_forward",
       "tl_hausdorff_dt_backward"]


# ---------------------------------------------------------------- float64 reference of the loss

def ref_field(M: np.ndarray) -> np.ndarray:
    """F(M): the distance to the nearest pixel of the other label if M holds both labels, else 0 (float64)."""
    M = np.asarray(M, dtype=bool)
    if M.all() or not M.any():
        return np.zeros(M.shape)
    return ndi.distance_transform_edt(M) + ndi.distance_transform_edt(~M)


def ref_D(p: np.ndarray, t: np.ndarray, alpha: float) -> np.ndarray:
    """D = F(p > 0.5)^alpha + F(t > 0.5)^alpha for [..., H, W] arrays."""
    p, t = np.asarray(p), np.asarray(t)
    H, W = p.shape[-2:]
    P, T = (p > 0.5).reshape(-1, H, W), (t > 0.5).reshape(-1, H, W)
    D = np.stack([ref_field(a) ** alpha + ref_field(b) ** alpha for a, b in zip(P, T)])
    return D.reshape(p.shape)


def ref_cost(p: np.ndarray, t: np.ndarray, alpha: float) -> np.ndarray:
    """Per-map cost (1 / HW) * sum (p - t)^2 D over the last two axes, float64; p are probabilities."""
    p64, t64 = np.asarray(p, np.float64), np.asarray(t, np.float64)
    return (((p64 - t64) ** 2) * ref_D(p, t, alpha)).mean(axis=(-2, -1))


# ---------------------------------------------------------------- CPU: hand-derived KATs of the reference

def test_kat_single_foreground_pixel_in_3x3():
    t = np.zeros((3, 3))
    t[1, 1] = 1
    r2 = math.sqrt(2.0)
    want = np.array([[r2, 1, r2], [1, 1, 1], [r2, 1, r2]])
    assert np.array_equal(ref_field(t > 0.5), want)


def test_kat_stripe_1xW():
    t = np.array([[0, 0, 1, 1, 1, 0, 0, 0]], dtype=np.float64)
    assert np.array_equal(ref_field(t > 0.5), np.array([[2, 1, 1, 2, 1, 1, 2, 3]], dtype=np.float64))


def test_kat_all_foreground_and_all_background_give_zero_fields():
    assert np.array_equal(ref_field(np.ones((4, 5), bool)), np.zeros((4, 5)))
    assert np.array_equal(ref_field(np.zeros((4, 5), bool)), np.zeros((4, 5)))
    # only the prediction's field counts when the target holds one label
    p = np.array([[0.2, 0.6, 0.7]])
    t = np.ones((1, 3))
    assert ref_cost(p, t, 2.0) == pytest.approx((0.64 * 1 + 0.16 * 1 + 0.09 * 4) / 3, rel=1e-15)
    assert ref_cost(np.full((1, 3), 0.9), t, 2.0) == 0.0  # both single-label: D = 0


@pytest.mark.parametrize("alpha", [1.0, 2.0, 0.5])
def test_kat_costs_for_alpha(alpha):
    # t = [0, 0, 1, 1], p = [0.2, 0.6, 0.7, 0.9]: P = [0, 1, 1, 1], F(P) = [1, 1, 2, 3], F(T) = [2, 1, 1, 2]
    p = np.array([[0.2, 0.6, 0.7, 0.9]])
    t = np.array([[0.0, 0.0, 1.0, 1.0]])
    sq = [0.04, 0.36, 0.09, 0.01]
    fp, ft = [1, 1, 2, 3], [2, 1, 1, 2]
    want = sum(s * (a ** alpha + b ** alpha) for s, a, b in zip(sq, fp, ft)) / 4
    assert {1.0: 0.29, 2.0: 0.375}.get(alpha, want) == pytest.approx(want, rel=1e-12)
    assert ref_cost(p, t, alpha) == pytest.approx(want, rel=1e-12)


# ---------------------------------------------------------------- CPU: the C ABI and the Python checks

def test_new_entry_points_are_declared_exported_and_bound():
    from dilabhelmholtzoct_b200 import _lib, build
    import dilabhelmholtzoct_b200 as tlb
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "topoloss.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(tl_[a-z_0-9]+)\s*\(", src))
    if not os.path.exists(build.LIB_PATH):
        build.build()
    L = ctypes.CDLL(build.LIB_PATH)
    for name in NEW:
        assert name in declared and hasattr(L, name) and name in _lib.SIGNATURES, name
    assert _lib.lib().tl_version() == _lib.ABI_VERSION == 5
    for name in ("distance_transform_edt", "hausdorff_dt_loss"):
        assert name in tlb.__all__ and callable(getattr(tlb, name))


BAD_SHAPES = ((0, 16, 16), (-1, 16, 16), (2, 0, 16), (2, 16, 0), (2, 4097, 16), (2, 16, 4097))


def test_workspace_queries():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    nb, ns, nc = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    assert L.tl_edt_workspace_bytes(3, 16, 16, None) == -1
    assert L.tl_hausdorff_dt_workspace_bytes(3, 16, 16, None, ctypes.byref(nc)) == -1
    assert L.tl_hausdorff_dt_workspace_bytes(3, 16, 16, ctypes.byref(ns), None) == -1
    for bad in BAD_SHAPES:
        assert L.tl_edt_workspace_bytes(*bad, ctypes.byref(nb)) == -1, bad
        assert L.tl_hausdorff_dt_workspace_bytes(*bad, ctypes.byref(ns), ctypes.byref(nc)) == -1, bad
    assert L.tl_edt_workspace_bytes(3, 4096, 4096, ctypes.byref(nb)) == 0 and nb.value == 4 * 3 * 4096 * 4096
    assert L.tl_hausdorff_dt_workspace_bytes(3, 16, 16, ctypes.byref(ns), ctypes.byref(nc)) == 0
    assert (ns.value, nc.value) == (3 * 256 * 4, 3 * 256 * 8)  # D in the state, one uint2 per pixel of scratch


def test_new_entry_points_reject_bad_arguments():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    fake = 4096  # never dereferenced: every call below fails its host-side checks before any launch
    nw = 4 * 3 * 16 * 16
    # tl_edt(mask, n, H, W, spacing, ws, ws_bytes, out, stream); every case fails with a null (unit) or a device spacing
    cases = [(0, None), (5, None), (7, None), (4, fake + 4), (5, fake + 2), (6, nw - 1)]
    cases += [(slice(1, 4), s) for s in BAD_SHAPES]
    for sp in (None, fake):
        ok = [fake, 3, 16, 16, sp, fake, nw, fake, None]
        for i, bad in cases:
            a = list(ok)
            a[i] = bad
            assert L.tl_edt(*a) == -1, (sp, i, bad)
        assert L.tl_edt(*(ok[:6] + [nw - 1] + ok[7:])) == -1 and b"tl_edt_workspace_bytes" in L.tl_last_error()

    ns, nc = 3 * 256 * 4, 3 * 256 * 8
    # tl_hausdorff_dt_forward(logits, target, n, H, W, alpha, spacing, state, state_bytes, scratch, scratch_bytes,
    # cost, stream)
    cases = [(0, None), (1, None), (7, None), (9, None), (11, None), (6, fake + 4), (7, fake + 2), (9, fake + 4),
             (5, 0.0), (5, -1.0), (5, math.inf), (5, -math.inf), (5, math.nan), (8, ns - 1), (10, nc - 1)]
    cases += [(slice(2, 5), s) for s in BAD_SHAPES]
    for sp in (None, fake):
        ok = [fake, fake, 3, 16, 16, 2.0, sp, fake, ns, fake, nc, fake, None]
        for i, bad in cases:
            a = list(ok)
            a[i] = bad
            assert L.tl_hausdorff_dt_forward(*a) == -1, (sp, i, bad)
        assert L.tl_hausdorff_dt_forward(*(ok[:10] + [nc - 1] + ok[11:])) == -1
        assert b"tl_hausdorff_dt_workspace_bytes" in L.tl_last_error()

    ok = [fake, fake, 3, 16, 16, fake, ns, fake, fake, None]
    cases = [(0, None), (1, None), (5, None), (7, None), (8, None), (6, ns - 1), (5, fake + 2)]
    cases += [(slice(2, 5), s) for s in BAD_SHAPES]
    for i, bad in cases:
        a = list(ok)
        a[i] = bad
        assert L.tl_hausdorff_dt_backward(*a) == -1, (i, bad)


def test_python_checks_raise_value_errors_on_the_cpu():
    import dilabhelmholtzoct_b200 as tlb
    with pytest.raises(ValueError, match="CUDA"):
        tlb.distance_transform_edt(torch.zeros(4, 4, dtype=torch.bool))
    with pytest.raises(ValueError, match="CUDA"):
        tlb.hausdorff_dt_loss(torch.zeros(1, 2, 4, 4), torch.zeros(1, 2, 4, 4))
    with pytest.raises(ValueError, match="same shape"):
        tlb.hausdorff_dt_loss(torch.zeros(1, 2, 4, 4), torch.zeros(1, 2, 4, 5))
    with pytest.raises(ValueError):
        tlb.distance_transform_edt(torch.zeros(4, dtype=torch.bool))
    with pytest.raises(TypeError):
        tlb.hausdorff_dt_loss(np.zeros((1, 1, 2, 2)), torch.zeros(1, 1, 2, 2))


# ---------------------------------------------------------------- GPU: the transform against scipy

def _check_edt(m: torch.Tensor):
    """distance_transform_edt(m) equals scipy per map bit for bit; maps without a zero pixel are +inf."""
    import dilabhelmholtzoct_b200 as tlb
    got = tlb.distance_transform_edt(m)
    assert got.dtype == torch.float32 and got.shape == m.shape and got.device == m.device
    H, W = m.shape[-2:]
    g = got.cpu().numpy().reshape(-1, H, W)
    for k, mk in enumerate(m.cpu().numpy().reshape(-1, H, W)):
        if (mk != 0).all():
            assert np.isposinf(g[k]).all(), k
        else:
            want = ndi.distance_transform_edt(mk != 0).astype(np.float32)
            assert np.array_equal(g[k], want), (k, np.abs(g[k] - want).max())


SHAPES = [(1, 1), (1, 4096), (4096, 1), (37, 53), (496, 512), (1024, 1024)]


@pytest.mark.gpu
@pytest.mark.parametrize("density", [0.01, 0.5, 0.99])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_edt_equals_scipy_on_random_masks(shape, density):
    rng = np.random.default_rng(hash((shape, density)) % 2 ** 32)
    n = 1 if shape[0] * shape[1] >= 496 * 512 else 6
    m = torch.from_numpy(rng.random((n,) + shape) < density).cuda()
    _check_edt(m)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 1), (3, 3), (37, 53), (256, 256), (4096, 1)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_edt_single_pixel_single_zero_all_zero_and_all_one_maps(shape):
    rng = np.random.default_rng(5)
    H, W = shape
    m = np.zeros((6, H, W), np.uint8)
    for k in range(2):                          # one feature pixel
        m[k, rng.integers(H), rng.integers(W)] = 1
    m[2:4] = 1                                  # one zero pixel
    for k in (2, 3):
        m[k, rng.integers(H), rng.integers(W)] = 0
    m[5] = 1                                    # all one: +inf; m[4] all zero: 0
    mt = torch.from_numpy(m).cuda()
    _check_edt(mt)
    got = __import__("dilabhelmholtzoct_b200").distance_transform_edt(mt)
    assert bool((got[4] == 0).all()) and bool(torch.isposinf(got[5]).all())


@pytest.mark.gpu
def test_edt_equals_scipy_on_synthetic_layer_masks():
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(2, 496, 512, seed=11, device="cuda")
    _check_edt(truth > 0.5)
    _check_edt(pred > 0.5)
    _check_edt(pred < 0.5)


@pytest.mark.gpu
def test_edt_uint8_values_bool_and_non_contiguous_inputs():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(2)
    vals = rng.integers(0, 4, (3, 40, 70)).astype(np.uint8) * 85  # 0, 85, 170, 255: nonzero is a feature
    u8 = torch.from_numpy(vals).cuda()
    _check_edt(u8)
    assert torch.equal(tlb.distance_transform_edt(u8), tlb.distance_transform_edt(u8 != 0))
    nc = u8.transpose(1, 2)[:, ::2, 1:]                                   # non-contiguous view
    assert not nc.is_contiguous()
    _check_edt(nc)
    _check_edt((u8 > 100).unsqueeze(0).expand(2, 3, 40, 70))            # extra leading dims, stride 0
    with pytest.raises(ValueError):
        tlb.distance_transform_edt(u8.float())
    with pytest.raises(ValueError):
        tlb.distance_transform_edt(torch.zeros(2, 4097, 3, dtype=torch.bool, device="cuda"))
    empty = tlb.distance_transform_edt(torch.zeros(0, 5, 6, dtype=torch.bool, device="cuda"))
    assert empty.shape == (0, 5, 6) and empty.dtype == torch.float32


# ---------------------------------------------------------------- GPU: the loss

def _ref_on(x: torch.Tensor, t: torch.Tensor, alpha: float) -> np.ndarray:
    p = torch.sigmoid(x).cpu().numpy()  # the fp32 p of the device, as the op computes it
    return ref_cost(p, t.float().cpu().numpy(), alpha)


def _random_batch(B, C, H, W, seed, scale=3.0):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    x = scale * torch.randn((B, C, H, W), generator=g, device="cuda")
    t = (torch.rand((B, C, H, W), generator=g, device="cuda") < 0.5).float()
    return x, t


@pytest.mark.gpu
def test_threshold_agrees_with_torch_sigmoid_at_the_boundary():
    import dilabhelmholtzoct_b200 as tlb
    f = lambda bits: torch.tensor([bits], dtype=torch.int32, device="cuda").view(torch.float32)  # noqa: E731
    lo, hi = 0, int(np.float32(1.0).view(np.int32))  # sigmoid(+0) = 0.5 is not > 0.5; sigmoid(1) is
    assert not bool(torch.sigmoid(f(lo)) > 0.5) and bool(torch.sigmoid(f(hi)) > 0.5)
    while hi - lo > 1:  # positive floats order like their bits
        mid = (lo + hi) // 2
        if bool(torch.sigmoid(f(mid)) > 0.5):
            hi = mid
        else:
            lo = mid
    c, below = f(hi).item(), f(lo).item()
    assert below < c
    probes = torch.tensor([c, below, 0.0, -0.0, 1.4e-45, -1.4e-45, 1e-40, -1e-40, math.nan, -c, 2 * c],
                          dtype=torch.float32, device="cuda")
    K = probes.numel()
    # per map [1, 4]: x = [-20, v, -20, -20], target all 0.  P holds one label unless v is labelled 1, and then
    # F(P) = [1, 1, 1, 2]: the cost is 0 exactly iff sigmoid(v) > 0.5 is false
    x = torch.full((1, K, 1, 4), -20.0, device="cuda")
    x[0, :, 0, 1] = probes
    cost = tlb.hausdorff_dt_loss(x, torch.zeros_like(x))
    want = torch.sigmoid(probes) > 0.5
    got = cost[0] != 0
    nan_map = 8
    assert torch.isnan(cost[0, nan_map])  # a NaN logit: NaN cost, and P is 0 there (sigmoid(NaN) > 0.5 is false)
    keep = torch.arange(K, device="cuda") != nan_map
    assert torch.equal(got[keep], want[keep]), (probes, cost, want)
    assert bool(want[0]) and not bool(want[1])


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", [2.0, 1.0, 0.5, 3.7])
def test_cost_equals_the_float64_reference_on_random_w1_batches(alpha):
    import dilabhelmholtzoct_b200 as tlb
    B = 64 if alpha == 2.0 else 4
    x, t = _random_batch(B, 14, 256, 256, seed=int(alpha * 10))
    cost = tlb.hausdorff_dt_loss(x, t, alpha)
    assert cost.shape == (B, 14) and cost.dtype == torch.float32
    np.testing.assert_allclose(cost.cpu().numpy(), _ref_on(x, t, alpha), rtol=1e-6, atol=0)


@pytest.mark.gpu
def test_cost_equals_the_float64_reference_on_synthetic_batches():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    for B, H, W in ((4, 256, 256), (1, 496, 512), (2, 37, 53)):
        pred, truth = make_batch(B, H, W, seed=H, device="cuda")
        x = torch.logit(pred.clamp(1e-6, 1 - 1e-6))
        np.testing.assert_allclose(tlb.hausdorff_dt_loss(x, truth).cpu().numpy(), _ref_on(x, truth, 2.0), rtol=1e-6, atol=0)
        # soft targets are thresholded for the field but enter (p - t)^2 as they are
        np.testing.assert_allclose(tlb.hausdorff_dt_loss(x, pred, 1.5).cpu().numpy(), _ref_on(x, pred, 1.5), rtol=1e-6, atol=0)


@pytest.mark.gpu
def test_cost_with_single_label_prediction_target_or_both():
    import dilabhelmholtzoct_b200 as tlb
    x, t = _random_batch(3, 4, 30, 41, seed=9)
    x[:, 0] = 25.0   # prediction all foreground
    x[:, 1] = -25.0  # prediction all background
    t[0, :] = 1.0    # target all foreground
    t[1, :] = 0.0    # target all background
    cost = tlb.hausdorff_dt_loss(x, t)
    np.testing.assert_allclose(cost.cpu().numpy(), _ref_on(x, t, 2.0), rtol=1e-6, atol=0)
    assert bool((cost[:2, :2] == 0).all())  # both single-label: a zero field


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", [2.0, 0.5])
def test_gradient_equals_autograd_of_the_composed_form(alpha):
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(2, 96, 128, seed=4, device="cuda")
    xr, tr = _random_batch(2, 14, 96, 128, seed=5)
    x = torch.cat([torch.logit(pred.clamp(1e-6, 1 - 1e-6)), xr, 2 * xr])  # 2x: some p saturate to 1, zero gradients
    t = torch.cat([truth, tr, tr])
    x[0, 3] = 25.0                                                           # single-label prediction
    w = torch.rand(x.shape[:2], device="cuda") + 0.5                         # an upstream gradient per map
    a = x.clone().requires_grad_(True)
    (tlb.hausdorff_dt_loss(a, t, alpha) * w).sum().backward()
    p0 = torch.sigmoid(x).cpu().numpy()
    D = torch.from_numpy(ref_D(p0, t.cpu().numpy(), alpha)).float().cuda()   # the field from scipy
    b = x.clone().requires_grad_(True)
    p = torch.sigmoid(b)
    (((p - t) ** 2 * D).mean((2, 3)) * w).sum().backward()
    assert torch.equal(a.grad == 0, b.grad == 0)
    torch.testing.assert_close(a.grad, b.grad, rtol=1e-5, atol=1e-35)


@pytest.mark.gpu
def test_two_runs_are_bit_identical():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(8, 256, 256, seed=3, device="cuda")
    x = torch.logit(pred.clamp(1e-6, 1 - 1e-6))
    outs = []
    for _ in range(2):
        a = x.clone().requires_grad_(True)
        c = tlb.hausdorff_dt_loss(a, truth)
        c.sum().backward()
        outs.append((c.detach(), a.grad))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


@pytest.mark.gpu
def test_forward_backward_and_transform_make_no_host_sync():
    import dilabhelmholtzoct_b200 as tlb
    x, t = _random_batch(2, 3, 64, 64, seed=1)
    tlb.hausdorff_dt_loss(x.clone().requires_grad_(True), t).sum().backward()  # warm: library loaded, scratch grown
    m = t > 0.5
    tlb.distance_transform_edt(m)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        a = x.clone().requires_grad_(True)
        tlb.hausdorff_dt_loss(a, t, 1.0).sum().backward()
        d = tlb.distance_transform_edt(m)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert bool(torch.isfinite(a.grad).all()) and d.shape == m.shape


@pytest.mark.gpu
def test_nan_logit_gives_nan_cost_for_its_map_only():
    import dilabhelmholtzoct_b200 as tlb
    x, t = _random_batch(2, 3, 32, 32, seed=6)
    x[1, 2, 5, 7] = math.nan
    a = x.clone().requires_grad_(True)
    cost = tlb.hausdorff_dt_loss(a, t).detach()
    nan = torch.isnan(cost)
    assert bool(nan[1, 2]) and int(nan.sum()) == 1
    keep = ~nan
    np.testing.assert_allclose(cost[keep].cpu().numpy(), _ref_on(x, t, 2.0)[keep.cpu().numpy()], rtol=1e-6, atol=0)


@pytest.mark.gpu
def test_empty_batch_and_no_gradient_for_the_target():
    import dilabhelmholtzoct_b200 as tlb
    for shape in ((0, 14, 16, 16), (2, 0, 8, 8)):
        x = torch.zeros(shape, device="cuda", requires_grad=True)
        c = tlb.hausdorff_dt_loss(x, torch.zeros(shape, device="cuda"))
        assert c.shape == shape[:2] and c.requires_grad
        c.sum().backward()
        assert x.grad.shape == shape
    x, t = _random_batch(1, 2, 16, 16, seed=7)
    a, g = x.clone().requires_grad_(True), t.clone().requires_grad_(True)
    tlb.hausdorff_dt_loss(a, g).sum().backward()
    assert a.grad is not None and g.grad is None
    # other target dtypes are cast to float32 first
    for dt in (torch.bool, torch.uint8, torch.float64, torch.float16):
        np.testing.assert_array_equal(tlb.hausdorff_dt_loss(x, t.to(dt)).cpu().numpy(),
                                      tlb.hausdorff_dt_loss(x, t).cpu().numpy())


@pytest.mark.gpu
def test_python_checks_on_the_gpu():
    import dilabhelmholtzoct_b200 as tlb
    x = torch.zeros(1, 2, 8, 8, device="cuda")
    with pytest.raises(ValueError, match="float32"):
        tlb.hausdorff_dt_loss(x.double(), x)
    with pytest.raises(ValueError, match="same shape"):
        tlb.hausdorff_dt_loss(x, x[:, :1])
    with pytest.raises(ValueError, match="same shape"):
        tlb.hausdorff_dt_loss(x[0], x[0])
    with pytest.raises(ValueError, match="real or bool"):
        tlb.hausdorff_dt_loss(x, x.to(torch.complex64))
    for alpha in (0.0, -1.0, math.inf, math.nan):
        with pytest.raises(ValueError, match="alpha"):
            tlb.hausdorff_dt_loss(x, x, alpha)
    with pytest.raises(ValueError, match="4096"):
        tlb.hausdorff_dt_loss(torch.zeros(1, 1, 4097, 2, device="cuda"), torch.zeros(1, 1, 4097, 2, device="cuda"))
