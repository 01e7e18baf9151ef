"""The boundary loss of Kervadec et al. and its signed distance map: ``boundary_loss`` and ``signed_distance_map``
(``tl_boundary_*``, ``tl_signed_distance*``, DESIGN §3.11).

The contract: on a map holding both labels, ``phi`` is the float64 expression
``edt(~M, sampling) * ~M - (edt(M, sampling) - 1) * M`` with scipy's ``distance_transform_edt``, rounded to float32;
on a map with one label only it is 0.  ``ref_phi`` is exactly that.  The GPU tests pin the map op to it bit for bit
(as uint32 patterns, so the sign of zero counts) and the loss to a float64 restatement built on the op's ``p`` and
``phi``.
"""
import ctypes
import math

import numpy as np
import pytest
import scipy.ndimage as ndi
import torch

SPACINGS = [(3.87, 11.29), (1.0, 3.0), (0.5, 1.25), (1e-3, 1.0), (1.0, 1000.0), (1e-6, 1e6)]


# ---------------------------------------------------------------- float64 references

def ref_phi(M, sampling=None) -> np.ndarray:
    """Kervadec's ``one_hot2dist`` expression for one map in float64, plus the single-label rule (0 everywhere)."""
    M = np.asarray(M, bool)
    if M.all() or not M.any():
        return np.zeros(M.shape)
    kw = {} if sampling is None else {"sampling": tuple(float(v) for v in sampling)}
    return ndi.distance_transform_edt(~M, **kw) * ~M - (ndi.distance_transform_edt(M, **kw) - 1) * M


def ref_cost_grad(p, phi, g):
    """Per-map cost and gradient of the loss in float64 from float32 ``p`` and ``phi`` ``[n, H, W]`` and ``g`` ``[n]``."""
    p64, f64 = p.astype(np.float64), phi.astype(np.float64)
    H, W = p.shape[-2:]
    cost = (p64 * f64).sum(axis=(1, 2)) / (H * W)
    grad = g.astype(np.float64)[:, None, None] * (1.0 / (H * W)) * f64 * p64 * (1.0 - p64)
    return cost, grad, np.abs(p64 * f64).mean(axis=(1, 2))


def _bits(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# ---------------------------------------------------------------- CPU: the reference and hand-derived cases

def test_kat_stripe():
    m = np.array([[0, 0, 1, 1, 1, 0, 0, 0]], bool)
    assert ref_phi(m).tolist() == [[2, 1, 0, -1, 0, 1, 2, 3]]


def test_kat_block_in_a_square_unit_and_anisotropic():
    m = np.zeros((5, 5), bool)
    m[1:4, 1:4] = True
    phi = ref_phi(m)
    r2 = math.sqrt(2.0)
    assert phi.tolist() == [[r2, 1, 1, 1, r2], [1, 0, 0, 0, 1], [1, 0, -1, 0, 1], [1, 0, 0, 0, 1], [r2, 1, 1, 1, r2]]
    phi = ref_phi(m, (1.0, 3.0))  # a row is 1, a column 3: corners sqrt(1 + 9), the centre row's inner pixels -1
    r10 = math.sqrt(10.0)
    assert phi.tolist() == [[r10, 1, 1, 1, r10], [3, 0, 0, 0, 3], [3, -1, -1, -1, 3], [3, 0, 0, 0, 3],
                            [r10, 1, 1, 1, r10]]


def test_kat_single_label_maps_are_zero():
    for m in (np.zeros((4, 6), bool), np.ones((4, 6), bool)):
        for sp in (None, (2.0, 0.5)):
            phi = ref_phi(m, sp)
            assert phi.shape == (4, 6) and not phi.any() and not np.signbit(phi).any()


def test_kat_zero_on_the_inner_boundary_is_positive():
    # 1 - 1 and 0 - (1 - 1) are both +0: the contract's sign of zero
    phi = ref_phi(np.array([[0, 1, 1, 1, 0]], bool)).astype(np.float32)
    assert _bits(phi[0]).tolist() == _bits([1.0, 0.0, -1.0, 0.0, 1.0]).tolist()


def test_kat_cost():
    # the stripe at p = sigmoid(0) = 1/2: cost = (1/2) * (2 + 1 + 0 - 1 + 0 + 1 + 2 + 3) / 8 = 1/2
    m = np.array([[0, 0, 1, 1, 1, 0, 0, 0]], bool)
    p = np.full((1, 1, 8), 0.5, np.float32)
    phi = ref_phi(m).astype(np.float32)[None]
    cost, grad, _ = ref_cost_grad(p, phi, np.ones(1, np.float32))
    assert cost.tolist() == [0.5]
    assert grad[0, 0].tolist() == [v / 32 for v in (2, 1, 0, -1, 0, 1, 2, 3)]


# ---------------------------------------------------------------- CPU: the C ABI

NEW_NAMES = ("tl_boundary_workspace_bytes", "tl_boundary_forward", "tl_boundary_backward", "tl_signed_distance")
BAD_SHAPES = ((0, 16, 16), (-1, 16, 16), (2, 0, 16), (2, 16, 0), (2, 4097, 16), (2, 16, 4097))


def test_new_entry_points_are_declared_exported_and_bound():
    import os
    import re
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(root, "include", "topoloss.h")).read(), flags=re.S)
    for name in NEW_NAMES:
        assert re.search(rf"\b{name}\s*\(", src) and name in _lib.SIGNATURES and hasattr(_lib.lib(), name), name
    for name in ("tl_boundary_forward_spaced", "tl_signed_distance_spaced"):  # ABI 5: spacing is an argument
        assert not re.search(rf"\b{name}\s*\(", src) and name not in _lib.SIGNATURES and not hasattr(_lib.lib(), name)
    assert _lib.lib().tl_version() == _lib.ABI_VERSION == 5
    for name in ("boundary_loss", "signed_distance_map"):
        assert name in tlb.__all__ and callable(getattr(tlb, name))


def test_workspace_query():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    ns, nc = ctypes.c_size_t(0), ctypes.c_size_t(0)
    assert L.tl_boundary_workspace_bytes(3, 16, 16, ctypes.byref(ns), ctypes.byref(nc)) == 0
    assert (ns.value, nc.value) == (4 * 3 * 256, 8 * 3 * 256)
    assert L.tl_boundary_workspace_bytes(2, 4096, 4096, ctypes.byref(ns), ctypes.byref(nc)) == 0
    assert (ns.value, nc.value) == (4 * 2 * 4096 ** 2, 8 * 2 * 4096 ** 2)
    for n, H, W in BAD_SHAPES:
        assert L.tl_boundary_workspace_bytes(n, H, W, ctypes.byref(ns), ctypes.byref(nc)) == -1
    assert L.tl_boundary_workspace_bytes(3, 16, 16, None, ctypes.byref(nc)) == -1
    assert L.tl_boundary_workspace_bytes(3, 16, 16, ctypes.byref(ns), None) == -1


def _all_fail(fn, ok, cases):
    for i, bad in cases:
        a = list(ok)
        a[i] = bad
        assert fn(*a) == -1, (i, bad)


def _short_buffer_names_the_query(fn, args):
    from dilabhelmholtzoct_b200 import _lib
    assert fn(*args) == -1
    assert "tl_boundary_workspace_bytes" in _lib.lib().tl_last_error().decode()


def test_new_entry_points_reject_bad_arguments():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    fake = 4096  # never dereferenced: every call below fails its host-side checks before any launch
    ns, nc = 3 * 256 * 4, 3 * 256 * 8
    shapes = lambda at: [(slice(at, at + 3), s) for s in BAD_SHAPES]  # noqa: E731

    # tl_boundary_forward(logits, target, n, H, W, spacing, state, state_bytes, scratch, scratch_bytes, cost, stream);
    # every case fails with a null (unit) or a device spacing
    for sp in (None, fake):
        ok = [fake, fake, 3, 16, 16, sp, fake, ns, fake, nc, fake, None]
        _all_fail(L.tl_boundary_forward, ok, [(0, None), (1, None), (6, None), (8, None), (10, None), (5, fake + 4),
                                              (6, fake + 2), (8, fake + 4), (7, ns - 1), (9, nc - 1)] + shapes(2))
        for i, bad in ((7, ns - 1), (9, nc - 1)):
            a = list(ok)
            a[i] = bad
            _short_buffer_names_the_query(L.tl_boundary_forward, a)

    # tl_boundary_backward(logits, n, H, W, state, state_bytes, grad_cost, grad_logits, stream)
    ok = [fake, 3, 16, 16, fake, ns, fake, fake, None]
    _all_fail(L.tl_boundary_backward, ok, [(0, None), (4, None), (6, None), (7, None), (4, fake + 2), (5, ns - 1)]
              + shapes(1))
    a = list(ok)
    a[5] = ns - 1
    _short_buffer_names_the_query(L.tl_boundary_backward, a)

    # tl_signed_distance(mask, n, H, W, spacing, scratch, scratch_bytes, out, stream)
    for sp in (None, fake):
        ok = [fake, 3, 16, 16, sp, fake, nc, fake, None]
        _all_fail(L.tl_signed_distance, ok, [(0, None), (5, None), (7, None), (4, fake + 4), (5, fake + 4), (6, nc - 1)]
                  + shapes(1))
        a = list(ok)
        a[6] = nc - 1
        _short_buffer_names_the_query(L.tl_signed_distance, a)


def test_python_checks_raise_on_the_cpu():
    import dilabhelmholtzoct_b200 as tlb
    m = torch.zeros(2, 3, 4, 4, dtype=torch.bool)
    x = torch.zeros(2, 3, 4, 4)
    with pytest.raises(TypeError):
        tlb.signed_distance_map(m.numpy())
    with pytest.raises(TypeError):
        tlb.boundary_loss(x, m.numpy())
    with pytest.raises(ValueError, match="CUDA"):
        tlb.signed_distance_map(m)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.signed_distance_map(m, sampling=(1.0, 2.0))
    with pytest.raises(ValueError, match="CUDA"):
        tlb.boundary_loss(x, m)
    with pytest.raises(ValueError):
        tlb.signed_distance_map(torch.zeros(4, dtype=torch.bool))
    with pytest.raises(ValueError):
        tlb.boundary_loss(x, x[:, :2])
    with pytest.raises(ValueError):
        tlb.boundary_loss(x[0], x[0])


# ---------------------------------------------------------------- GPU: the map

def _check_map(m: torch.Tensor, sampling=None):
    import dilabhelmholtzoct_b200 as tlb
    got = tlb.signed_distance_map(m, sampling=sampling)
    assert got.dtype == torch.float32 and got.shape == m.shape and not got.requires_grad
    H, W = m.shape[-2:]
    maps = (m.cpu().numpy() != 0).reshape(-1, H, W)
    if sampling is None:
        sp = [None] * len(maps)
    else:
        sp = np.broadcast_to(np.asarray(sampling, np.float64), m.shape[:-2] + (2,)).reshape(-1, 2)
    g = got.cpu().numpy().reshape(-1, H, W)
    for k, (mm, s) in enumerate(zip(maps, sp)):
        want = ref_phi(mm, s).astype(np.float32)
        assert np.array_equal(_bits(g[k]), _bits(want)), (k, s, np.abs(g[k] - want).max())
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("sampling", [None] + SPACINGS, ids=str)
@pytest.mark.parametrize("density", [0.01, 0.5, 0.99])
def test_map_equals_the_reference_on_random_masks(sampling, density):
    rng = np.random.default_rng(int(density * 1000) + (0 if sampling is None else int(sampling[0] * 97)))
    for shape in ((1, 1), (1, 97), (89, 1), (31, 127), (61, 53)):
        _check_map(torch.from_numpy(rng.random((3,) + shape) < density).cuda(), sampling)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(496, 512), (1, 4096), (4096, 3)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_map_large_shapes(shape):
    rng = np.random.default_rng(shape[0] + shape[1])
    m = np.stack([rng.random(shape) < d for d in (0.01, 0.5, 0.99)])
    for sp in (None, (3.87, 11.29), (1.0, 1000.0)):
        _check_map(torch.from_numpy(m).cuda(), sp)


@pytest.mark.gpu
def test_map_layer_masks_single_label_and_per_map_spacing():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    _, truth = make_batch(2, 128, 160, seed=5, device="cuda")
    m = truth > 0.5
    m[0, 0] = False                                             # all background
    m[1, 1] = True                                              # all foreground
    for sp in (None, (3.87, 11.29), (1.0, 3.0), np.random.default_rng(1).uniform(0.05, 20.0, tuple(m.shape[:2]) + (2,))):
        got = _check_map(m, sp)
        assert not got[0, 0].any() and not got[1, 1].any()
        assert not torch.signbit(got[0, 0]).any() and not torch.signbit(got[1, 1]).any()
    unit = tlb.signed_distance_map(m)
    for sp in ((1, 1), 1.0, np.ones(tuple(m.shape[:2]) + (2,))):
        assert torch.equal(tlb.signed_distance_map(m, sampling=sp).view(torch.int32), unit.view(torch.int32))
    assert torch.equal(tlb.signed_distance_map(m.to(torch.uint8) * 7).view(torch.int32), unit.view(torch.int32))


# ---------------------------------------------------------------- GPU: the loss

def _batch(B, C, H, W, seed, density=0.5, scale=3.0):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    x = scale * torch.randn((B, C, H, W), generator=g, device="cuda")
    t = (torch.rand((B, C, H, W), generator=g, device="cuda") < density).float()
    return x, t


def _check_loss(x, t, spacing=None):
    """Cost and gradient against the float64 restatement on the op's p and phi, and against torch autograd."""
    import dilabhelmholtzoct_b200 as tlb
    xr = x.detach().clone().requires_grad_(True)
    cost = tlb.boundary_loss(xr, t, spacing=spacing)
    assert cost.dtype == torch.float32 and cost.shape == x.shape[:2]
    g_cost = torch.linspace(0.5, 1.5, cost.numel(), device="cuda").reshape(cost.shape)
    (cost * g_cost).sum().backward()
    H, W = x.shape[-2:]
    phi = tlb.signed_distance_map(t > 0.5, sampling=spacing)
    p = torch.sigmoid(x.detach())
    want, wgrad, mabs = ref_cost_grad(p.cpu().numpy().reshape(-1, H, W), phi.cpu().numpy().reshape(-1, H, W),
                                      g_cost.cpu().numpy().reshape(-1))
    got = cost.detach().cpu().numpy().reshape(-1).astype(np.float64)
    tol = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64) + 2.0 ** -40 * mabs
    assert (np.abs(got - want) <= tol).all(), (got, want)
    gg = xr.grad.cpu().numpy().reshape(-1, H, W).astype(np.float64)
    gtol = np.spacing(np.abs(wgrad).astype(np.float32)).astype(np.float64)
    assert (np.abs(gg - wgrad) <= gtol).all(), np.abs(gg - wgrad).max()
    # torch autograd of the same loss composed from the map
    xa = x.detach().clone().requires_grad_(True)
    ((torch.sigmoid(xa) * phi).mean((2, 3)) * g_cost).sum().backward()
    scale = xa.grad.abs().max().item()
    assert (xr.grad - xa.grad).abs().max().item() <= 1e-6 * scale
    return cost, xr.grad


@pytest.mark.gpu
@pytest.mark.parametrize("spacing", [None, (3.87, 11.29), (1.0, 3.0), (1e-3, 1.0)], ids=str)
@pytest.mark.parametrize("density", [0.01, 0.5, 0.99])
def test_loss_equals_the_float64_reference(spacing, density):
    x, t = _batch(2, 3, 48, 64, seed=int(density * 100), density=density)
    _check_loss(x, t, spacing)


@pytest.mark.gpu
def test_loss_layer_masks_per_map_spacing_and_unit_spacing():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(2, 96, 128, seed=3, device="cuda")
    x = 4.0 * (pred - 0.5)
    _check_loss(x, truth)
    _check_loss(x, truth, np.random.default_rng(2).uniform(0.1, 10.0, tuple(x.shape[:2]) + (2,)))
    _check_loss(x, truth, (3.9e-3, 11.7e-3))
    unit = tlb.boundary_loss(x, truth)
    for sp in ((1, 1), 1.0):
        assert torch.equal(unit.view(torch.int32), tlb.boundary_loss(x, truth, spacing=sp).view(torch.int32))


@pytest.mark.gpu
def test_padded_targets_give_zero_and_nan_stays_in_its_map():
    x, t = _batch(2, 3, 40, 56, seed=8)
    t[0, 1] = 0.0                                               # an all-zero padded target
    t[1, 0] = 1.0                                               # all foreground
    x[1, 2, 7, 9] = float("nan")
    cost, grad = _check_loss_nan_tolerant(x, t)
    c = cost.detach().cpu()
    assert c[0, 1].item() == 0.0 and c[1, 0].item() == 0.0
    assert not grad[0, 1].any() and not grad[1, 0].any()
    assert math.isnan(c[1, 2].item())
    finite = torch.ones(2, 3, dtype=torch.bool)
    finite[1, 2] = False
    assert torch.isfinite(c[finite]).all()
    assert torch.isfinite(grad.cpu()[finite]).all()
    _check_loss(x.nan_to_num(0.0), t)                           # the same batch without the NaN is the reference


def _check_loss_nan_tolerant(x, t):
    import dilabhelmholtzoct_b200 as tlb
    xr = x.detach().clone().requires_grad_(True)
    cost = tlb.boundary_loss(xr, t)
    cost.sum().backward()
    return cost, xr.grad


@pytest.mark.gpu
def test_no_gradient_reaches_the_target_and_runs_are_bit_identical():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(4, 256, 256, seed=3, device="cuda")
    x = 4.0 * (pred - 0.5)
    for sp in (None, (3.87, 11.29)):
        outs = []
        for _ in range(2):
            xr = x.clone().requires_grad_(True)
            tr = truth.clone().requires_grad_(True)
            c = tlb.boundary_loss(xr, tr, spacing=sp)
            c.mean().backward()
            assert tr.grad is None
            outs.append((c.detach(), xr.grad, tlb.signed_distance_map(truth > 0.5, sampling=sp)))
        for a, b in zip(*outs):
            assert torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.gpu
def test_no_host_sync():
    import dilabhelmholtzoct_b200 as tlb
    x, t = _batch(2, 3, 64, 64, seed=4)
    m = t > 0.5
    per_map = np.full((2, 3, 2), 0.5)
    tlb.signed_distance_map(m, sampling=(1.0, 2.0))  # warm: library loaded, pinned pool primed
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for sp in (None, (3.0, 1.0), per_map, torch.from_numpy(per_map)):
            tlb.signed_distance_map(m, sampling=sp)
            xr = x.clone().requires_grad_(True)
            tlb.boundary_loss(xr, t, spacing=sp).sum().backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)


@pytest.mark.gpu
def test_views_inference_mode_and_empty_batch():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(2)
    u8 = torch.from_numpy(rng.integers(0, 4, (2, 3, 40, 70)).astype(np.uint8) * 85).cuda()
    nc = u8.transpose(2, 3)[..., ::2, 1:]
    assert not nc.is_contiguous()
    _check_map(nc)
    _check_map(nc, (3.87, 11.29))
    _check_map((u8[0, 0] > 100).expand(2, 2, 40, 70), (1.0, 3.0))
    assert _check_map(u8[0, 0]).shape == (40, 70)
    x, t = _batch(2, 3, 40, 70, seed=6)
    _check_loss(x.transpose(2, 3), t.transpose(2, 3), (3.87, 11.29))
    _check_loss(x[:, ::2], t[:, ::2].bool())                    # a bool target, cast to float32
    with torch.inference_mode():
        e = tlb.signed_distance_map(u8, sampling=(1.0, 3.0))
        c = tlb.boundary_loss(x, t)
    assert torch.equal(e, tlb.signed_distance_map(u8, sampling=(1.0, 3.0))) and not e.requires_grad
    assert torch.equal(c, tlb.boundary_loss(x, t))
    empty = torch.zeros(0, 5, 6, dtype=torch.bool, device="cuda")
    assert tlb.signed_distance_map(empty).shape == (0, 5, 6)
    xe = torch.zeros(0, 3, 5, 6, device="cuda", requires_grad=True)
    ce = tlb.boundary_loss(xe, torch.zeros(0, 3, 5, 6, device="cuda"))
    assert ce.shape == (0, 3)
    ce.sum().backward()
    assert xe.grad.shape == xe.shape


@pytest.mark.gpu
def test_bad_inputs_raise():
    import dilabhelmholtzoct_b200 as tlb
    m = torch.zeros(2, 3, 8, 8, dtype=torch.bool, device="cuda")
    x = torch.zeros(2, 3, 8, 8, device="cuda")
    for bad in (0.0, -1.0, math.nan, math.inf, 1e-7, 2e6, (1.0, math.nan), (1.0, 2.0, 3.0), np.ones((2, 2)), "1.0",
                True, torch.ones(2, device="cuda")):
        with pytest.raises(ValueError, match="spacing"):
            tlb.signed_distance_map(m, sampling=bad)
        with pytest.raises(ValueError, match="spacing"):
            tlb.boundary_loss(x, x, spacing=bad)
    with pytest.raises(ValueError):
        tlb.signed_distance_map(m.float())
    with pytest.raises(ValueError):
        tlb.boundary_loss(x.double(), x)
    with pytest.raises(ValueError):
        tlb.boundary_loss(x, x.to(torch.complex64))
    with pytest.raises(ValueError):
        tlb.signed_distance_map(torch.zeros(2, 4097, 1, dtype=torch.bool, device="cuda"))
