"""Physical pixel spacing for the distance family: ``distance_transform_edt(sampling=...)``,
``hausdorff_dt_loss(spacing=...)`` and ``surface_distances(spacing=...)`` (``tl_*_spaced``, DESIGN §3.10).

The contract: for a zero pixel at offset ``(dy, dx)`` the squared distance is the fp64 value
``a = float64(dy) * sy; b = float64(dx) * sx; s = a*a + b*b`` (each operation rounded, no FMA), and the distance is
``float32(sqrt(min s))``.  ``ref_edt_spaced`` is that minimum by brute force; the CPU tests pin it to scipy's sampled
transform bit for bit, and the GPU tests pin the ops to scipy (the transform and the metrics) and to a float64
restatement built on it (the loss).
"""
import ctypes
import math

import numpy as np
import pytest
import scipy.ndimage as ndi
import torch

from tests.test_surface_distance import ref_percentile, ref_surface

SPACINGS = [(0.5, 1.25), (2.0, 0.75), (3.0, 3.0), (3.87, 11.29), (0.1, 0.3), (1.0, 1000.0), (1e-3, 1.0), (0.7, 0.7)]
FIELDS = ("hausdorff", "hausdorff_percentile", "assd", "nsd")


# ---------------------------------------------------------------- float64 references

def ref_edt_spaced(m: np.ndarray, sy: float, sx: float) -> np.ndarray:
    """float32(sqrt(min over the zero pixels of s)), s evaluated as the contract states (numpy: no FMA)."""
    m = np.asarray(m, bool)
    H, W = m.shape
    zy, zx = np.nonzero(~m)
    uy, ux = np.indices((H, W))
    a = (zy[None, :] - uy.reshape(-1, 1)).astype(np.float64) * sy
    b = (zx[None, :] - ux.reshape(-1, 1)).astype(np.float64) * sx
    return np.sqrt((a * a + b * b).min(1)).astype(np.float32).reshape(H, W)


def ref_metrics_spaced(pred, target, q, tol, spacing):
    """(hausdorff, hausdorff_percentile, assd, nsd) of one map pair in float64, distances from scipy's sampled EDT."""
    Sp, St = ref_surface(pred), ref_surface(target)
    if not Sp.any() and not St.any():
        return (math.nan,) * 4
    if not Sp.any() or not St.any():
        return (math.inf, math.inf, math.inf, 0.0)
    d_pt = ndi.distance_transform_edt(~St, sampling=spacing)[Sp]
    d_tp = ndi.distance_transform_edt(~Sp, sampling=spacing)[St]
    n = len(d_pt) + len(d_tp)
    return (max(d_pt.max(), d_tp.max()), max(ref_percentile(d_pt, q), ref_percentile(d_tp, q)),
            (d_pt.sum() + d_tp.sum()) / n, (int((d_pt <= tol).sum()) + int((d_tp <= tol).sum())) / n)


def ref_field_spaced(M, spacing):
    M = np.asarray(M, bool)
    if M.all() or not M.any():
        return np.zeros(M.shape)
    return ndi.distance_transform_edt(M, sampling=spacing) + ndi.distance_transform_edt(~M, sampling=spacing)


def ref_loss_spaced(p, t, alpha, spacings):
    """Per-map cost and d cost / d x of the loss in float64; p the fp32 probabilities, spacings [n, 2]."""
    H, W = p.shape[-2:]
    p64, t64 = p.reshape(-1, H, W).astype(np.float64), t.reshape(-1, H, W).astype(np.float64)
    D = np.stack([ref_field_spaced(a > 0.5, sp) ** alpha + ref_field_spaced(b > 0.5, sp) ** alpha
                  for a, b, sp in zip(p.reshape(-1, H, W), t.reshape(-1, H, W), spacings)])
    cost = ((p64 - t64) ** 2 * D).mean(axis=(1, 2))
    grad = 2.0 / (H * W) * (p64 - t64) * D * p64 * (1.0 - p64)
    return cost, grad, D


# ---------------------------------------------------------------- CPU: the reference and hand-derived cases

def test_brute_force_reference_equals_scipy_bit_for_bit():
    rng = np.random.default_rng(0)
    for sp in SPACINGS:
        for _ in range(25):
            H, W = (int(v) for v in rng.integers(1, 40, 2))
            m = rng.random((H, W)) < rng.choice([0.5, 0.9, 0.99])
            if m.all():
                m[rng.integers(H), rng.integers(W)] = False
            want = ndi.distance_transform_edt(m, sampling=sp).astype(np.float32)
            assert np.array_equal(ref_edt_spaced(m, *sp).view(np.int32), want.view(np.int32)), (sp, H, W)


def test_kat_single_pixels_three_apart_along_a_row_and_along_a_column():
    # spacing (2, 0.5): 3 columns apart is 1.5, 3 rows apart is 6
    p, t = np.zeros((7, 7), bool), np.zeros((7, 7), bool)
    p[3, 1], t[3, 4] = True, True
    assert ref_metrics_spaced(p, t, 95.0, 1.5, (2.0, 0.5)) == (1.5, 1.5, 1.5, 1.0)
    assert ref_metrics_spaced(p.T, t.T, 95.0, 1.5, (2.0, 0.5)) == (6.0, 6.0, 6.0, 0.0)
    m = np.ones((7, 7), bool)
    m[3, 1] = False
    e = ref_edt_spaced(m, 2.0, 0.5)
    assert e[3, 4] == 1.5 and e[0, 1] == 6.0 and e[3, 1] == 0.0


def test_kat_shifted_square_at_an_anisotropic_spacing():
    # rings of 12, shifted by one column: six pixels of each ring are on the other ring, six are one column (sx) away
    p, t = np.zeros((10, 10), bool), np.zeros((10, 10), bool)
    p[2:6, 2:6] = True
    t[2:6, 3:7] = True
    assert ref_metrics_spaced(p, t, 95.0, 1.0, (3.0, 0.25)) == (0.25, 0.25, 0.125, 1.0)
    # shifted by one row instead: the four pixels of each ring's outer row are a row (3) away; the two pixels of the
    # row next to it that are not on the other ring are a column (0.25) from its side: assd = (12.5 + 12.5) / 24
    assert ref_metrics_spaced(p, np.roll(p, 1, 0), 95.0, 1.0, (3.0, 0.25))[::2] == (3.0, 25 / 24)


def test_kat_nsd_counts_distances_equal_to_the_tolerance():
    # one row: d_pt = [2, 1, 0, 0] and d_tp = [0, 0, 1, 2, 3] in columns; at sx = 0.5 they are halved
    p = np.array([[0, 1, 1, 1, 1, 0, 0, 0]], bool)
    t = np.array([[0, 0, 0, 1, 1, 1, 1, 1]], bool)
    assert ref_metrics_spaced(p, t, 100.0, 0.5, (7.0, 0.5))[3] == 6 / 9     # 0, 0, 0, 0 and 0.5, 0.5 are <= 0.5
    assert ref_metrics_spaced(p, t, 100.0, 0.4999, (7.0, 0.5))[3] == 4 / 9


# ---------------------------------------------------------------- CPU: the C ABI

def test_new_entry_points_are_declared_and_bound():
    import os
    import re
    from dilabhelmholtzoct_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(root, "include", "topoloss.h")).read(), flags=re.S)
    for name in ("tl_edt_spaced", "tl_hausdorff_dt_forward_spaced", "tl_surface_distances_spaced"):
        assert re.search(rf"\b{name}\s*\(", src) and name in _lib.SIGNATURES and hasattr(_lib.lib(), name)
    assert _lib.lib().tl_version() == _lib.ABI_VERSION == 4


BAD_SHAPES = ((0, 16, 16), (-1, 16, 16), (2, 0, 16), (2, 16, 0), (2, 4097, 16), (2, 16, 4097))


def _all_fail(fn, ok, cases):
    for i, bad in cases:
        a = list(ok)
        a[i] = bad
        assert fn(*a) == -1, (i, bad)


def test_new_entry_points_reject_bad_arguments():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    fake = 4096  # never dereferenced: every call below fails its host-side checks before any launch
    nw = 4 * 3 * 16 * 16
    ok = [fake, 3, 16, 16, fake, fake, nw, fake, None]
    _all_fail(L.tl_edt_spaced, ok, [(0, None), (4, None), (5, None), (7, None), (4, fake + 4), (5, fake + 2),
                                    (6, nw - 1)] + [(slice(1, 4), s) for s in BAD_SHAPES])

    ns, nc = 3 * 256 * 4, 3 * 256 * 8
    ok = [fake, fake, 3, 16, 16, 2.0, fake, fake, ns, fake, nc, fake, None]
    _all_fail(L.tl_hausdorff_dt_forward_spaced, ok,
              [(0, None), (1, None), (6, None), (7, None), (9, None), (11, None), (6, fake + 4), (7, fake + 2),
               (9, fake + 4), (5, 0.0), (5, -1.0), (5, math.inf), (5, math.nan), (8, ns - 1), (10, nc - 1)]
              + [(slice(2, 5), s) for s in BAD_SHAPES])

    nb = ctypes.c_size_t(0)
    assert L.tl_surface_workspace_bytes(3, 16, 16, ctypes.byref(nb)) == 0
    nw = nb.value
    ok = [fake, fake, 3, 16, 16, fake, 95.0, 1.0, fake, nw, fake, None]
    _all_fail(L.tl_surface_distances_spaced, ok,
              [(0, None), (1, None), (5, None), (8, None), (10, None), (5, fake + 4), (8, fake + 2), (9, nw - 1),
               (6, -1e-9), (6, 100.5), (6, math.nan), (7, -0.5), (7, math.inf), (7, math.nan)]
              + [(slice(2, 5), s) for s in BAD_SHAPES])


def test_python_checks_raise_value_errors_on_the_cpu():
    import dilabhelmholtzoct_b200 as tlb
    m = torch.zeros(2, 4, 4, dtype=torch.bool)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.distance_transform_edt(m, sampling=(1.0, 2.0))
    with pytest.raises(ValueError, match="CUDA"):
        tlb.surface_distances(m, m, spacing=(1.0, 2.0))


# ---------------------------------------------------------------- GPU: the transform

def _check_edt(m: torch.Tensor, sampling):
    import dilabhelmholtzoct_b200 as tlb
    got = tlb.distance_transform_edt(m, sampling=sampling)
    assert got.dtype == torch.float32 and got.shape == m.shape
    H, W = m.shape[-2:]
    maps = (m.cpu().numpy() != 0).reshape(-1, H, W)
    sp = np.broadcast_to(np.asarray(sampling, np.float64), m.shape[:-2] + (2,)).reshape(-1, 2)
    g = got.cpu().numpy().reshape(-1, H, W)
    for k, (mm, s) in enumerate(zip(maps, sp)):
        if mm.all():
            assert np.isposinf(g[k]).all()
            continue
        want = ndi.distance_transform_edt(mm, sampling=tuple(s)).astype(np.float32)
        assert np.array_equal(g[k].view(np.int32), want.view(np.int32)), (k, tuple(s), np.abs(g[k] - want).max())
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("spacing", SPACINGS + [(0.25, 4.0), (1e-6, 1e6)], ids=str)
@pytest.mark.parametrize("density", [0.5, 0.9, 0.995])
def test_edt_equals_scipy_on_random_masks(spacing, density):
    rng = np.random.default_rng(int(density * 1000) + int(spacing[0] * 97))
    for shape in ((37, 53), (61, 41)):
        _check_edt(torch.from_numpy(rng.random((4,) + shape) < density).cuda(), spacing)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 97), (89, 1), (1, 1), (31, 127), (496, 512), (1, 4096), (4096, 3)],
                         ids=lambda s: f"{s[0]}x{s[1]}")
def test_edt_shapes(shape):
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    m = rng.random((2,) + shape) < 0.97
    m[1] = rng.random(shape) < 0.5
    m[0].flat[rng.integers(m[0].size)] = False
    for sp in ((3.87, 11.29), (1.0, 1000.0), (1e-3, 1.0)):
        _check_edt(torch.from_numpy(m).cuda(), sp)


@pytest.mark.gpu
def test_edt_sparse_zero_sets_with_exact_ties():
    # few zero pixels on a grid: at spacing (1, 2) the offsets (2, 0) and (0, 1) have the same s, and dyadic spacings
    # make every s exact, so equal s from different offsets are everywhere
    rng = np.random.default_rng(11)
    m = np.ones((3, 160, 192), bool)
    for k in range(3):
        m[k, rng.integers(0, 160, 60), rng.integers(0, 192, 60)] = False
    m[2, ::6, ::4] = False
    for sp in ((1.0, 2.0), (0.5, 0.25), (2.0, 1.0), (3.87, 11.29), (0.1, 0.3)):
        _check_edt(torch.from_numpy(m).cuda(), sp)


@pytest.mark.gpu
def test_edt_per_map_spacing_scalar_and_no_zero_pixel():
    rng = np.random.default_rng(3)
    m = torch.from_numpy(rng.random((2, 3, 40, 50)) < 0.95).cuda()
    m[1, 2] = True                                              # no zero pixel: +inf
    per_map = rng.uniform(0.05, 20.0, (2, 3, 2))
    _check_edt(m, per_map)
    _check_edt(m, torch.from_numpy(per_map))                    # a CPU tensor
    _check_edt(m, per_map[:, :1])                               # broadcast over C
    _check_edt(m, 0.7)                                          # isotropic
    import dilabhelmholtzoct_b200 as tlb
    unit = tlb.distance_transform_edt(m)
    assert torch.equal(tlb.distance_transform_edt(m, sampling=(1, 1)).view(torch.int32), unit.view(torch.int32))
    assert torch.equal(tlb.distance_transform_edt(m, sampling=1.0).view(torch.int32), unit.view(torch.int32))


# ---------------------------------------------------------------- GPU: the metrics

def _check_surface(pred, target, q, tol, spacing):
    import dilabhelmholtzoct_b200 as tlb
    got = tlb.surface_distances(pred, target, q, tol, spacing=spacing)
    H, W = pred.shape[-2:]
    g = np.stack([x.cpu().numpy().reshape(-1) for x in got], 1)
    P, T = (m.cpu().numpy().reshape(-1, H, W) != 0 for m in (pred, target))
    sp = np.broadcast_to(np.asarray(spacing, np.float64), pred.shape[:-2] + (2,)).reshape(-1, 2)
    want = np.array([ref_metrics_spaced(p, t, q, tol, tuple(s)) for p, t, s in zip(P, T, sp)],
                    dtype=np.float64).reshape(-1, 4).astype(np.float32)
    for f in (0, 1, 3):
        assert np.array_equal(g[:, f], want[:, f], equal_nan=True), (FIELDS[f], q, tol, spacing, g[:, f], want[:, f])
    a, b = g[:, 2], want[:, 2]
    fin = np.isfinite(b)
    assert np.array_equal(a[~fin], b[~fin], equal_nan=True)
    ulps = np.abs(a[fin].view(np.int32).astype(np.int64) - b[fin].view(np.int32).astype(np.int64))
    assert ulps.size == 0 or ulps.max() <= 1, (a[fin], b[fin])
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("q", [0.0, 50.0, 95.0, 100.0])
@pytest.mark.parametrize("tol", [0.0, 1.0, 7.5])
def test_surface_equals_the_reference(q, tol):
    rng = np.random.default_rng(int(q * 10 + tol * 1000))
    for shape, density in (((37, 53), 0.1), ((96, 80), 0.6)):
        p = torch.from_numpy(rng.random((4,) + shape) < density).cuda()
        t = torch.from_numpy(rng.random((4,) + shape) < density).cuda()
        for sp in ((3.87, 11.29), (0.5, 1.25), (1.0, 1000.0), (1e-3, 1.0)):
            _check_surface(p, t, q, tol, sp)
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(1, 128, 160, seed=int(q) + 1, device="cuda")
    _check_surface(pred > 0.5, truth > 0.5, q, tol, (3.87, 11.29))


@pytest.mark.gpu
def test_surface_ties_at_the_selection_boundary():
    """Equal fp64 s from different offsets: at spacing (1, 2) the offsets (2, 0) and (0, 1) give s = 4, and lines and
    boxes give long runs of equal s, so both the "next key is equal" and the "next key is larger" paths are taken."""
    H, W = 64, 200
    p, t = np.zeros((4, H, W), bool), np.zeros((4, H, W), bool)
    p[0, 10, :] = True
    t[0, 12, : W // 3] = True                               # 2 rows away: s = 4
    t[0, 10, W // 3 + 1:: 3] = True                         # every third column of the same row: s = 0 or 4
    p[1, 20:40, 30:170] = True
    t[1, 22:42, 31:171] = True
    coarse = np.random.default_rng(3).random((2, H // 8, W // 8)) < 0.4
    p[2], t[2] = (np.kron(c, np.ones((8, 8), bool)) for c in coarse)
    p[3, 30, 100], t[3, 32, 100] = True, True
    t[3, 30, 101] = True
    pt, tt = torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda()
    for q in np.linspace(0.0, 100.0, 21):
        _check_surface(pt, tt, float(q), 2.0, (1.0, 2.0))
    for q in (33.0, 66.5, 97.3, 99.99):
        _check_surface(pt, tt, q, 2.0, (0.5, 0.25))


@pytest.mark.gpu
def test_surface_empty_masks_per_map_spacing_and_unit_spacing():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(5)
    p = rng.random((2, 3, 40, 56)) < 0.3
    t = rng.random((2, 3, 40, 56)) < 0.3
    p[0, 0] = t[0, 0] = False                               # both empty: NaN
    p[0, 1] = False                                         # one empty: inf, inf, inf, 0
    t[1, 2] = False
    pt, tt = torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda()
    got = _check_surface(pt, tt, 95.0, 3.0, rng.uniform(0.1, 10.0, (2, 3, 2)))
    assert all(math.isnan(float(x[0, 0])) for x in got)
    assert [float(x[0, 1]) for x in got] == [math.inf, math.inf, math.inf, 0.0]
    unit = tlb.surface_distances(pt, tt, 90.0, 1.5)
    for sp in ((1, 1), 1.0, np.ones((2, 3, 2))):
        for x, y in zip(unit, tlb.surface_distances(pt, tt, 90.0, 1.5, spacing=sp)):
            assert torch.equal(x.view(torch.int32), y.view(torch.int32))


@pytest.mark.gpu
def test_surface_hand_derived_cases():
    p, t = np.zeros((10, 10), bool), np.zeros((10, 10), bool)
    p[2:6, 2:6] = True
    t[2:6, 3:7] = True
    row_p = np.zeros((10, 10), bool)
    row_t = np.zeros((10, 10), bool)
    row_p[4, 1:5] = True
    row_t[4, 3:8] = True
    P = torch.from_numpy(np.stack([p, p, row_p])).cuda()
    T = torch.from_numpy(np.stack([t, np.roll(p, 1, 0), row_t])).cuda()
    got = _check_surface(P, T, 95.0, 0.5, (3.0, 0.25))
    assert [float(x[0]) for x in got] == [0.25, 0.25, 0.125, 1.0]
    assert float(got.hausdorff[1]) == 3.0 and float(got.assd[1]) == np.float32(25 / 24)
    got = _check_surface(P, T, 100.0, 0.5, (7.0, 0.5))     # the row pair: distances equal to the tolerance count
    assert float(got.nsd[2]) == np.float32(6 / 9)


# ---------------------------------------------------------------- GPU: the loss

def _random_batch(B, C, H, W, seed, scale=3.0):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    x = scale * torch.randn((B, C, H, W), generator=g, device="cuda")
    t = (torch.rand((B, C, H, W), generator=g, device="cuda") < 0.5).float()
    return x, t


def _check_loss(x, t, alpha, spacing):
    import dilabhelmholtzoct_b200 as tlb
    xr = x.clone().requires_grad_(True)
    cost = tlb.hausdorff_dt_loss(xr, t, alpha, spacing=spacing)
    g_cost = torch.linspace(0.5, 1.5, cost.numel(), device="cuda").reshape(cost.shape)
    (cost * g_cost).sum().backward()
    sp = np.broadcast_to(np.asarray(spacing, np.float64), x.shape[:2] + (2,)).reshape(-1, 2)
    p = torch.sigmoid(x).cpu().numpy()
    want, wgrad, _ = ref_loss_spaced(p, t.cpu().numpy(), alpha, sp)
    np.testing.assert_allclose(cost.detach().cpu().numpy().reshape(-1), want, rtol=1e-6, atol=0)
    wgrad = wgrad * g_cost.cpu().numpy().reshape(-1, 1, 1).astype(np.float64)
    np.testing.assert_allclose(xr.grad.cpu().numpy().reshape(wgrad.shape), wgrad, rtol=1e-5, atol=1e-30)
    return cost


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", [0.5, 1.0, 2.0, 3.0])
def test_loss_equals_the_float64_reference(alpha):
    x, t = _random_batch(2, 3, 48, 64, seed=int(alpha * 10))
    for sp in ((3.87, 11.29), (0.5, 1.25), (1e-3, 1.0)):
        _check_loss(x, t, alpha, sp)
    _check_loss(x, t, alpha, np.random.default_rng(1).uniform(0.1, 10.0, (2, 3, 2)))
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(1, 96, 128, seed=int(alpha * 10), device="cuda")
    _check_loss(4.0 * (pred - 0.5), truth, alpha, (3.9e-3, 11.7e-3))


@pytest.mark.gpu
def test_loss_single_label_maps_and_unit_spacing():
    import dilabhelmholtzoct_b200 as tlb
    x, t = _random_batch(2, 2, 32, 40, seed=9)
    x[0, 0] = 5.0                                          # prediction all foreground
    t[0, 1] = 0.0                                          # target all background
    x[1, 0], t[1, 0] = -5.0, 1.0                           # both single-label
    _check_loss(x, t, 2.0, (2.0, 0.75))
    unit = tlb.hausdorff_dt_loss(x, t, 1.5)
    for sp in ((1, 1), 1.0):
        assert torch.equal(unit.view(torch.int32), tlb.hausdorff_dt_loss(x, t, 1.5, spacing=sp).view(torch.int32))
    a, b = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    tlb.hausdorff_dt_loss(a, t).sum().backward()
    tlb.hausdorff_dt_loss(b, t, spacing=(1.0, 1.0)).sum().backward()
    assert torch.equal(a.grad.view(torch.int32), b.grad.view(torch.int32))


# ---------------------------------------------------------------- GPU: all three

@pytest.mark.gpu
def test_two_runs_are_bit_identical():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(4, 256, 256, seed=3, device="cuda")
    sp = (3.87, 11.29)
    for f in (lambda: [tlb.distance_transform_edt(pred > 0.5, sampling=sp)],
              lambda: list(tlb.surface_distances(pred > 0.5, truth > 0.5, spacing=sp)),
              lambda: [tlb.hausdorff_dt_loss(4.0 * (pred - 0.5), truth, spacing=sp)]):
        for a, b in zip(f(), f()):
            assert torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.gpu
def test_no_host_sync():
    import dilabhelmholtzoct_b200 as tlb
    x, t = _random_batch(2, 3, 64, 64, seed=4)
    m, mt = x > 0, t > 0.5
    per_map = np.full((2, 3, 2), 0.5)
    tlb.distance_transform_edt(m, sampling=(1.0, 2.0))  # warm: library loaded, pinned pool primed
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for sp in ((3.0, 1.0), per_map, torch.from_numpy(per_map)):
            tlb.distance_transform_edt(m, sampling=sp)
            tlb.surface_distances(m, mt, 90.0, 2.0, spacing=sp)
            xr = x.clone().requires_grad_(True)
            tlb.hausdorff_dt_loss(xr, t, spacing=sp).sum().backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)


@pytest.mark.gpu
def test_views_leading_dims_and_inference_mode():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(2)
    u8 = torch.from_numpy(rng.integers(0, 4, (2, 3, 40, 70)).astype(np.uint8) * 85).cuda()
    tb = torch.from_numpy(rng.random((2, 3, 40, 70)) < 0.5).cuda()
    sp = (3.87, 11.29)
    nc_p, nc_t = u8.transpose(2, 3)[..., ::2, 1:], tb.transpose(2, 3)[..., ::2, 1:]
    assert not nc_p.is_contiguous()
    _check_edt(nc_p, sp)
    _check_surface(nc_p, nc_t, 95.0, 20.0, sp)
    _check_edt((u8[0, 0] > 100).expand(2, 2, 40, 70), sp)
    one = _check_surface(u8[0, 0], tb[0, 0], 95.0, 20.0, sp)
    assert one.hausdorff.shape == ()
    x, t = _random_batch(2, 3, 40, 70, seed=6)
    _check_loss(x.transpose(2, 3), t.transpose(2, 3), 2.0, sp)
    with torch.inference_mode():
        e = tlb.distance_transform_edt(u8, sampling=sp)
        s = tlb.surface_distances(u8, tb, spacing=sp)
        c = tlb.hausdorff_dt_loss(x, t, spacing=sp)
    assert torch.equal(e, tlb.distance_transform_edt(u8, sampling=sp)) and not e.requires_grad
    for a, b in zip(s, tlb.surface_distances(u8, tb, spacing=sp)):
        assert torch.equal(a, b)
    assert torch.equal(c, tlb.hausdorff_dt_loss(x, t, spacing=sp))
    empty = torch.zeros(0, 5, 6, dtype=torch.bool, device="cuda")
    assert tlb.distance_transform_edt(empty, sampling=sp).shape == (0, 5, 6)
    assert tlb.surface_distances(empty, empty, spacing=sp).nsd.shape == (0,)


@pytest.mark.gpu
@pytest.mark.parametrize("bad", [0.0, -1.0, math.nan, math.inf, 1e-7, 2e6, (1.0, math.nan), (1.0, 0.0), (1.0, 2.0, 3.0),
                                 [1.0], np.ones((2, 2)), np.ones((2, 3, 3)), "1.0", ("a", "b"), True, None],
                         ids=lambda b: f"shape{b.shape}" if isinstance(b, np.ndarray) else repr(b))
def test_bad_spacing_raises_value_error(bad):
    import dilabhelmholtzoct_b200 as tlb
    m = torch.zeros(2, 3, 8, 8, dtype=torch.bool, device="cuda")
    x = torch.zeros(2, 3, 8, 8, device="cuda")
    if bad is None:  # a CUDA tensor: reading it would synchronise
        bad = torch.ones(2, device="cuda")
    with pytest.raises(ValueError, match="spacing"):
        tlb.distance_transform_edt(m, sampling=bad)
    with pytest.raises(ValueError, match="spacing"):
        tlb.surface_distances(m, m, spacing=bad)
    with pytest.raises(ValueError, match="spacing"):
        tlb.hausdorff_dt_loss(x, x, spacing=bad)
