"""Surface-distance metrics (``surface_distances``, ``tl_surface_distances``): Hausdorff distance, percentile Hausdorff
distance, ASSD and normalized surface Dice of binary mask pairs.

The op is pinned against a float64 numpy / scipy restatement of its definition (``ref_metrics``): surfaces from
``scipy.ndimage.binary_erosion``, distances from ``scipy.ndimage.distance_transform_edt``, the percentile restated from
numpy's linear method (``ref_percentile``, itself pinned bit for bit to ``np.percentile``).  The CPU tests check the
reference on hand-derived cases.
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
NEW = ["tl_surface_workspace_bytes", "tl_surface_distances"]
FIELDS = ("hausdorff", "hausdorff_percentile", "assd", "nsd")


# ---------------------------------------------------------------- float64 reference

def ref_surface(M: np.ndarray) -> np.ndarray:
    """S(M) = M & ~binary_erosion(M): cross structure, outside the image counts as background."""
    M = np.asarray(M, dtype=bool)
    return M & ~ndi.binary_erosion(M, border_value=0)


def ref_percentile(d, q: float) -> float:
    """np.percentile(d, q) (method "linear"), restated step by step in float64 without fused operations."""
    d = np.sort(np.asarray(d, dtype=np.float64))
    n = len(d)
    h = (n - 1) * (q / 100.0)
    if h >= n - 1:
        return float(d[n - 1])
    lo = math.floor(h)
    g = h - lo
    a, b = float(d[lo]), float(d[lo + 1])
    diff = b - a
    return b - diff * (1 - g) if g >= 0.5 else a + diff * g


def ref_metrics(pred: np.ndarray, target: np.ndarray, q: float = 95.0, tol: float = 1.0):
    """(hausdorff, hausdorff_percentile, assd, nsd) of one [H, W] map pair, float64."""
    Sp, St = ref_surface(pred), ref_surface(target)
    if not Sp.any() and not St.any():
        return (math.nan,) * 4
    if not Sp.any() or not St.any():
        return (math.inf, math.inf, math.inf, 0.0)
    d_pt = ndi.distance_transform_edt(~St)[Sp]
    d_tp = ndi.distance_transform_edt(~Sp)[St]
    n = len(d_pt) + len(d_tp)
    return (max(d_pt.max(), d_tp.max()), max(ref_percentile(d_pt, q), ref_percentile(d_tp, q)),
            (d_pt.sum() + d_tp.sum()) / n, (int((d_pt <= tol).sum()) + int((d_tp <= tol).sum())) / n)


# ---------------------------------------------------------------- CPU: the reference

def test_ref_percentile_equals_numpy_bit_for_bit():
    rng = np.random.default_rng(0)
    qs = [0.0, 100.0, 50.0, 95.0, 99.0, 1.0, 25.0, 75.0, 5.0, 99.9]
    for trial in range(3000):
        n = int(rng.integers(1, 60)) if trial % 3 else int(rng.integers(1, 3000))
        d = np.sqrt(rng.integers(0, 1 << int(rng.integers(1, 25)), n).astype(np.float64))
        for q in qs + list(rng.random(2) * 100.0):
            want = np.percentile(d, q)
            got = ref_percentile(d, q)
            assert np.float64(got).view(np.int64) == np.float64(want).view(np.int64), (n, q, got, want)


def test_surface_rule_is_the_four_neighbour_rule():
    """The kernel's rule: a foreground pixel is on the surface iff a 4-neighbour is background or outside."""
    rng = np.random.default_rng(1)
    for trial in range(200):
        H, W = (int(v) for v in rng.integers(1, 24, 2))
        M = rng.random((H, W)) < rng.choice([0.05, 0.5, 0.9, 1.0])
        P = np.pad(M, 1)
        interior = P[:-2, 1:-1] & P[2:, 1:-1] & P[1:-1, :-2] & P[1:-1, 2:]
        assert np.array_equal(ref_surface(M), M & ~interior), (H, W)


def _pixel(H, W, r, c):
    m = np.zeros((H, W), bool)
    m[r, c] = True
    return m


def test_kat_two_single_pixels_three_apart():
    p, t = _pixel(5, 7, 2, 1), _pixel(5, 7, 2, 4)
    assert ref_metrics(p, t, 95.0, 1.0) == (3.0, 3.0, 3.0, 0.0)
    assert ref_metrics(p, t, 50.0, 3.0)[3] == 1.0
    assert ref_metrics(p, t, 0.0, 2.5)[3] == 0.0


def test_kat_square_against_the_square_shifted_by_one():
    # rings of 12: six pixels of each ring lie on the other ring, six are 1 away
    p = np.zeros((10, 10), bool)
    t = np.zeros((10, 10), bool)
    p[2:6, 2:6] = True
    t[2:6, 3:7] = True
    assert ref_metrics(p, t, 95.0, 1.0) == (1.0, 1.0, 0.5, 1.0)
    assert ref_metrics(p, t, 50.0, 0.0) == (1.0, 0.5, 0.5, 0.5)  # h = 5.5: halfway between d[5] = 0 and d[6] = 1
    assert ref_metrics(p, t, 0.0, 0.5)[1:] == (0.0, 0.5, 0.5)


def test_kat_full_map_has_the_image_border_as_its_surface():
    full = np.ones((5, 5), bool)
    border = np.ones((5, 5), bool)
    border[1:-1, 1:-1] = False
    assert np.array_equal(ref_surface(full), border)
    assert ref_metrics(full, full) == (0.0, 0.0, 0.0, 1.0)
    # against the centre pixel: corners sqrt(8), edge midpoints 2, the other 8 border pixels sqrt(5); centre -> 2
    hd, _, assd, nsd = ref_metrics(full, _pixel(5, 5, 2, 2), 100.0, 2.0)
    assert hd == math.sqrt(8.0)
    assert assd == pytest.approx((4 * math.sqrt(8.0) + 4 * 2.0 + 8 * math.sqrt(5.0) + 2.0) / 17, rel=1e-15)
    assert nsd == 5 / 17


def test_kat_one_row_and_one_column_maps():
    # one row: every foreground pixel is on the surface
    p = np.array([[0, 1, 1, 1, 1, 0, 0, 0]], bool)
    t = np.array([[0, 0, 0, 1, 1, 1, 1, 1]], bool)
    # d_pt = [2, 1, 0, 0], d_tp = [0, 0, 1, 2, 3]
    want = (3.0, 3.0, 1.0, 6 / 9)
    assert ref_metrics(p, t, 100.0, 1.0) == want
    assert ref_metrics(p.T, t.T, 100.0, 1.0) == want
    assert ref_metrics(p, t, 50.0, 1.0)[1] == 1.0  # pct(d_pt) = 0.5, pct(d_tp) = 1


def test_kat_one_empty_and_both_empty_maps():
    e = np.zeros((4, 6), bool)
    assert ref_metrics(e, _pixel(4, 6, 1, 1)) == (math.inf, math.inf, math.inf, 0.0)
    assert ref_metrics(_pixel(4, 6, 1, 1), e) == (math.inf, math.inf, math.inf, 0.0)
    assert all(math.isnan(v) for v in ref_metrics(e, e))


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
    for name in ("surface_distances", "SurfaceDistances"):
        assert name in tlb.__all__ and callable(getattr(tlb, name))
    assert tlb.SurfaceDistances._fields == FIELDS


BAD_SHAPES = ((0, 16, 16), (-1, 16, 16), (2, 0, 16), (2, 16, 0), (2, 4097, 16), (2, 16, 4097))


def test_workspace_query_and_bad_arguments():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    nb = ctypes.c_size_t(0)
    assert L.tl_surface_workspace_bytes(3, 16, 16, None) == -1
    for bad in BAD_SHAPES:
        assert L.tl_surface_workspace_bytes(*bad, ctypes.byref(nb)) == -1, bad
    assert L.tl_surface_workspace_bytes(3, 16, 16, ctypes.byref(nb)) == 0
    nw = nb.value
    assert nw >= 16 * 3 * 256 + 16 * 3
    fake = 4096  # never dereferenced: every call below fails its host-side checks before any launch
    # tl_surface_distances(pred, target, n, H, W, spacing, percentile, tolerance, ws, ws_bytes, out, stream); every
    # case fails with a null (unit) or a device spacing
    cases = [(0, None), (1, None), (8, None), (10, None), (5, fake + 4), (8, fake + 2), (9, nw - 1),
             (6, -1e-9), (6, 100.5), (6, math.nan), (6, math.inf), (6, -math.inf),
             (7, -0.5), (7, math.inf), (7, math.nan)]
    cases += [(slice(2, 5), s) for s in BAD_SHAPES]
    for sp in (None, fake):
        ok = [fake, fake, 3, 16, 16, sp, 95.0, 1.0, fake, nw, fake, None]
        for i, bad in cases:
            a = list(ok)
            a[i] = bad
            assert L.tl_surface_distances(*a) == -1, (sp, i, bad)
        assert L.tl_surface_distances(*(ok[:9] + [nw - 1] + ok[10:])) == -1
        assert b"tl_surface_workspace_bytes" in L.tl_last_error()
        a = list(ok)
        a[6] = 101.0
        assert L.tl_surface_distances(*a) == -1 and b"percentile" in L.tl_last_error()
        a = list(ok)
        a[7] = -1.0
        assert L.tl_surface_distances(*a) == -1 and b"tolerance" in L.tl_last_error()


def test_python_checks_raise_value_errors_on_the_cpu():
    import dilabhelmholtzoct_b200 as tlb
    m = torch.zeros(2, 4, 4, dtype=torch.bool)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.surface_distances(m, m)
    with pytest.raises(ValueError, match="same shape"):
        tlb.surface_distances(m, m[:, :, :3])
    with pytest.raises(ValueError, match="same shape"):
        tlb.surface_distances(m[0, 0], m[0, 0])
    with pytest.raises(TypeError):
        tlb.surface_distances(np.zeros((4, 4), bool), m[0])


# ---------------------------------------------------------------- GPU: the op against the reference

def _check(pred, target, q=95.0, tol=1.0):
    """surface_distances(pred, target) equals ref_metrics per map: hausdorff, hausdorff_percentile and nsd bit for bit
    after rounding to float32, assd within one float32 ulp."""
    import dilabhelmholtzoct_b200 as tlb
    got = tlb.surface_distances(pred, target, q, tol)
    assert isinstance(got, tlb.SurfaceDistances)
    H, W = pred.shape[-2:]
    for g in got:
        assert g.dtype == torch.float32 and g.shape == pred.shape[:-2] and g.device == pred.device
    g = np.stack([x.cpu().numpy().reshape(-1) for x in got], 1)
    P, T = (m.cpu().numpy().reshape(-1, H, W) != 0 for m in (pred, target))
    want = np.array([ref_metrics(p, t, q, tol) for p, t in zip(P, T)], dtype=np.float64).reshape(-1, 4).astype(np.float32)
    for f in (0, 1, 3):
        assert np.array_equal(g[:, f], want[:, f], equal_nan=True), (FIELDS[f], g[:, f], want[:, f])
    a, b = g[:, 2], want[:, 2]
    assert np.array_equal(np.isfinite(a), np.isfinite(b)) and np.array_equal(a[~np.isfinite(a)], b[~np.isfinite(b)],
                                                                            equal_nan=True)
    fin = np.isfinite(b)
    ulps = np.abs(a[fin].view(np.int32).astype(np.int64) - b[fin].view(np.int32).astype(np.int64))
    assert ulps.size == 0 or ulps.max() <= 1, (a[fin], b[fin])
    return got


SHAPES = [(1, 1), (1, 4096), (4096, 1), (37, 53), (496, 512), (1024, 1024)]


@pytest.mark.gpu
@pytest.mark.parametrize("density", [0.01, 0.5, 0.99])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_equals_the_reference_on_random_masks(shape, density):
    rng = np.random.default_rng(hash((shape, density)) % 2 ** 32)
    n = 1 if shape[0] * shape[1] >= 496 * 512 else 6
    p = torch.from_numpy(rng.random((n,) + shape) < density).cuda()
    t = torch.from_numpy(rng.random((n,) + shape) < density).cuda()
    _check(p, t)


@pytest.mark.gpu
@pytest.mark.parametrize("q", [0.0, 50.0, 95.0, 100.0])
@pytest.mark.parametrize("tol", [0.0, 1.0, 2.5])
def test_percentiles_and_tolerances(q, tol):
    rng = np.random.default_rng(int(q * 10 + tol * 1000))
    for shape, density in (((37, 53), 0.1), ((96, 80), 0.6)):
        p = torch.from_numpy(rng.random((4,) + shape) < density).cuda()
        t = torch.from_numpy(rng.random((4,) + shape) < density).cuda()
        _check(p, t, q, tol)
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(1, 128, 160, seed=int(q) + 1, device="cuda")
    _check(pred > 0.5, truth > 0.5, q, tol)


@pytest.mark.gpu
def test_equals_the_reference_on_synthetic_layer_masks():
    from dilabhelmholtzoct_b200.synthetic import make_batch
    for B, H, W in ((2, 256, 256), (1, 496, 512)):
        pred, truth = make_batch(B, H, W, seed=H, device="cuda")
        _check(pred > 0.5, truth > 0.5)
        _check(pred > 0.5, truth > 0.5, 50.0, 2.5)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 1), (3, 3), (37, 53), (256, 256), (4096, 1)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_single_pixel_full_one_empty_and_both_empty_maps(shape):
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(5)
    H, W = shape
    p = np.zeros((7, H, W), bool)
    t = np.zeros((7, H, W), bool)
    for k in range(2):                                     # single pixels
        p[k, rng.integers(H), rng.integers(W)] = True
        t[k, rng.integers(H), rng.integers(W)] = True
    p[2] = t[2] = True                                     # full against full
    p[3] = True                                            # full against a pixel
    t[3, rng.integers(H), rng.integers(W)] = True
    p[4, rng.integers(H), rng.integers(W)] = True          # target empty
    t[5] = True                                            # prediction empty; map 6 both empty
    got = _check(torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda())
    hd, hp, assd, nsd = (x.cpu() for x in got)
    assert hd[2] == 0 and assd[2] == 0 and nsd[2] == 1
    for k in (4, 5):
        assert math.isinf(hd[k]) and math.isinf(hp[k]) and math.isinf(assd[k]) and nsd[k] == 0
    assert all(math.isnan(x[6]) for x in (hd, hp, assd, nsd))
    assert isinstance(tlb.SurfaceDistances(*got), tuple)


@pytest.mark.gpu
def test_hausdorff_equals_the_100th_percentile():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(8)
    p = torch.from_numpy(rng.random((8, 64, 96)) < 0.2).cuda()
    t = torch.from_numpy(rng.random((8, 64, 96)) < 0.2).cuda()
    got = tlb.surface_distances(p, t, 100.0)
    assert torch.equal(got.hausdorff, got.hausdorff_percentile)


@pytest.mark.gpu
def test_percentile_ties_at_the_selection_boundary():
    """Few distinct distances in long runs: across a sweep of q the selected rank lands inside runs and at their ends,
    so both the "next key is equal" and the "next key is larger" paths are taken."""
    H, W = 64, 200
    p = np.zeros((3, H, W), bool)
    t = np.zeros((3, H, W), bool)
    p[0, 10, :] = True                                     # a line against lines 2 and 5 rows away: runs of 2 and 5
    t[0, 12, : W // 3] = True
    t[0, 15, W // 3:] = True
    p[1, 20:40, 30:170] = True                             # a box against itself shifted: runs of 0, 1, 2
    t[1, 22:42, 31:171] = True
    coarse = np.random.default_rng(3).random((2, H // 8, W // 8)) < 0.4
    p[2], t[2] = (np.kron(c, np.ones((8, 8), bool)) for c in coarse)  # blocky masks: many equal s
    pt, tt = torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda()
    for q in np.linspace(0.0, 100.0, 41):
        _check(pt, tt, float(q), 1.0)
    for q in (33.0, 66.5, 97.3, 99.99):
        _check(pt, tt, q, 2.0)


@pytest.mark.gpu
def test_two_runs_are_bit_identical():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(8, 256, 256, seed=3, device="cuda")
    P, T = pred > 0.5, truth > 0.5
    a, b = tlb.surface_distances(P, T), tlb.surface_distances(P, T)
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))


@pytest.mark.gpu
def test_no_host_sync():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(4)
    p = torch.from_numpy(rng.random((2, 3, 64, 64)) < 0.3).cuda()
    t = torch.from_numpy(rng.random((2, 3, 64, 64)) < 0.3).cuda()
    tlb.surface_distances(p, t)  # warm: library loaded
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = tlb.surface_distances(p, t, 90.0, 2.0)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert got.hausdorff.shape == (2, 3)


@pytest.mark.gpu
def test_bool_uint8_non_contiguous_leading_dims_and_inference_mode():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(2)
    vals = rng.integers(0, 4, (2, 3, 40, 70)).astype(np.uint8) * 85  # 0, 85, 170, 255: nonzero is foreground
    u8 = torch.from_numpy(vals).cuda()
    tb = torch.from_numpy(rng.random((2, 3, 40, 70)) < 0.5).cuda()
    ref = _check(u8, tb, 90.0, 1.5)
    for x, y in zip(ref, tlb.surface_distances(u8 != 0, tb.to(torch.uint8), 90.0, 1.5)):
        assert torch.equal(x, y)
    nc_p, nc_t = u8.transpose(2, 3)[..., ::2, 1:], tb.transpose(2, 3)[..., ::2, 1:]  # non-contiguous views
    assert not nc_p.is_contiguous()
    _check(nc_p, nc_t)
    _check((u8[0, 0] > 100).expand(2, 2, 40, 70), tb[0, 1].expand(2, 2, 40, 70))  # extra leading dims, stride 0
    one = _check(u8[0, 0], tb[0, 0])                                                 # a single [H, W] map
    assert one.hausdorff.shape == ()
    with torch.inference_mode():
        inf = tlb.surface_distances(u8, tb, 90.0, 1.5)
    for x, y in zip(ref, inf):
        assert torch.equal(x, y) and not y.requires_grad
    empty = tlb.surface_distances(torch.zeros(0, 5, 6, dtype=torch.bool, device="cuda"),
                                  torch.zeros(0, 5, 6, dtype=torch.bool, device="cuda"))
    assert all(x.shape == (0,) and x.dtype == torch.float32 for x in empty)


@pytest.mark.gpu
def test_python_checks_on_the_gpu():
    import dilabhelmholtzoct_b200 as tlb
    m = torch.zeros(2, 8, 8, dtype=torch.bool, device="cuda")
    with pytest.raises(ValueError, match="bool or uint8"):
        tlb.surface_distances(m.float(), m)
    with pytest.raises(ValueError, match="bool or uint8"):
        tlb.surface_distances(m, m.to(torch.int32))
    with pytest.raises(ValueError, match="same shape"):
        tlb.surface_distances(m, m[:1])
    with pytest.raises(ValueError, match="CUDA"):
        tlb.surface_distances(m, m.cpu())
    for q in (-1.0, 100.01, math.nan, math.inf):
        with pytest.raises(ValueError, match="percentile"):
            tlb.surface_distances(m, m, q)
    for tol in (-0.5, math.inf, math.nan):
        with pytest.raises(ValueError, match="tolerance"):
            tlb.surface_distances(m, m, 95.0, tol)
    big = torch.zeros(1, 4097, 2, dtype=torch.bool, device="cuda")
    with pytest.raises(ValueError, match="4096"):
        tlb.surface_distances(big, big)
