"""Betti matching (``dilabhelmholtzoct_b200.betti``): image persistence, induced matching and its gradient.

CPU: the literal image-persistence oracle (``tests/betti_oracle.py::image_pairs_literal``) is the ordinary barcode for
the identity image and has the rank of ``H_d(L_t) -> H_d(C_t)`` at every threshold, counted with
``scipy.ndimage.label``; the union-find restatement (``betti_oracle.betti_matching``) equals the literal matching, cells
and order included; matching properties; hand-derived KATs that the Wasserstein cost cannot see; the C entry points
are declared, bound and reject bad arguments; CPU tensors raise.
GPU: the kernel's barcodes equal ``cubical_persistence``; records, order and cost equal the oracle; the gradients
equal torch autograd of the cost formula; NaN, empty and constant maps; determinism; no host sync in the backward.
"""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import oracle
from oracle.oracle_literal import _cells, cubical_pairs_literal
from tests import betti_oracle
from tests.betti_oracle import betti_matching_literal, image_pairs_literal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["tl_betti_workspace_bytes", "tl_betti_compute", "tl_betti_gather", "tl_betti_backward"]
KEYS = ("matched", "unmatched_pred", "unmatched_target")


def _np_map(rng, kind, H, W):
    if kind == "random":
        return rng.random((H, W)).astype(np.float32)
    if kind.startswith("levels"):
        k = int(kind[6:])
        return (np.floor(rng.random((H, W)) * k) / k).astype(np.float32)
    if kind == "const":
        return np.full((H, W), 0.5, np.float32)
    if kind == "mask":
        return (rng.random((H, W)) < 0.4).astype(np.float32)
    raise ValueError(kind)


SMALL = [(kind, seed) for seed in range(6) for kind in ("random", "levels2", "levels4", "levels32", "mask")]


def _pair(kind, seed, H=None, W=None):
    rng = np.random.default_rng(1000 + seed)
    H = H or int(rng.integers(1, 15))
    W = W or int(rng.integers(1, 15))
    return _np_map(rng, kind, H, W), _np_map(rng, "levels4" if kind == "mask" else kind, H, W)


# ---------------------------------------------------------------- CPU: the oracles

@pytest.mark.parametrize("kind,seed", SMALL + [("const", 0)])
def test_identity_image_is_the_barcode(kind, seed):
    f, _ = _pair(kind, seed)
    h0, h1, ess = cubical_pairs_literal(f)
    p0, e0 = image_pairs_literal(f, f, 0)
    p1, e1 = image_pairs_literal(f, f, 1)
    assert [(r[2], r[3]) for r in p0] == h0 and [(r[2], r[3]) for r in p1] == h1
    assert e0[1] == ess[0] and e1 is None


@pytest.mark.parametrize("kind,seed", SMALL)
def test_image_rank_equals_connected_component_counts(kind, seed):
    """For every t: #image intervals alive = rank of H_d(L_t) -> H_d(C_t), from scipy's labelling (the conventions
    of test_oracle.test_betti_curves_match_connected_component_counts: closed pixels, 8-connected components,
    4-connected complement)."""
    from scipy import ndimage
    L, G = _pair(kind, seed)
    C = np.minimum(L, G)
    vL, vC = _cells(L)[0].ravel(), _cells(C)[0].ravel()
    eight, four = np.ones((3, 3), int), ndimage.generate_binary_structure(2, 1)
    p0, _ = image_pairs_literal(L, C, 0)
    p1, _ = image_pairs_literal(L, C, 1)
    for t in np.unique(np.concatenate([L.ravel(), C.ravel()])):
        n0 = sum(1 for s, d, _, _ in p0 if vL[s] <= t < vC[d]) + int(L.min() <= t)
        lab, _ = ndimage.label(C <= t, structure=eight)
        assert n0 == len(set(np.unique(lab[L <= t])) - {0}), t
        n1 = sum(1 for s, d, _, _ in p1 if vL[s] <= t < vC[d])
        lab, _ = ndimage.label(np.pad(L > t, 1, constant_values=True), structure=four)
        assert n1 == len(set(np.unique(lab[np.pad(C > t, 1, constant_values=True)])) - {0}) - 1, t


def _same(a, b, rtol=1e-12):
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k
    assert abs(a["cost"] - b["cost"]) <= rtol * max(1.0, abs(a["cost"]))


@pytest.mark.parametrize("dim", [0, 1])
@pytest.mark.parametrize("kind,seed", SMALL + [("const", 0)])
def test_union_find_equals_the_literal_oracle(kind, seed, dim):
    L, G = _pair(kind, seed)
    _same(betti_oracle.betti_matching(L, G, dim), betti_matching_literal(L, G, dim))


def _check_properties(L, G, dim):
    r = betti_oracle.betti_matching(L, G, dim)
    s = betti_oracle.betti_matching(G, L, dim)
    # symmetric: same cost, matched columns swapped (the rows follow the other map's nodes, so compare as sets)
    assert abs(r["cost"] - s["cost"]) <= 1e-12 * max(1.0, r["cost"])
    assert sorted(map(tuple, r["matched"][:, [2, 3, 0, 1]])) == sorted(map(tuple, s["matched"]))
    assert sorted(map(tuple, r["unmatched_pred"])) == sorted(map(tuple, s["unmatched_target"]))
    # every interval once, in matched or unmatched
    for m, cols, un in ((L, [0, 1], "unmatched_pred"), (G, [2, 3], "unmatched_target")):
        bars = sorted(map(tuple, oracle.cubical_pairs(m, dim)))
        got = sorted(map(tuple, r["matched"][:, cols])) + sorted(map(tuple, r[un]))
        assert sorted(got) == bars
    # a map against itself: everything matched, cost 0
    same = betti_oracle.betti_matching(L, L, dim)
    assert same["cost"] == 0 and len(same["unmatched_pred"]) == 0 and len(same["unmatched_target"]) == 0
    assert np.array_equal(same["matched"][:, :2], same["matched"][:, 2:])
    return r


@pytest.mark.parametrize("dim", [0, 1])
@pytest.mark.parametrize("kind,seed", SMALL[:15])
def test_matching_properties(kind, seed, dim):
    _check_properties(*_pair(kind, seed), dim)


@pytest.mark.parametrize("dim", [0, 1])
def test_union_find_on_headline_maps(dim):
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(1, 256, 256, seed=3, n_classes=14)
    rng = np.random.default_rng(5)
    noise = rng.random((256, 256)).astype(np.float32)
    for c in (0, 5):
        r = _check_properties(pred[0, c].numpy(), truth[0, c].numpy(), dim)
        assert r["cost"] > 0
    _check_properties(noise, pred[0, 2].numpy(), dim)


def _blobs(spec, H=12, W=18, bg=0.0):
    x = np.full((H, W), bg, np.float32)
    for (r, c), v in spec:
        x[r:r + 2, c:c + 2] = v
    return x


def test_kat_h0_blobs_superlevel():
    """Blobs at A (0.9) and B (0.8) in the target, at A (0.9) and C (0.8) in the prediction.  Superlevel, i.e. the
    sublevel filtration of the negated maps: both diagrams are {(-0.9, 0) essential, (-0.8, 0)}, so the Wasserstein
    cost is 0.  In min(-L, -G) the blobs at B and C are separate components, so the two (-0.8, 0) intervals are
    unmatched: cost = 2 * (0 - (-0.8))^2 / 2 = 0.8^2; the essential classes match at zero cost."""
    A, B, C = (2, 2), (2, 12), (8, 8)
    G = _blobs([(A, 0.9), (B, 0.8)])
    L = _blobs([(A, 0.9), (C, 0.8)])
    dl, dg = oracle.cubical_pairs(-L, 0), oracle.cubical_pairs(-G, 0)
    vals = lambda m, p: sorted((float(m.ravel()[a]), float(m.ravel()[b])) for a, b in p)
    assert vals(-L, dl) == vals(-G, dg)
    assert oracle.wasserstein((-L).ravel()[dl], (-G).ravel()[dg], 2.0)[0] == 0.0
    want = float(np.float32(0.8)) ** 2
    for r in (betti_oracle.betti_matching(-L, -G, 0), betti_matching_literal(-L, -G, 0)):
        assert len(r["matched"]) == 1 and len(r["unmatched_pred"]) == 1 and len(r["unmatched_target"]) == 1
        assert r["unmatched_pred"][0][0] // 18 == C[0] and r["unmatched_target"][0][0] // 18 == B[0]
        assert abs(r["cost"] - want) <= 1e-12


def _rings(spec, H=15, W=21):
    """Low-valued 3x3 rings around one high pixel, on a high background (sublevel: one hole each)."""
    x = np.ones((H, W), np.float32)
    for (r, c), v in spec:
        x[r:r + 3, c:c + 3] = v
        x[r + 1, c + 1] = 1.0
    return x


def test_kat_h1_rings():
    """Rings at A (0.1) and B (0.2) in the target, at A (0.1) and C (0.2) in the prediction: both H1 diagrams are
    {(0.1, 1), (0.2, 1)} (Wasserstein cost 0); the holes at B and C die at different squares of min(L, G), so the
    cost is 2 * (1 - 0.2)^2 / 2 = 0.8^2 (in float32 values)."""
    A, B, C = (1, 1), (1, 15), (10, 8)
    G = _rings([(A, 0.1), (B, 0.2)])
    L = _rings([(A, 0.1), (C, 0.2)])
    dl, dg = oracle.cubical_pairs(L, 1), oracle.cubical_pairs(G, 1)
    assert sorted(map(tuple, L.ravel()[dl].tolist())) == sorted(map(tuple, G.ravel()[dg].tolist()))
    assert oracle.wasserstein(L.ravel()[dl], G.ravel()[dg], 2.0)[0] == 0.0
    want = (1.0 - float(np.float32(0.2))) ** 2
    for r in (betti_oracle.betti_matching(L, G, 1), betti_matching_literal(L, G, 1)):
        m = r["matched"]
        assert len(m) == 1 and m[0][0] == m[0][2] and m[0][1] == m[0][3] == (A[0] + 1) * 21 + A[1] + 1
        assert r["unmatched_pred"][0][1] == (C[0] + 1) * 21 + C[1] + 1
        assert r["unmatched_target"][0][1] == (B[0] + 1) * 21 + B[1] + 1
        assert abs(r["cost"] - want) <= 1e-12


# ---------------------------------------------------------------- CPU: the C ABI and the Python checks

def test_new_entry_points_are_declared_exported_and_bound():
    from dilabhelmholtzoct_b200 import _lib, build
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "topoloss.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(tl_[a-z_0-9]+)\s*\(", src))
    if not os.path.exists(build.LIB_PATH):
        build.build()
    L = ctypes.CDLL(build.LIB_PATH)
    for name in NEW:
        assert name in declared and hasattr(L, name) and name in _lib.SIGNATURES, name
    assert _lib.lib().tl_version() == _lib.ABI_VERSION == 4


def test_new_entry_points_reject_bad_arguments():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    nb = ctypes.c_size_t(0)
    assert L.tl_betti_workspace_bytes(3, 16, 16, 1, None) == -1
    assert L.tl_betti_workspace_bytes(3, 16, 16, 2, ctypes.byref(nb)) == -1
    assert L.tl_betti_workspace_bytes(0, 16, 16, 1, ctypes.byref(nb)) == -1
    assert L.tl_betti_workspace_bytes(3, 16, 0, 1, ctypes.byref(nb)) == -1
    assert L.tl_betti_workspace_bytes(3, 16, 16, 1, ctypes.byref(nb)) == 0 and nb.value > 0
    need = nb.value
    fake = 4096  # never dereferenced: every call below fails its host-side checks first
    ok = [fake, fake, 3, 16, 16, 1, fake, need, fake, fake, None, None]
    for i, bad in ((0, None), (1, None), (6, None), (8, None), (9, None), (5, 2), (2, 0), (7, need - 1)):
        a = list(ok)
        a[i] = bad
        assert L.tl_betti_compute(*a) == -1, i
    host = (ctypes.c_int32 * 12)(0, 1, 2, 3, 0, 0, 1, 1, 0, 2, 2, 2)
    g = [3, 16, 16, 1, fake, need, fake, host, 3, 1, 2, fake, fake, fake, None]
    # g is valid as it stands (it would launch): only altered copies are passed
    for i, bad in ((4, None), (6, None), (7, None), (8, 4), (9, 0), (10, 3), (11, None), (12, None), (13, None),
                   (3, 2), (5, need // 2), (11, fake + 4), (13, fake + 4)):
        a = list(g)
        a[i] = bad
        assert L.tl_betti_gather(*a) == -1, i
    dec = (ctypes.c_int32 * 12)(0, 1, 0, 3, 0, 0, 1, 1, 0, 2, 2, 2)
    a = list(g); a[7] = dec
    assert L.tl_betti_gather(*a) == -1 and b"decrease" in L.tl_last_error()
    b = [fake, fake, 3, 16, 16, fake, fake, 3, fake, 1, fake, 2, fake, fake, None, None]
    for i, bad in ((0, None), (1, None), (5, None), (6, None), (8, None), (10, None), (12, None), (13, None),
                   (2, 0), (7, -1), (6, fake + 4), (8, fake + 4), (10, fake + 4)):
        a = list(b)
        a[i] = bad
        assert L.tl_betti_backward(*a) == -1, i


def test_python_checks_raise_value_errors():
    import dilabhelmholtzoct_b200 as tlb
    x = torch.rand(2, 8, 8)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.betti_matching(x, x, 1)
    if torch.cuda.is_available():
        y = x.cuda()
        with pytest.raises(ValueError, match="shape"):
            tlb.betti_matching(y, y[:, :4], 1)
        with pytest.raises(ValueError, match="float32"):
            tlb.betti_matching(y.double(), y.double(), 1)
        with pytest.raises(ValueError, match="dim"):
            tlb.betti_matching(y, y, 2)


# ---------------------------------------------------------------- GPU

def _gpu_maps(kind, n, H, W, seed):
    rng = np.random.default_rng(seed)
    if kind == "signed":  # +-0.0, +-inf on a coarse grid
        x = rng.choice(np.array([-np.inf, -1.0, -0.0, 0.0, 0.5, 1.0, np.inf], np.float32), size=(n, H, W))
        return torch.from_numpy(x.astype(np.float32)).cuda()
    return torch.from_numpy(np.stack([_np_map(rng, kind, H, W) for _ in range(n)])).cuda()


def _records(bm, i):
    hm, hp, ht = bm.host_matched_offsets, bm.host_pred_offsets, bm.host_target_offsets
    return {"matched": bm.matched[hm[i]:hm[i + 1]].cpu().numpy(), "unmatched_pred": bm.unmatched_pred[hp[i]:hp[i + 1]].cpu().numpy(),
            "unmatched_target": bm.unmatched_target[ht[i]:ht[i + 1]].cpu().numpy()}


def _check_against_oracle(pred, target, dim, maps=None):
    import dilabhelmholtzoct_b200 as tlb
    bm = tlb.betti_matching(pred, target, dim)
    n = pred.reshape(-1, *pred.shape[-2:]).shape[0]
    P = pred.reshape(n, *pred.shape[-2:]).cpu().numpy()
    T = target.reshape(n, *pred.shape[-2:]).cpu().numpy()
    cost = bm.cost.detach().cpu().numpy()
    for i in (range(n) if maps is None else maps):
        want = betti_oracle.betti_matching(P[i], T[i], dim)
        got = _records(bm, i)
        for k in KEYS:
            assert np.array_equal(got[k], want[k]), (i, k)
        assert abs(float(cost[i]) - want["cost"]) <= 1e-6 * abs(want["cost"]) + 1e-30, (i, float(cost[i]), want["cost"])
    for off, host in ((bm.matched_offsets, bm.host_matched_offsets), (bm.pred_offsets, bm.host_pred_offsets),
                      (bm.target_offsets, bm.host_target_offsets)):
        assert off.cpu().tolist() == host
    return bm


BARCODE_CASES = [("random", 6, 32, 32), ("levels2", 5, 40, 40), ("levels32", 5, 48, 48), ("mask", 4, 64, 64),
                 ("signed", 4, 24, 24), ("random", 3, 1, 77), ("levels32", 3, 23, 1), ("random", 3, 24, 37),
                 ("levels32", 2, 256, 256), ("random", 1, 496, 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
@pytest.mark.parametrize("case", BARCODE_CASES, ids=lambda c: f"{c[0]}-{c[1]}x{c[2]}x{c[3]}")
def test_self_matching_is_the_barcode_of_cubical_persistence(case, dim):
    import dilabhelmholtzoct_b200 as tlb
    kind, n, H, W = case
    x = _gpu_maps(kind, n, H, W, seed=7 * H + W + n)
    bm = tlb.betti_matching(x, x, dim)
    D = tlb.cubical_persistence(x, dim)
    assert bm.host_pred_offsets[-1] == 0 and bm.host_target_offsets[-1] == 0
    flat = x.reshape(n, -1)
    for i in range(n):
        m = bm.matched[bm.host_matched_offsets[i]:bm.host_matched_offsets[i + 1]].long()
        assert torch.equal(m[:, :2], m[:, 2:])
        want = D.pairs[D.host_offsets[i]:D.host_offsets[i + 1]].long()
        assert sorted(map(tuple, m[:, :2].tolist())) == sorted(map(tuple, want.tolist())), i
        # values at those pixels, bit for bit, equal the diagram
        got_vals = {tuple(p): tuple(flat[i, p].view(torch.int32).tolist()) for p in m[:, :2].tolist()}
        want_vals = {tuple(p): tuple(v) for p, v in zip(want.tolist(), D.diagram[D.host_offsets[i]:D.host_offsets[i + 1]].detach().view(torch.int32).tolist())}
        assert got_vals == want_vals
    if kind != "signed":  # inf - inf is NaN
        assert torch.equal(bm.cost, torch.zeros_like(bm.cost))


ORACLE_CASES = [("random", "random", 6, 24, 24), ("levels2", "levels2", 6, 32, 32), ("levels4", "mask", 6, 32, 32),
                ("levels32", "levels32", 4, 48, 40), ("random", "mask", 3, 1, 64), ("random", "levels4", 2, 256, 256),
                ("signed", "signed", 4, 16, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
@pytest.mark.parametrize("case", ORACLE_CASES, ids=lambda c: f"{c[0]}-{c[1]}-{c[2]}x{c[3]}x{c[4]}")
def test_records_order_and_cost_equal_the_oracle(case, dim):
    kp, kt, n, H, W = case
    pred, target = _gpu_maps(kp, n, H, W, seed=H + n), _gpu_maps(kt, n, H, W, seed=W + 2 * n + 1)
    if kp == "signed":  # infinities make inf - inf terms; keep the signed zeros only
        pred, target = torch.nan_to_num(pred, posinf=2.0, neginf=-2.0), torch.nan_to_num(target, posinf=2.0, neginf=-2.0)
    _check_against_oracle(pred, target, dim)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
def test_full_c2_batch_sample_equals_the_oracle(dim):
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(64, 256, 256, seed=11, n_classes=14)
    _check_against_oracle(pred.cuda(), truth.cuda(), dim, maps=[0, 13, 200, 451, 777, 895])


def _autograd_reference(bm, pred, target, g):
    """d(sum_i g_i cost_i) by torch autograd of the cost formula on x.ravel()[indices] of the returned records."""
    n = pred.shape[0]
    p = pred.detach().reshape(n, -1).clone().requires_grad_(True)
    t = target.detach().reshape(n, -1).clone().requires_grad_(True)
    mid = lambda host: torch.repeat_interleave(torch.arange(n, device="cuda"), torch.tensor(np.diff(host), device="cuda"))
    m, up, ut = bm.matched.long(), bm.unmatched_pred.long(), bm.unmatched_target.long()
    im, ip, it = mid(bm.host_matched_offsets), mid(bm.host_pred_offsets), mid(bm.host_target_offsets)
    c = torch.zeros(n, device="cuda")
    c = c.index_add(0, im, (p[im, m[:, 0]] - t[im, m[:, 2]]) ** 2 + (p[im, m[:, 1]] - t[im, m[:, 3]]) ** 2)
    c = c.index_add(0, ip, (p[ip, up[:, 1]] - p[ip, up[:, 0]]) ** 2 / 2)
    c = c.index_add(0, it, (t[it, ut[:, 1]] - t[it, ut[:, 0]]) ** 2 / 2)
    (c * g).sum().backward()
    # magnitude bound: sum of |contributions| per pixel (the atomics add those in no fixed order)
    return c.detach(), p.grad, t.grad


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
def test_gradients_equal_autograd_of_the_cost(dim):
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(2, 64, 64, seed=2, n_classes=4)
    pred, truth = pred.cuda().reshape(-1, 64, 64), (0.8 * truth + 0.1 * torch.rand(truth.shape)).cuda().reshape(-1, 64, 64)
    p, t = pred.clone().requires_grad_(True), truth.clone().requires_grad_(True)
    bm = tlb.betti_matching(p, t, dim)
    g = torch.randn(len(bm), device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    (bm.cost * g).sum().backward()
    c, gp, gt = _autograd_reference(bm, pred, truth, g)
    assert torch.allclose(bm.cost.detach(), c, rtol=1e-5, atol=0)
    scale = max(float(gp.abs().max()), float(gt.abs().max()))
    assert float((p.grad.reshape(len(bm), -1) - gp).abs().max()) <= 1e-5 * scale
    assert float((t.grad.reshape(len(bm), -1) - gt).abs().max()) <= 1e-5 * scale
    # the target without requires_grad gets none, the prediction the same gradient
    p2 = pred.clone().requires_grad_(True)
    (tlb.betti_matching(p2, truth, dim).cost * g).sum().backward()
    assert torch.allclose(p2.grad, p.grad, rtol=0, atol=1e-6 * scale)


@pytest.mark.gpu
def test_backward_takes_a_misaligned_upstream_gradient():
    import dilabhelmholtzoct_b200 as tlb
    pred, truth = _gpu_maps("random", 3, 24, 24, 1), _gpu_maps("mask", 3, 24, 24, 2)
    p = pred.clone().requires_grad_(True)
    bm = tlb.betti_matching(p, truth, 1)
    head = torch.zeros(1, device="cuda", requires_grad=True)
    cat = torch.cat([head, bm.cost])
    w = torch.randn(cat.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    seen = {}
    bm.cost.register_hook(lambda gr: seen.update(ptr=gr.data_ptr()))
    (cat * w).sum().backward()
    torch.cuda.synchronize()
    assert seen["ptr"] % 8 == 4, "the graph no longer produces a misaligned gradient"
    _, gp, _ = _autograd_reference(bm, pred, truth, w[1:])
    assert float((p.grad.reshape(3, -1) - gp).abs().max()) <= 1e-5 * float(gp.abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
def test_superlevel_is_the_op_on_negated_maps(dim):
    import dilabhelmholtzoct_b200 as tlb
    pred, truth = _gpu_maps("levels32", 3, 32, 32, 4), _gpu_maps("mask", 3, 32, 32, 5)
    a = tlb.betti_matching(pred, truth, dim, superlevel=True)
    b = tlb.betti_matching(-pred, -truth, dim)
    assert torch.equal(a.cost, b.cost) and torch.equal(a.matched, b.matched)
    assert torch.equal(a.unmatched_pred, b.unmatched_pred) and torch.equal(a.unmatched_target, b.unmatched_target)
    p1, p2 = pred.clone().requires_grad_(True), (-pred).clone().requires_grad_(True)
    tlb.betti_matching(p1, truth, dim, superlevel=True).cost.sum().backward()
    tlb.betti_matching(p2, -truth, dim).cost.sum().backward()
    assert torch.allclose(p1.grad, -p2.grad, rtol=0, atol=1e-6)


@pytest.mark.gpu
def test_nan_map_raises():
    import dilabhelmholtzoct_b200 as tlb
    x = _gpu_maps("random", 3, 16, 16, 4)
    t = x.clone()
    t[2, 3, 3] = float("nan")
    with pytest.raises(RuntimeError, match="NaN"):
        tlb.betti_matching(x, t, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
def test_empty_and_constant_maps(dim):
    import dilabhelmholtzoct_b200 as tlb
    e = torch.zeros((0, 16, 16), device="cuda")
    bm = tlb.betti_matching(e, e, dim)
    assert len(bm) == 0 and bm.cost.shape == (0,)
    c = torch.full((3, 16, 16), 0.25, device="cuda").requires_grad_(True)
    bm = tlb.betti_matching(c, c.detach().clone(), dim)
    assert torch.equal(bm.cost.detach(), torch.zeros(3, device="cuda"))
    assert bm.host_pred_offsets[-1] == 0 and bm.host_matched_offsets[-1] == (3 if dim == 0 else 0)
    bm.cost.sum().backward()
    assert torch.equal(c.grad, torch.zeros_like(c))


@pytest.mark.gpu
def test_two_runs_give_identical_outputs():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(4, 128, 128, seed=9, n_classes=14)
    pred, truth = pred.cuda(), truth.cuda()
    for dim in (0, 1):
        a, b = tlb.betti_matching(pred, truth, dim), tlb.betti_matching(pred, truth, dim)
        for k in ("cost", "matched", "unmatched_pred", "unmatched_target"):
            assert torch.equal(getattr(a, k), getattr(b, k)), k


@pytest.mark.gpu
def test_backward_makes_no_host_sync():
    import dilabhelmholtzoct_b200 as tlb
    p = _gpu_maps("random", 4, 32, 32, 1).requires_grad_(True)
    t = _gpu_maps("mask", 4, 32, 32, 2).requires_grad_(True)
    bm = tlb.betti_matching(p, t, 1)
    loss = bm.cost.mean()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert bool(torch.isfinite(p.grad).all()) and bool(torch.isfinite(t.grad).all())
