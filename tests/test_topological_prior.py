"""Topological prior loss (``dilabhelmholtzoct_b200.prior``): per-map Betti-number priors on cubical persistence.

CPU: a numpy oracle on ``oracle.cubical_pairs`` (stable argsort, fp64) gives the cost and a float64 per-pixel
gradient; hand-derived KATs, sub- and superlevel, with their values written out; the C entry points are declared,
exported, bound and reject bad arguments without a launch; CPU tensors and bad ``betti`` raise.
GPU: cost and gradient against the oracle on random, tie-heavy, two-valued, constant and rectangular maps with
per-map betti (0 and above the count included), a persistence tie at the betti boundary, value and gradient against
torch autograd of the composed form on ``cubical_persistence``, every form of ``betti``, determinism, no host sync,
NaN maps, negative device betti, no maps.
"""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["tl_prior_workspace_bytes", "tl_prior_forward", "tl_prior_backward"]
EPS32 = float(np.finfo(np.float32).eps)


def prior_oracle(f, dim, beta, superlevel=False):
    """Cost (fp64), d cost / d f (float64 [H, W]), the per-pixel sum of |contributions|, and per record of the
    diagram (gudhi order) its persistence p (fp32) and whether it is selected."""
    f = np.ascontiguousarray(f, dtype=np.float32)
    g = -f if superlevel else f
    pairs = oracle.cubical_pairs(g, dim).astype(np.int64).reshape(-1, 2)
    flat = g.ravel()
    b, d = flat[pairs[:, 0]], flat[pairs[:, 1]]
    p = np.abs(d - b)  # fp32 subtraction, as the op
    rank = np.empty(len(p), np.int64)
    rank[np.argsort(-p, kind="stable")] = np.arange(len(p))  # p descending, ties by position
    sel = rank < beta
    p64 = p.astype(np.float64)
    cost = float(np.sum(np.where(sel, 1.0 - p64 * p64, p64 * p64))) + max(0, beta - len(p))
    gd = np.where(sel, -2.0, 2.0) * (d.astype(np.float64) - b.astype(np.float64))
    grad, mag = np.zeros(f.size), np.zeros(f.size)
    np.add.at(grad, pairs[:, 1], gd)
    np.add.at(grad, pairs[:, 0], -gd)
    np.add.at(mag, pairs[:, 1], np.abs(gd))
    np.add.at(mag, pairs[:, 0], np.abs(gd))
    if superlevel:
        grad = -grad
    return {"cost": cost, "grad": grad.reshape(f.shape), "mag": mag.reshape(f.shape), "p": p, "sel": sel}


# ---------------------------------------------------------------- hand-derived KATs

def _blobs(vals, bg, H=12, W=18):
    """2x2 blobs of the given values at fixed places on a constant background."""
    x = np.full((H, W), bg, np.float32)
    for (r, c), v in zip([(2, 2), (7, 11)], vals):
        x[r:r + 2, c:c + 2] = v
    return x


def _ring(v, bg, H=9, W=11):
    """A 3x3 ring of value v around one pixel of the background value."""
    x = np.full((H, W), bg, np.float32)
    x[3:6, 4:7] = v
    x[4, 5] = bg
    return x


# (name, map, dim, superlevel, {beta: cost}).  Two blobs: H0 = {(0.6, 1) or (-0.6, 0): p 0.6, essential: p 0.9};
# cost = 0.81 + 0.36 for beta 0, (1 - 0.81) + 0.36 for 1, (1 - 0.81) + (1 - 0.36) for 2, and + 1 of padding for 3.
# Ring: H1 = {p 0.8}: 0.64 for beta 0, 1 - 0.64 for beta 1.  Constant map: H0 = {essential, p 0}, H1 = {}.
KATS = [
    ("blobs-sub", _blobs([0.1, 0.4], 1.0), 0, False, {0: 1.17, 1: 0.55, 2: 0.83, 3: 1.83}),
    ("blobs-super", _blobs([0.9, 0.6], 0.0), 0, True, {0: 1.17, 1: 0.55, 2: 0.83, 3: 1.83}),
    ("ring-sub", _ring(0.2, 1.0), 1, False, {0: 0.64, 1: 0.36}),
    ("ring-super", _ring(0.8, 0.0), 1, True, {0: 0.64, 1: 0.36}),
    ("const-h0", np.full((6, 7), 0.5, np.float32), 0, False, {0: 0.0, 1: 1.0, 2: 2.0}),
    ("const-h1", np.full((6, 7), 0.5, np.float32), 1, True, {0: 0.0, 1: 1.0}),
]


@pytest.mark.parametrize("kat", KATS, ids=lambda k: k[0])
def test_kats_on_the_oracle(kat):
    _, x, dim, sup, want = kat
    for beta, cost in want.items():
        r = prior_oracle(x, dim, beta, sup)
        assert abs(r["cost"] - cost) <= 1e-6, (beta, r["cost"], cost)


def test_kat_gradients_by_hand():
    """Superlevel blobs, beta = 1: the essential class (p = 0.9) is pushed up, the second blob (p = 0.6) down.  On
    f = -x: d(1 - p^2)/d death = -2 * 0.9 at the argmax (a background pixel, f = 0), +2 * 0.9 at the blob's minimum
    pixel; d(p^2)/d death = +2 * 0.6, d/d birth = -2 * 0.6.  With respect to x the signs flip: -1.8 on the first
    blob, +1.2 on the second, the rest on background pixels."""
    x = _blobs([0.9, 0.6], 0.0)
    r = prior_oracle(x, 0, 1, True)
    g = r["grad"]
    assert abs(g[2:4, 2:4].sum() - (-2 * 0.9)) <= 1e-6 and abs(g[7:9, 11:13].sum() - 2 * 0.6) <= 1e-6
    assert abs(g.sum()) <= 1e-6                 # every record moves a birth and a death by opposite amounts
    assert np.count_nonzero(g[2:4, 2:4]) == 1 and np.count_nonzero(g[7:9, 11:13]) == 1
    assert list(r["sel"]) == [False, True]      # the finite pair first, the essential class last


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
    assert "topological_prior" in tlb.__all__ and callable(tlb.topological_prior)


def _sizes(L, n, H, W, dim):
    ns, nc = ctypes.c_size_t(0), ctypes.c_size_t(0)
    rc = L.tl_prior_workspace_bytes(n, H, W, dim, ctypes.byref(ns), ctypes.byref(nc))
    return rc, ns.value, nc.value


def test_new_entry_points_reject_bad_arguments():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    nb = ctypes.c_size_t(0)
    assert L.tl_prior_workspace_bytes(3, 16, 16, 1, None, ctypes.byref(nb)) == -1
    assert L.tl_prior_workspace_bytes(3, 16, 16, 1, ctypes.byref(nb), None) == -1
    for bad in ((3, 16, 16, 2), (0, 16, 16, 1), (3, 0, 16, 1), (3, 16, -1, 0)):
        assert _sizes(L, *bad)[0] == -1, bad
    rc, ns, nc = _sizes(L, 3, 16, 16, 1)
    assert rc == 0 and ns > 0 and nc > 0
    # the state holds the pairs layout's state part plus the thresholds; the scratch its scratch part
    pb = ctypes.c_size_t(0)
    assert L.tl_diagrams_workspace_bytes(3, 16, 16, 1, ctypes.byref(pb)) == 0
    assert ns + nc == pb.value + 256  # one 256-byte block of threshold keys for 3 maps
    fake = 4096  # never dereferenced: every call below fails its host-side checks first
    ok = [fake, 3, 16, 16, 1, fake, fake, ns, fake, nc, fake, None]
    for i, bad in ((0, None), (5, None), (6, None), (8, None), (10, None), (1, 0), (2, 0), (4, 2), (4, -1),
                   (7, ns - 1), (9, nc - 1)):
        a = list(ok)
        a[i] = bad
        assert L.tl_prior_forward(*a) == -1, i
    assert L.tl_prior_forward(*(ok[:7] + [ns - 1] + ok[8:])) == -1 and b"tl_prior_workspace_bytes" in L.tl_last_error()
    b = [fake, 3, 16, 16, 1, fake, ns, fake, fake, None]
    for i, bad in ((0, None), (5, None), (7, None), (8, None), (1, -2), (3, 0), (4, 5), (6, ns // 2)):
        a = list(b)
        a[i] = bad
        assert L.tl_prior_backward(*a) == -1, i


def test_python_checks_raise_value_errors():
    import dilabhelmholtzoct_b200 as tlb
    x = torch.rand(2, 3, 8, 8)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.topological_prior(x, 0, 1)
    with pytest.raises(ValueError, match="dim"):
        tlb.topological_prior(x, 2, 1)
    for bad, what in ((-1, ">= 0"), ([1, -2, 0], ">= 0"), (torch.tensor([[0], [-1]]), ">= 0"), ([1, 2], "broadcast"),
                      (torch.ones(3, 2, dtype=torch.int64), "broadcast"), (torch.ones(2, 3, 1, dtype=torch.int32), "broadcast"),
                      (1.0, "integer"), ([0.5, 1.0, 2.0], "integer"), (torch.ones(3), "integer"), (True, "integer"),
                      ("one", "int")):
        with pytest.raises(ValueError, match=what):
            tlb.topological_prior(x, 0, bad)
    with pytest.raises(ValueError):
        tlb.topological_prior(torch.rand(8), 0, 1)
    if torch.cuda.is_available():
        y = x.cuda()
        with pytest.raises(ValueError, match="float32"):
            tlb.topological_prior(y.double(), 0, 1)
        with pytest.raises(ValueError, match="broadcast"):
            tlb.topological_prior(y, 1, torch.zeros(4, dtype=torch.int32, device="cuda"))


# ---------------------------------------------------------------- GPU

def _np_map(rng, kind, H, W):
    if kind == "random":
        return rng.random((H, W)).astype(np.float32)
    if kind.startswith("levels"):
        k = int(kind[6:])
        return (np.floor(rng.random((H, W)) * k) / k).astype(np.float32)
    if kind == "mask":
        return (rng.random((H, W)) < 0.4).astype(np.float32)
    if kind == "const":
        return np.full((H, W), 0.5, np.float32)
    raise ValueError(kind)


def _check(x, dim, betti, superlevel, g=None, c=8.0):
    """Cost and gradient of the op on x [n, H, W] (CUDA) against the oracle, map by map."""
    import dilabhelmholtzoct_b200 as tlb
    n = x.shape[0]
    xr = x.clone().requires_grad_(True)
    cost = tlb.topological_prior(xr, dim, torch.tensor(betti, dtype=torch.int32), superlevel=superlevel)
    g = torch.ones(n, device="cuda") if g is None else g
    (cost * g).sum().backward()
    X, got_c, got_g, gh = x.cpu().numpy(), cost.detach().cpu().numpy(), xr.grad.cpu().numpy(), g.cpu().numpy()
    out = []
    for i in range(n):
        r = prior_oracle(X[i], dim, int(betti[i]), superlevel)
        assert abs(float(got_c[i]) - r["cost"]) <= EPS32 * abs(r["cost"]), (i, float(got_c[i]), r["cost"])
        want = r["grad"] * float(gh[i])
        tol = c * EPS32 * r["mag"] * abs(float(gh[i]))
        assert np.all(np.abs(got_g[i] - want) <= tol), (i, float(np.abs(got_g[i] - want).max()))
        out.append(r)
    return got_c, got_g, out


CASES = [("random", 6, 32, 32), ("levels2", 5, 24, 24), ("levels4", 5, 32, 32), ("levels32", 5, 40, 40),
         ("mask", 4, 48, 48), ("const", 3, 16, 16), ("random", 3, 24, 37), ("levels4", 3, 1, 50),
         ("levels32", 2, 256, 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("superlevel", [False, True], ids=["sub", "super"])
@pytest.mark.parametrize("dim", [0, 1])
@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-{c[1]}x{c[2]}x{c[3]}")
def test_cost_and_gradient_equal_the_oracle(case, dim, superlevel):
    kind, n, H, W = case
    rng = np.random.default_rng(31 * H + W + n + 7 * dim)
    X = np.stack([_np_map(rng, kind, H, W) for _ in range(n)])
    counts = [len(oracle.cubical_pairs(-X[i] if superlevel else X[i], dim)) for i in range(n)]
    # per map: 0, 1, half the count, the count, above it
    betti = [(0, 1, counts[i] // 2, counts[i], counts[i] + 3)[i % 5] for i in range(n)]
    g = torch.from_numpy(rng.standard_normal(n).astype(np.float32)).cuda()
    _check(torch.from_numpy(X).cuda(), dim, betti, superlevel, g=g)


@pytest.mark.gpu
@pytest.mark.parametrize("superlevel", [False, True], ids=["sub", "super"])
@pytest.mark.parametrize("dim", [0, 1])
def test_tie_at_the_betti_boundary(dim, superlevel):
    """levels4 maps: many equal persistences.  Each map's betti cuts a group of equal p, so which records of the
    group are selected rests on the position rule alone.  Values are multiples of 1/4, so every term is exact and
    the gradient equals the oracle's bit for bit, support included."""
    rng = np.random.default_rng(5 + dim)
    X = np.stack([_np_map(rng, "levels4", 32, 32) for _ in range(6)])
    betti, tied = [], []
    for i in range(len(X)):
        r = prior_oracle(X[i], dim, 0, superlevel)
        p = np.sort(r["p"])[::-1]
        ks = [k for k in range(1, len(p)) if p[k - 1] == p[k] and p[k] > 0]
        betti.append(ks[len(ks) // 2] if ks else 1)
        tied.append(bool(ks))
    assert sum(tied) >= 4, "the maps no longer have ties at the boundary"
    _, got, rs = _check(torch.from_numpy(X).cuda(), dim, betti, superlevel)
    for i, r in enumerate(rs):
        sel, p = r["sel"], r["p"]
        assert sel.sum() == min(betti[i], len(p))
        if tied[i]:  # the group of equal p at the boundary is split: some of it selected, some not
            t = np.sort(p)[::-1][betti[i] - 1]
            assert sel[p == t].any() and not sel[p == t].all()
        assert np.array_equal(got[i], r["grad"]), i
        assert np.array_equal(got[i] != 0, r["grad"] != 0), i


def _composed(x, dim, betti, superlevel=False):
    """The same loss from cubical_persistence, two stable sorts and the formula in torch (fp64 terms)."""
    import dilabhelmholtzoct_b200 as tlb
    D = tlb.cubical_persistence(x, dim, superlevel=superlevel)
    n, P, dev = len(D), D.host_offsets[-1], x.device
    cnt = (D.offsets[1:] - D.offsets[:-1]).long()
    p = (D.diagram[:, 1] - D.diagram[:, 0]).abs()
    seg = torch.repeat_interleave(torch.arange(n, device=dev), cnt, output_size=P)
    o1 = torch.sort(p.detach(), descending=True, stable=True).indices
    order = o1[torch.sort(seg[o1], stable=True).indices]  # by map, p descending, ties by position
    rank = torch.empty_like(order)
    rank[order] = torch.arange(P, device=dev) - D.offsets[:-1].long()[seg[order]]
    b = betti.to(dev).long().reshape(-1)
    p64 = p.double()
    terms = torch.where(rank < b[seg], 1.0 - p64 * p64, p64 * p64)
    cost = torch.zeros(n, dtype=torch.float64, device=dev).index_add(0, seg, terms)
    return (cost + (b - cnt).clamp(min=0).double()).float()


@pytest.mark.gpu
@pytest.mark.parametrize("superlevel", [False, True], ids=["sub", "super"])
@pytest.mark.parametrize("dim", [0, 1])
def test_value_and_gradient_equal_autograd_of_the_composed_form(dim, superlevel):
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, _ = make_batch(2, 64, 64, seed=4, n_classes=4)
    pred = pred.cuda()
    betti = torch.tensor([[1, 0, 2, 5], [0, 1, 1, 40]], dtype=torch.int32)
    g = torch.randn(2, 4, device="cuda", generator=torch.Generator("cuda").manual_seed(2))
    a, b = pred.clone().requires_grad_(True), pred.clone().requires_grad_(True)
    ca = tlb.topological_prior(a, dim, betti, superlevel=superlevel)
    cb = _composed(b, dim, betti, superlevel=superlevel)
    assert ca.shape == (8,)
    assert torch.allclose(ca.detach(), cb.detach(), rtol=2 * EPS32, atol=0)
    (ca * g.reshape(-1)).sum().backward()
    (cb * g.reshape(-1)).sum().backward()
    scale = float(b.grad.abs().max())
    assert scale > 0 and float((a.grad - b.grad).abs().max()) <= 1e-5 * scale


@pytest.mark.gpu
def test_betti_forms_give_identical_costs():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(3)
    x = torch.from_numpy(np.stack([_np_map(rng, "levels32", 24, 24) for _ in range(6)])).cuda().reshape(2, 3, 24, 24)
    for dim in (0, 1):
        ref = tlb.topological_prior(x, dim, 2)
        for b in (torch.tensor(2), torch.full((2, 3), 2, dtype=torch.int16), torch.full((3,), 2, device="cuda"),
                  torch.tensor([[2], [2]], dtype=torch.int32, device="cuda"), [2, 2, 2], [[2, 2, 2], [2, 2, 2]]):
            assert torch.equal(tlb.topological_prior(x, dim, b), ref), b
        per = [[0, 1, 2], [3, 4, 5]]
        ref = tlb.topological_prior(x, dim, per)
        for b in (torch.tensor(per), torch.tensor(per, dtype=torch.int32, device="cuda"), np.array(per)):
            assert torch.equal(tlb.topological_prior(x, dim, b), ref)


@pytest.mark.gpu
def test_two_runs_are_bit_identical():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, _ = make_batch(4, 128, 128, seed=9, n_classes=14)
    pred = pred.cuda()
    for dim, beta in ((0, 1), (1, 0), (1, 3)):
        outs = []
        for _ in range(2):
            p = pred.clone().requires_grad_(True)
            c = tlb.topological_prior(p, dim, beta, superlevel=True)
            c.sum().backward()
            outs.append((c.detach(), p.grad))
        assert torch.equal(outs[0][0].view(torch.int32), outs[1][0].view(torch.int32))
        assert bool(torch.isfinite(outs[0][0]).all())
        scale = float(outs[0][1].abs().max())
        assert float((outs[0][1] - outs[1][1]).abs().max()) <= 1e-6 * scale  # atomics add in any order


@pytest.mark.gpu
def test_forward_and_backward_make_no_host_sync():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(8)
    x = torch.from_numpy(np.stack([_np_map(rng, "random", 32, 32) for _ in range(6)])).cuda()
    bdev = torch.tensor([0, 1, 2, 0, 1, 2], dtype=torch.int64, device="cuda")
    for beta in (1, bdev):  # warm-up: buffers, the status ring, module loading
        tlb.topological_prior(x.clone().requires_grad_(True), 0, beta, superlevel=True).sum().backward()
    torch.cuda.synchronize()
    grads = []
    torch.cuda.set_sync_debug_mode("error")
    try:
        for dim, beta in ((0, 1), (1, bdev)):
            p = x.clone().requires_grad_(True)
            tlb.topological_prior(p, dim, beta, superlevel=True).mean().backward()
            grads.append(p.grad)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert all(bool(torch.isfinite(g).all()) for g in grads)


@pytest.mark.gpu
def test_nan_map_gives_nan_costs_then_raises():
    import dilabhelmholtzoct_b200 as tlb
    tlb.check_status()
    rng = np.random.default_rng(4)
    x = torch.from_numpy(np.stack([_np_map(rng, "random", 16, 16) for _ in range(3)])).cuda()
    x[1, 3, 3] = float("nan")
    cost = tlb.topological_prior(x, 1, 0)
    assert bool(torch.isnan(cost).all())
    with pytest.raises(RuntimeError, match="topological_prior"):
        tlb.check_status()
    tlb.check_status()  # reported once


@pytest.mark.gpu
def test_negative_device_betti_gives_nan_for_that_map_only():
    import dilabhelmholtzoct_b200 as tlb
    rng = np.random.default_rng(6)
    X = np.stack([_np_map(rng, "random", 20, 20) for _ in range(3)])
    x = torch.from_numpy(X).cuda().requires_grad_(True)
    cost = tlb.topological_prior(x, 0, torch.tensor([1, -1, 0], device="cuda"))
    cost.nansum().backward()
    c = cost.detach().cpu().numpy()
    assert np.isnan(c[1]) and np.isfinite(c[[0, 2]]).all()
    for i, beta in ((0, 1), (2, 0)):
        r = prior_oracle(X[i], 0, beta)
        assert abs(float(c[i]) - r["cost"]) <= EPS32 * r["cost"]
    assert bool(torch.isnan(x.grad[1]).all()) and bool(torch.isfinite(x.grad[[0, 2]]).all())
    tlb.check_status()  # a negative betti is not a status bit


@pytest.mark.gpu
def test_no_maps_give_an_empty_cost():
    import dilabhelmholtzoct_b200 as tlb
    for shape in ((0, 16, 16), (2, 0, 8, 8)):
        x = torch.zeros(shape, device="cuda", requires_grad=True)
        c = tlb.topological_prior(x, 1, 0)
        assert c.shape == (0,) and c.dtype == torch.float32
        c.sum().backward()
        assert x.grad.shape == x.shape


@pytest.mark.gpu
@pytest.mark.parametrize("kat", KATS, ids=lambda k: k[0])
def test_kats_on_the_gpu(kat):
    import dilabhelmholtzoct_b200 as tlb
    _, x, dim, sup, want = kat
    betas = list(want)
    X = torch.from_numpy(np.stack([x] * len(betas))).cuda()
    got = tlb.topological_prior(X, dim, betas, superlevel=sup).cpu().numpy()
    for j, beta in enumerate(betas):
        assert abs(float(got[j]) - want[beta]) <= 1e-6, (beta, float(got[j]), want[beta])
