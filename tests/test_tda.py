"""Differentiable persistence diagrams and Wasserstein distances (``dilabhelmholtzoct_b200.diagrams``) and the
torch_topological-compatible layer over them (``dilabhelmholtzoct_b200.tda``).

CPU: the new C entry points are declared and exported and reject bad arguments on the host; CPU tensors raise;
``batch_iter`` and the nesting helpers equal the torch_topological stand-ins in ``tests/golden/ref_stubs``.
GPU: pairs equal ``persistence_pairs``; diagram values equal ``x.ravel()[pairs]`` bit for bit; the backwards equal
torch autograd; the Wasserstein cost equals the transport LP; the reference orchestration written against the
compatibility layer reproduces the committed orchestration vectors; the composed loss equals the fused one.
"""
import ctypes
import importlib.util
import itertools
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STUBS = os.path.join(ROOT, "tests", "golden", "ref_stubs")
NEW = ["tl_diagrams_workspace_bytes", "tl_diagrams_compute", "tl_diagrams_gather", "tl_diagrams_backward",
       "tl_wasserstein_backward"]


def _load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _stub_data():
    return _load(os.path.join(STUBS, "torch_topological", "nn", "data.py"), "_stub_tt_data")


def _stub_nn():
    """The stand-ins' WassersteinDistance (its _make_distance_matrix) and ot.emd2 (scipy HiGHS)."""
    old = list(sys.path)
    sys.path[:0] = [STUBS, ROOT]
    try:
        import ot
        import torch_topological.nn as ttnn
    finally:
        sys.path[:] = old
    return ttnn, ot


# ---------------------------------------------------------------- CPU

def test_new_entry_points_are_declared_exported_and_bound():
    from dilabhelmholtzoct_b200 import _lib, build
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "topoloss.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(tl_[a-z_0-9]+)\s*\(", src))
    if not os.path.exists(build.LIB_PATH):
        build.build()
    L = ctypes.CDLL(build.LIB_PATH)
    for name in NEW:
        assert name in declared and hasattr(L, name) and name in _lib.SIGNATURES, name
    assert _lib.lib().tl_version() == _lib.ABI_VERSION == 5


def test_new_entry_points_reject_bad_arguments():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    nb = ctypes.c_size_t(0)
    assert L.tl_diagrams_workspace_bytes(3, 16, 16, 1, None) == -1
    assert L.tl_diagrams_workspace_bytes(3, 16, 16, 2, ctypes.byref(nb)) == -1 and b"feat_d" in L.tl_last_error()
    assert L.tl_diagrams_workspace_bytes(0, 16, 16, 1, ctypes.byref(nb)) == -1
    assert L.tl_diagrams_workspace_bytes(3, 16, 16, 1, ctypes.byref(nb)) == 0 and nb.value > 0
    need = nb.value
    fake = 4096  # never dereferenced: every call below fails its host-side checks first
    # compute: null pointers, dim = 2, a workspace smaller than the query asks for
    assert L.tl_diagrams_compute(None, 3, 16, 16, 1, fake, need, fake, None, None) == -1 and b"null" in L.tl_last_error()
    assert L.tl_diagrams_compute(fake, 3, 16, 16, 1, fake, need, None, None, None) == -1
    assert L.tl_diagrams_compute(fake, 3, 16, 16, 1, None, need, fake, None, None) == -1
    assert L.tl_diagrams_compute(fake, 3, 16, 16, 2, fake, need, fake, None, None) == -1
    assert L.tl_diagrams_compute(fake, 3, 16, 16, 1, fake, need - 1, fake, None, None) == -1
    assert b"workspace" in L.tl_last_error()
    # gather: P must agree with the host offsets
    host = (ctypes.c_int32 * 4)(0, 3, 5, 9)
    assert L.tl_diagrams_gather(fake, 3, 16, 16, 1, fake, need, fake, host, 8, fake, fake, None) == -1
    assert b"disagrees" in L.tl_last_error()
    bad = (ctypes.c_int32 * 4)(0, 5, 3, 9)
    assert L.tl_diagrams_gather(fake, 3, 16, 16, 1, fake, need, fake, bad, 9, fake, fake, None) == -1
    assert L.tl_diagrams_gather(fake, 3, 16, 16, 1, fake, need, fake, host, 9, None, fake, None) == -1
    assert L.tl_diagrams_gather(fake, 3, 16, 16, 1, fake, need, fake, None, 9, fake, fake, None) == -1
    assert L.tl_diagrams_gather(fake, 3, 16, 16, 2, fake, need, fake, host, 9, fake, fake, None) == -1
    assert L.tl_diagrams_gather(fake, 3, 16, 16, 1, fake, need // 2, fake, host, 9, fake, fake, None) == -1
    # backward
    assert L.tl_diagrams_backward(fake, None, fake, 9, 3, 16, 16, fake, None) == -1
    assert L.tl_diagrams_backward(None, fake, fake, 9, 3, 16, 16, fake, None) == -1
    assert L.tl_diagrams_backward(fake, fake, fake, 9, 3, 16, 16, None, None) == -1
    assert L.tl_diagrams_backward(fake, fake, fake, 9, 0, 16, 16, fake, None) == -1
    assert L.tl_diagrams_backward(fake, fake, fake, -1, 3, 16, 16, fake, None) == -1
    # wasserstein backward
    args = [fake] * 4 + [2, 2.0] + [fake] * 4 + [None]  # valid as they stand (would launch): only altered copies are passed
    for i in (0, 1, 2, 3, 6, 7):
        a = list(args)
        a[i] = None
        assert L.tl_wasserstein_backward(*a) == -1, i
    a = list(args); a[4] = 0
    assert L.tl_wasserstein_backward(*a) == -1
    a = list(args); a[5] = 0.0
    assert L.tl_wasserstein_backward(*a) == -1
    # [P][2] buffers are read as 8-byte pairs: a pointer 4 bytes off is an argument error, never a launch
    odd = fake + 4
    assert L.tl_diagrams_gather(fake, 3, 16, 16, 1, fake, need, fake, host, 9, odd, fake, None) == -1
    assert b"aligned" in L.tl_last_error()
    assert L.tl_diagrams_gather(fake, 3, 16, 16, 1, fake, need, fake, host, 9, fake, odd, None) == -1
    assert L.tl_diagrams_backward(odd, fake, fake, 9, 3, 16, 16, fake, None) == -1 and b"aligned" in L.tl_last_error()
    assert L.tl_diagrams_backward(fake, fake, odd, 9, 3, 16, 16, fake, None) == -1
    for i in (0, 2, 8, 9):
        a = list(args)
        a[i] = odd
        assert L.tl_wasserstein_backward(*a) == -1 and b"aligned" in L.tl_last_error(), i


def test_cpu_tensors_raise_value_errors_that_name_cuda():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200 import diagrams, tda
    x = torch.rand(2, 3, 8, 8)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.cubical_persistence(x, 1)
    with pytest.raises(ValueError, match="CUDA"):
        tda.CubicalComplex()(x)
    d = torch.rand(4, 2)
    with pytest.raises(ValueError, match="CUDA"):
        diagrams._wasserstein_packed(d, torch.tensor([0, 4]), [0, 4], d, torch.tensor([0, 4]), [0, 4])
    with pytest.raises(ValueError, match="p=inf"):
        tda.WassersteinDistance(p=2)
    with pytest.raises(ValueError):
        tda.CubicalComplex(dim=3)(x)
    with pytest.raises(RuntimeError, match="leading dimensions"):  # the exception torch_topological raises
        tda.CubicalComplex()(torch.rand(2, 2, 2, 8, 8))


def _nested(PI, depth, rng):
    """Nested lists of PersistenceInformation as CubicalComplex returns them: one map -> [PI0, PI1]."""
    def leaf():
        return [PI(pairing=int(rng.integers(100)), diagram=int(rng.integers(100)), dimension=d) for d in (0, 1)]
    if depth == 0:
        return leaf()
    if depth == 1:
        return [leaf() for _ in range(3)]
    return [[leaf() for _ in range(4)] for _ in range(2)]


def _plain(v):
    """PersistenceInformation -> plain tuple, lists and iterators -> lists (the two classes compare equal then)."""
    if isinstance(v, tuple):
        return tuple(v)
    if isinstance(v, int):
        return v
    return [_plain(e) for e in v]


def _outcome(batch_iter, x, dim):
    """What iterating batch_iter yields, or the exception it raises (one map filtered by dimension raises, as the
    reference does for B == C == 1)."""
    try:
        return [_plain(it) for it in batch_iter(x, dim=dim)]
    except Exception as e:  # noqa: BLE001
        return type(e)


def test_batch_iter_and_nesting_equal_the_stand_in():
    from dilabhelmholtzoct_b200 import tda
    stub = _stub_data()
    for depth in (0, 1, 2):
        for dim in (None, 0, 1):
            a = _nested(tda.PersistenceInformation, depth, np.random.default_rng(depth))
            b = _nested(stub.PersistenceInformation, depth, np.random.default_rng(depth))
            assert tda.nesting_level(a) == stub.nesting_level(b)
            assert _outcome(tda.batch_iter, a, dim) == _outcome(stub.batch_iter, b, dim), (depth, dim)
    assert tda.nesting_level([]) == stub.nesting_level([]) == 1
    pi = tda.PersistenceInformation(pairing=1, diagram=2)
    assert pi.dimension is None and tuple(pi) == tuple(stub.PersistenceInformation(pairing=1, diagram=2))


def test_total_persistence_equals_the_stand_in():
    from dilabhelmholtzoct_b200 import tda
    stub = _load(os.path.join(STUBS, "torch_topological", "utils", "__init__.py"), "_stub_tt_utils")
    D = torch.tensor([[0.1, 0.5], [0.2, float("inf")], [0.3, 0.35]])
    for p in (1, 2, 3):
        assert torch.equal(tda.total_persistence(D, p=p), stub.total_persistence(D, p=p))


# ---------------------------------------------------------------- GPU helpers

def _maps(kind, n, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "random":
        x = torch.rand((n, H, W), generator=g)
    elif kind == "levels2":
        x = torch.randint(0, 2, (n, H, W), generator=g).float() * 0.5
    elif kind == "levels32":
        x = torch.randint(0, 32, (n, H, W), generator=g).float() / 31
    elif kind == "mask":  # two-valued segmentation-like masks: blobs with holes
        x = torch.zeros((n, H, W))
        for i in range(n):
            for _ in range(4):
                r, c = torch.randint(0, H - 8, (2,), generator=g).tolist()
                x[i, r:r + 8, c:c + 8] = 1.0
                x[i, r + 3, c + 3] = 0.0
    elif kind == "const":
        x = torch.full((n, H, W), 0.25)
    else:
        raise ValueError(kind)
    return x.cuda()


def _check_against_pairs(x, dim, reference_shape_order=False):
    import dilabhelmholtzoct_b200 as tlb
    D = tlb.cubical_persistence(x, dim, reference_shape_order=reference_shape_order)
    want = tlb.persistence_pairs(x, dim, reference_shape_order=reference_shape_order)
    assert len(D) == len(want) and D.counts == [len(w) for w in want]
    assert D.offsets.cpu().tolist() == D.host_offsets
    got = D.pairs.cpu()
    for i, w in enumerate(want):
        assert torch.equal(got[D.host_offsets[i]:D.host_offsets[i + 1]], w.cpu()), i
    # values: x.ravel()[pairs] of each map, bit for bit
    flat = x.reshape(len(D), -1)
    mid = torch.repeat_interleave(torch.arange(len(D), device=x.device), torch.tensor(D.counts, device=x.device))
    vals = flat[mid[:, None], D.pairs.long()]
    assert torch.equal(D.diagram.detach().view(torch.int32), vals.view(torch.int32))
    return D


CASES = [("random", 6, 32, 32), ("levels2", 5, 40, 40), ("levels32", 5, 48, 48), ("mask", 4, 64, 64),
         ("random", 2, 512, 512), ("levels32", 1, 512, 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-{c[1]}x{c[2]}x{c[3]}")
def test_pairs_and_values_equal_persistence_pairs(case, dim):
    kind, n, H, W = case
    x = _maps(kind, n, H, W, seed=11 * H + n)
    _check_against_pairs(x, dim)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
def test_rectangular_maps_in_both_readings(dim):
    x = _maps("levels32", 3, 24, 37, seed=5).reshape(3, 1, 24, 37)
    a = _check_against_pairs(x, dim)
    b = _check_against_pairs(x, dim, reference_shape_order=True)
    assert a.host_offsets != b.host_offsets or not torch.equal(a.pairs, b.pairs)


@pytest.mark.gpu
def test_constant_map_and_empty_diagrams():
    import dilabhelmholtzoct_b200 as tlb
    x = _maps("const", 3, 16, 16, 0)
    D1 = _check_against_pairs(x, 1)
    assert D1.host_offsets == [0, 0, 0, 0] and D1.diagram.shape == (0, 2)
    D0 = _check_against_pairs(x, 0)
    assert D0.counts == [1, 1, 1] and torch.all(D0.diagram == 0.25)
    xr = x.clone().requires_grad_(True)
    D = tlb.cubical_persistence(xr, 1)
    D.diagram.sum().backward()  # no pairs: the gradient is all zeros
    assert torch.equal(xr.grad, torch.zeros_like(x))


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [0, 1])
def test_superlevel_is_the_op_on_minus_x(dim):
    import dilabhelmholtzoct_b200 as tlb
    x = _maps("levels32", 4, 40, 40, seed=3)
    a = tlb.cubical_persistence(x, dim, superlevel=True)
    b = tlb.cubical_persistence(-x, dim)
    assert a.host_offsets == b.host_offsets and torch.equal(a.pairs, b.pairs)
    assert torch.equal(a.diagram.view(torch.int32), b.diagram.view(torch.int32))
    # gradients: the scatter adds a pixel's contributions with atomics in no fixed order, so two runs agree within
    # the rounding of those sums (the bound of test_diagram_backward_equals_autograd_of_the_gather), not bit for bit
    xr = x.clone().requires_grad_(True)
    g = torch.randn(b.diagram.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    (tlb.cubical_persistence(xr, dim, superlevel=True).diagram * g).sum().backward()
    xm = (-x).clone().requires_grad_(True)
    (tlb.cubical_persistence(xm, dim).diagram * g).sum().backward()
    N = 40 * 40
    mid = torch.repeat_interleave(torch.arange(4, device="cuda"), torch.tensor(b.counts, device="cuda"))
    idx = (mid[:, None] * N + b.pairs.long()).reshape(-1)
    mag = torch.zeros(4 * N, dtype=torch.float64, device="cuda").index_put_((idx,), g.reshape(-1).double().abs(), accumulate=True)
    err = (xr.grad.reshape(-1).double() + xm.grad.reshape(-1).double()).abs()
    assert bool((err <= 2e-6 * mag).all()), float((err - 2e-6 * mag).max())


@pytest.mark.gpu
def test_backward_takes_a_misaligned_upstream_gradient():
    """Autograd can hand the backward a contiguous gradient that starts 4 bytes into its storage (a slice of a
    concatenation); the library reads [P, 2] rows as 8-byte pairs, so the op copies such a gradient first."""
    import dilabhelmholtzoct_b200 as tlb
    x = _maps("random", 2, 24, 24, 6)
    xr = x.clone().requires_grad_(True)
    D = tlb.cubical_persistence(xr, 1)
    head = torch.zeros(3, device="cuda", requires_grad=True)
    cat = torch.cat([head, D.diagram.view(-1)])
    w = torch.randn(cat.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(8))
    seen = {}
    D.diagram.register_hook(lambda gr: seen.update(ptr=gr.data_ptr()))  # returns None: the gradient is left as is
    (cat * w).sum().backward()
    torch.cuda.synchronize()
    assert seen["ptr"] % 8 == 4, "the graph no longer produces a misaligned gradient"
    N = 24 * 24
    mid = torch.repeat_interleave(torch.arange(2, device="cuda"), torch.tensor(D.counts, device="cuda"))
    idx = (mid[:, None] * N + D.pairs.long()).reshape(-1)
    gw = w[3:].double()
    ref = torch.zeros(2 * N, dtype=torch.float64, device="cuda").index_put_((idx,), gw, accumulate=True)
    mag = torch.zeros(2 * N, dtype=torch.float64, device="cuda").index_put_((idx,), gw.abs(), accumulate=True)
    assert bool(((xr.grad.reshape(-1).double() - ref).abs() <= 1e-6 * mag).all())
    # the Wasserstein op, with diagrams that start 4 bytes into their storage
    buf = torch.cat([torch.zeros(1, device="cuda"), D.diagram.detach().reshape(-1)])
    d1 = buf[1:].view(-1, 2)
    assert d1.data_ptr() % 8 == 4
    d1.requires_grad_(True)
    from dilabhelmholtzoct_b200 import diagrams
    T = tlb.cubical_persistence(_maps("mask", 2, 24, 24, 7), 1)
    cost = diagrams._wasserstein_packed(d1, D.offsets, D.host_offsets, T.diagram, T.offsets, T.host_offsets, 2)
    want = tlb.wasserstein_distance(D, T, 2)
    assert torch.equal(cost.detach(), want.detach())
    cost.sum().backward()
    assert bool(torch.isfinite(d1.grad).all())


@pytest.mark.gpu
def test_packed_wasserstein_checks_its_offsets():
    from dilabhelmholtzoct_b200 import diagrams
    d = torch.rand(4, 2, device="cuda")
    good = torch.tensor([0, 4], dtype=torch.int32, device="cuda")
    for off in (torch.tensor([0, 4], device="cuda"),                     # int64
                torch.tensor([0, 4], dtype=torch.int32),                 # host
                torch.tensor([0, 4, 4], dtype=torch.int32, device="cuda")):  # length
        with pytest.raises(ValueError, match="off1"):
            diagrams._wasserstein_packed(d, off, [0, 4], d, good, [0, 4])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["random", "levels2", "levels32"])
@pytest.mark.parametrize("dim", [0, 1])
def test_diagram_backward_equals_autograd_of_the_gather(kind, dim):
    import dilabhelmholtzoct_b200 as tlb
    x = _maps(kind, 3, 48, 48, seed=21).reshape(3, 1, 48, 48)
    xr = x.clone().requires_grad_(True)
    D = tlb.cubical_persistence(xr, dim)
    g = torch.randn(D.diagram.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(2))
    (D.diagram * g).sum().backward()
    # torch autograd through x.ravel()[pairs]: the gather's backward is index_put_(accumulate=True)
    N = 48 * 48
    mid = torch.repeat_interleave(torch.arange(3, device="cuda"), torch.tensor(D.counts, device="cuda"))
    idx = (mid[:, None] * N + D.pairs.long()).reshape(-1)
    ref = torch.zeros(3 * N, dtype=torch.float64, device="cuda").index_put_((idx,), g.reshape(-1).double(), accumulate=True)
    mag = torch.zeros(3 * N, dtype=torch.float64, device="cuda").index_put_((idx,), g.reshape(-1).double().abs(), accumulate=True)
    if kind != "levels2":  # (two-valued maps have a few pairs with distinct pixels)
        assert (torch.bincount(idx, minlength=3 * N) > 1).any(), "no pixel critical for several pairs"
    err = (xr.grad.reshape(-1).double() - ref).abs()
    assert bool((err <= 1e-6 * mag + 1e-30).all()), float((err - 1e-6 * mag).max())


# ---------------------------------------------------------------- Wasserstein

def _wcases():
    g = np.random.default_rng(7)

    def rnd(k):
        b = g.random(k).astype(np.float32)
        return np.stack([b, b + g.random(k).astype(np.float32) * (1 - b)], 1).astype(np.float32)
    out = {
        "random": (rnd(9), rnd(5)),
        "empty D1": (np.zeros((0, 2), np.float32), rnd(4)),
        "empty D2": (rnd(6), np.zeros((0, 2), np.float32)),
        "both empty": (np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32)),
        "diagonal points": (np.array([[0.3, 0.3], [0.1, 0.6], [0.5, 0.5]], np.float32),
                            np.array([[0.2, 0.2], [0.1, 0.55]], np.float32)),
        # |db| == |dd| for the matched pairs (L-inf ties) and equal costs among several matchings
        "ties": (np.array([[0.0, 0.5], [0.25, 0.75], [0.5, 1.0]], np.float32),
                 np.array([[0.125, 0.625], [0.375, 0.875]], np.float32)),
    }
    return out


def _plan_from_match(n, m, match):
    """The transport plan of the (n+1) x (m+1) problem that a matching of D1's rows describes."""
    G = np.zeros((n + 1, m + 1))
    used = np.zeros(m, bool)
    for i, j in enumerate(match):
        if j >= 0:
            G[i, j] = 1.0
            used[j] = True
        else:
            G[i, m] = 1.0
    G[n, np.nonzero(~used)[0]] = 1.0
    G[n, m] = m - (~used).sum()
    return G


def _grad_or_zeros(t):
    return t.grad if t.grad is not None else torch.zeros_like(t)


@pytest.mark.gpu
@pytest.mark.parametrize("q", [1, 2, 3])
def test_wasserstein_value_and_gradient_equal_the_lp_and_autograd(q):
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200 import diagrams
    ttnn, ot = _stub_nn()
    cases = _wcases()
    names = list(cases)
    A = [torch.tensor(cases[k][0], device="cuda") for k in names]
    B = [torch.tensor(cases[k][1], device="cuda") for k in names]
    d1, off1, h1 = diagrams._pack(A)
    d2, off2, h2 = diagrams._pack(B)
    d1 = d1.clone().requires_grad_(True)
    d2 = d2.clone().requires_grad_(True)
    cost = diagrams._wasserstein_packed(d1, off1, h1, d2, off2, h2, q)
    want, match = tlb.wasserstein_cost(A, B, q)
    assert torch.equal(cost.detach(), want.float())
    gc = torch.arange(1, len(names) + 1, dtype=torch.float32, device="cuda") * 0.5
    (cost * gc).sum().backward()
    wd = ttnn.WassersteinDistance(q=q)
    for k, name in enumerate(names):
        D1 = torch.tensor(cases[name][0], requires_grad=True)
        D2 = torch.tensor(cases[name][1], requires_grad=True)
        n, m = len(D1), len(D2)
        M = wd._make_distance_matrix(D1, D2)
        a, b = torch.ones(n + 1), torch.ones(m + 1)
        a[-1], b[-1] = m, n
        lp = float(ot.emd2(a, b, M))
        assert abs(float(cost[k]) - lp) <= 1e-6 * abs(lp) + 1e-12, (name, float(cost[k]), lp)
        # gradient: autograd of <G, M> with G the optimal plan of the matching (optimal: its cost is the LP's)
        G = _plan_from_match(n, m, match[k].cpu().tolist())
        assert abs(float((G * M.detach().double().numpy()).sum()) - lp) <= 1e-6 * abs(lp) + 1e-12, name
        (torch.tensor(G, dtype=torch.float32) * M).sum().mul(float(gc[k])).backward()
        g1 = d1.grad[h1[k]:h1[k + 1]].cpu()
        g2 = d2.grad[h2[k]:h2[k + 1]].cpu()
        w1, w2 = _grad_or_zeros(D1), _grad_or_zeros(D2)
        scale = max(float(w1.abs().max()) if n else 0.0, float(w2.abs().max()) if m else 0.0, 1e-30)
        assert torch.allclose(g1, w1, rtol=0, atol=1e-6 * scale), (name, g1, w1)
        assert torch.allclose(g2, w2, rtol=0, atol=1e-6 * scale), (name, g2, w2)
        if name == "random":  # unique optimum: the stand-in's own emd2 gradient (the LP's plan) agrees as well
            D1.grad, D2.grad = None, None
            ot.emd2(a, b, wd._make_distance_matrix(D1, D2)).mul(float(gc[k])).backward()
            assert torch.allclose(g1, D1.grad, rtol=0, atol=1e-6 * scale)
            assert torch.allclose(g2, D2.grad, rtol=0, atol=1e-6 * scale)


@pytest.mark.gpu
def test_wasserstein_skips_the_side_without_grad():
    from dilabhelmholtzoct_b200 import diagrams
    A = [torch.rand(5, 2, device="cuda")]
    B = [torch.rand(3, 2, device="cuda")]
    d1, off1, h1 = diagrams._pack(A)
    d2, off2, h2 = diagrams._pack(B)
    d1.requires_grad_(True)
    diagrams._wasserstein_packed(d1, off1, h1, d2, off2, h2, 2).sum().backward()
    assert d1.grad is not None and d2.grad is None


@pytest.mark.gpu
def test_ops_make_no_host_sync():
    import dilabhelmholtzoct_b200 as tlb
    x = _maps("random", 4, 32, 32, 1).requires_grad_(True)
    t = _maps("mask", 4, 32, 32, 2)
    Dx, Dt = tlb.cubical_persistence(x, 1), tlb.cubical_persistence(t, 1)
    De = tlb.cubical_persistence(_maps("const", 4, 32, 32, 0), 1)  # empty diagrams
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        cost = tlb.wasserstein_distance(Dx, Dt, q=2) + tlb.wasserstein_distance(Dx, De, q=2)
        cost.sum().backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert x.grad is not None and bool(torch.isfinite(x.grad).all())


@pytest.mark.gpu
def test_nan_map_raises_in_the_same_call():
    import dilabhelmholtzoct_b200 as tlb
    x = _maps("random", 3, 16, 16, 4)
    x[1, 5, 7] = float("nan")
    with pytest.raises(RuntimeError, match="NaN"):
        tlb.cubical_persistence(x, 1)


@pytest.mark.gpu
def test_batched_total_persistence_equals_per_map():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200 import tda
    D = tlb.cubical_persistence(_maps("random", 5, 24, 24, 9), 0)
    got = tlb.total_persistence(D, p=2)
    want = torch.stack([tda.total_persistence(d, p=2) for d in D.split()])
    assert torch.allclose(got, want, rtol=1e-6, atol=0)


# ---------------------------------------------------------------- compositions

def _reference_topo_loss(pred_obj, true_obj, lamda, interp=0, feat_d=2, loss_q=2, loss_r=False):
    """octsam/models/topological_loss.py:11-96 (SURVEY.md section 3.2) on the compatibility layer."""
    import torch.nn.functional as F
    from dilabhelmholtzoct_b200.tda import CubicalComplex, WassersteinDistance, batch_iter, total_persistence
    if lamda == 0.0:
        return 0.0
    if interp != 0:
        size = (interp, interp)
        pred_obj_ = F.interpolate(pred_obj, size=size, mode="bilinear", align_corners=True)
        true_obj_ = F.interpolate(true_obj, size=size, mode="bilinear", align_corners=True)
    else:
        pred_obj_, true_obj_ = pred_obj, true_obj
    cubical_complex = CubicalComplex(dim=2, superlevel=False)
    pers_info_pred = cubical_complex(pred_obj_.squeeze())
    pers_info_true = cubical_complex(true_obj_.squeeze())
    dim = feat_d if 0 <= feat_d <= 2 else None
    pred_batch = batch_iter(pers_info_pred, dim=dim)
    true_batch = batch_iter(pers_info_true, dim=dim)
    wasserstein = WassersteinDistance(q=loss_q)
    topo_losses = [wasserstein(p, t) for p, t in zip(pred_batch, true_batch)]
    topological_loss = torch.stack(topo_losses).mean()
    if loss_r:
        reg = [total_persistence(info.diagram, p=loss_q)
               for info in itertools.chain.from_iterable(batch_iter(pers_info_pred, dim=dim))]
        topological_loss = topological_loss + torch.stack(reg).mean()
    return lamda * topological_loss


@pytest.mark.gpu
def test_reference_orchestration_on_the_layer_reproduces_the_vectors():
    with open(os.path.join(ROOT, "tests", "golden", "orchestration_vectors.json")) as fh:
        doc = json.load(fh)
    REL = 1e-5
    assert len(doc["cases"]) == 18
    for case in doc["cases"]:
        p = torch.tensor(case["pred"], device="cuda", requires_grad=True)
        loss = _reference_topo_loss(p, torch.tensor(case["truth"], device="cuda"), case["lamda"], interp=case["interp"],
                                    feat_d=case["feat_d"], loss_q=case["q"], loss_r=case["loss_r"])
        loss.backward()
        want_g = np.array(case["grad"], np.float32)
        assert abs(float(loss) - case["loss"]) <= REL * abs(case["loss"]) + 1e-12, (case["note"], float(loss), case["loss"])
        tol = (10 * REL if case["interp"] else REL) * np.abs(want_g).max() + 1e-12
        g = p.grad.cpu().numpy()
        assert g.shape == want_g.shape and np.abs(g - want_g).max() <= tol, case["note"]
        if not case["interp"]:
            assert np.array_equal(g != 0, want_g != 0), ("critical pixels differ", case["note"])


def composed_topo_loss(pred, truth, lamda, feat_d=1, q=2):
    """The fused loss (interp = 0, B > 1, C > 1) composed from the batched ops."""
    import dilabhelmholtzoct_b200 as tlb
    B, C = pred.shape[:2]
    cost = tlb.wasserstein_distance(tlb.cubical_persistence(pred, feat_d), tlb.cubical_persistence(truth, feat_d), q=q)
    return lamda * cost.view(B, C).sum(1).pow(1.0 / q).mean()


@pytest.mark.gpu
def test_composed_loss_equals_the_fused_loss():
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200.synthetic import make_batch
    pred, truth = make_batch(4, 256, 256, seed=3)
    pred, truth = pred.cuda(), truth.cuda()
    assert pred.shape[:2] == (4, 14)
    a = pred.clone().requires_grad_(True)
    fused = tlb.topo_loss(a, truth, 0.1, feat_d=1)
    fused.backward()
    b = pred.clone().requires_grad_(True)
    comp = composed_topo_loss(b, truth, 0.1)
    comp.backward()
    assert abs(float(comp) - float(fused)) <= 1e-5 * abs(float(fused)), (float(comp), float(fused))
    ga, gb = a.grad, b.grad
    assert float((ga - gb).abs().max()) <= 1e-5 * float(ga.abs().max())
    assert torch.equal(ga != 0, gb != 0)
