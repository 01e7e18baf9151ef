"""The loss's diagram matching on every path it takes, under ties and at every loss_q, against a float64 reference.

Between the persistence pairs and the gradient, every map of ``topo_loss`` goes through one of these branches
(``match_small.cuh``, ``match_kernel.cuh``), chosen by its pair counts n (prediction) and m (ground truth):

* ``R0``       min(n, m) == 0: the cost is the two diagonal sums the persistence kernel formed while emitting;
* ``cached``   1 <= min(n, m) <= kSmallR and max(n, m) <= kColCache: ``match_one_map`` with its columns in shared memory;
* ``uncached`` 1 <= min(n, m) <= kSmallR and max(n, m) > kColCache: the same, columns read from global memory;
* ``heavy``    min(n, m) > kSmallR: the map goes to the heavy list and ``match_kernel``.

Each comes in two orientations: the ground truth is the rows (n > m), or the prediction is (n < m, ``swapped``);
plus n == m (rows = ground truth).  The matching runs in the persistence launch's tail (default), in its own launch
(``OPT_NO_FUSED_MATCH``, and after the global-memory persistence kernel, ``OPT_FORCE_GLOBAL_KERNEL``), or in
``match_kernel``; the gradient in the tail or in ``grad_kernel`` (``OPT_NO_FUSED_GRAD``).  Every GPU case runs under
all four routes, two-valued cases also without the two-valued H1 path (``OPT_NO_BINARY_PATH``).

Inputs are maps with designed diagrams: isolated single-pixel peaks (H1) or pits (H0), and 3 x 3 blocks whose
centre and ring set the point's two values.  Every count and value is checked against ``oracle.cubical_pairs``.

Reference (CPU, float64).  Cost entries are formed as the kernels form them: fp32 L-inf, then ``powq`` in fp32
(``x * x`` for q = 2, ``powf`` otherwise).  The optimum is checked with ``scipy.optimize.linear_sum_assignment`` on
the augmented square form of torch_topological's (n+1) x (m+1) emd2 LP, which shares no code with the oracle's
Hungarian solver.  Large diagrams with few rows are first reduced exactly: in an optimal matching each row is on
the diagonal or on one of its R cheapest columns by ``c(r, k) - diag(k)`` (otherwise one of those R is free and
no dearer), so only the union of those columns is kept.  The assignment is ``oracle.wasserstein``'s, after its
cost has been shown to equal the LSA optimum to 1e-12 of the magnitude summed (the diagonal costs: both are fp64
sums of the same fp32 entries in different orders).  The kernels match the diagrams in the order the
persistence kernels emit the records -- raster order of the dying basin: the destroyer pixel for H1, the creator
pixel for H0 (the root vertex is the creator pixel's top-left corner in every map built here; single-band maps
only) -- so the oracle is run on the diagrams in that order: its tie-breaks (smallest column, earliest tree row)
then name the kernels' matching.  The gradient is built in float64 from that assignment with the formulas of
``pair_gradient`` / ``image_coef``, together with the per-pixel sum of the absolute values of its terms and their
number.

Tolerances.
* Gradient, per pixel: ``|got - ref| <= (k + 1) * 2^-24 * sum|terms| + tiny``, k = the number of terms added into
  the pixel.  The kernels round each fp64 term to fp32 and add it with atomics in any order; a pixel is never
  bounded relative to its own value (two terms that cancel there would break that).  For q not in {1, 2} the
  image coefficient ``S_b^(1/q - 1)`` inherits the cost's 1e-6 relative uncertainty (device ``powf``), so
  ``|1/q - 1| * 1e-6 * sum|coefficient parts|`` is added.  That sum is taken over the terms' coefficient parts alone:
  with loss_r each term is the coefficient part minus the regulariser's part, and where the two nearly cancel the
  coefficient's error is far larger than the term.
* Exact assignments, q in {1, 2}: the entries are bit-reproducible on the host (q = 2 squares an fp32 L-inf; for
  q = 1 the device's ``powf(x, 1.0f)`` returns x, which ``test_q1_cost_entries_are_exact`` confirms).  The matching
  must then be the oracle's own, ties included, so the gradient support equals the reference's exactly: a pixel
  without terms must be exactly 0, and a pixel whose reference value exceeds its bound must be non-zero.
* q not in {1, 2}: the device ``powf`` may differ from the host's in the last bits, so only inputs whose optimum is
  unique are used: with float64 entries, the best assignment beats every alternative by more than 1e-4 of the
  optimal cost (each row's match, or its diagonal, forbidden in turn and the problem re-solved).  Entries that are
  a few ulps off move an assignment's cost by far less than that.
* Loss: 1e-6 relative against the reference (its S_b summed in fp32 as the kernels do).  The loss is identical
  bit for bit across the default route, ``OPT_NO_FUSED_GRAD`` and ``OPT_NO_FUSED_MATCH``; the global-memory
  persistence kernel and the generic H1 path may sum the diagonal costs in another order, so they get the 1e-6.
"""
import ctypes
import ctypes.util
import functools
import os
import re
import zlib

import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dilabhelmholtzoct_b200", "csrc")

F32 = np.float32
EPS24 = 2.0 ** -24
TINY = float(np.finfo(np.float32).tiny)
LAMDA = 0.1
REL_LOSS = 1e-6
REL_COST = 1e-6    # kernel cost against the reference for q not in {1, 2}
MARGIN = 1e-4      # unique optimum: every alternative dearer by this fraction of the optimal cost


# ------------------------------------------------------------------ constants of the kernels, read from the sources

def _const(fname, name):
    with open(os.path.join(CSRC, fname)) as f:
        text = f.read()
    m = re.search(rf"constexpr\s+(?:int|size_t)\s+{name}\s*=\s*([^;,]+)[;,]", text)
    assert m, f"{name} not found in {fname}: update the path model"
    expr = re.sub(r"(\d+)u\b", r"\1", m.group(1).strip())
    assert re.fullmatch(r"[\d\s*+\-()<]+", expr), expr
    return int(eval(expr))  # digits and + - * << ( ) only, checked above


K_SMALL_R = _const("match_small.cuh", "kSmallR")
K_COL_CACHE = _const("match_small.cuh", "kColCache")
K_HEAVY_SLOTS_MIN = _const("topoloss_api.cu", "kHeavySlotsMin")
K_MATCH_SLOTS = _const("topoloss_api.cu", "kMatchSlots")
K_HEAVY_BYTES = _const("topoloss_api.cu", "kHeavyBytes")
K_SMALL_SMEM = _const("ph_small.cuh", "kSmallSmemBytes")


def heavy_slots(S, feat_d):
    """CTAs of match_kernel over the heavy list for S x S maps (make_scratch in topoloss_api.cu)."""
    nn = S * S + 1 if feat_d == 1 else (S + 1) * (S + 1)
    cap = nn // 2 + 2
    stride_c = -(-(2 * cap + 2) // 32) * 32
    return min(max(K_HEAVY_BYTES // (29 * stride_c), K_HEAVY_SLOTS_MIN), K_MATCH_SLOTS)


# ------------------------------------------------------------------ path model

def path_of(n, m):
    """(branch, orientation) the matching of a map with n prediction and m ground-truth points takes."""
    R, Cn = min(n, m), max(n, m)
    orient = "swapped" if n < m else ("equal" if n == m else "rows_truth")
    if R == 0:
        return "R0", orient
    if R > K_SMALL_R:
        return "heavy", orient
    return ("cached" if Cn <= K_COL_CACHE else "uncached"), orient


def required_paths(feat_d):
    """Every feasible branch x orientation.  H0 diagrams always hold the essential class, so R0 needs H1; n == m
    never exceeds kColCache with R <= kSmallR."""
    req = {(b, o) for b in ("cached", "heavy") for o in ("swapped", "rows_truth", "equal")}
    req |= {("uncached", "swapped"), ("uncached", "rows_truth")}
    if feat_d == 1:
        req |= {("R0", o) for o in ("swapped", "rows_truth", "equal")}
    return req


# ------------------------------------------------------------------ maps with designed diagrams

BG1 = F32(0.5)   # H1 maps: background; a point (b, d) needs b <= BG1 < ... and b < d
BG0 = F32(0.0)   # H0 block maps: background, the essential class's birth
TOP0 = F32(1.0)  # H0 pit maps: plateau, every point's death


def _sites(S, step):
    """Feature centres off the border: every other pixel (step 2) or 3 x 3 blocks one pixel apart (step 4)."""
    c = np.arange(2, S - 2, 4) if step == 4 else np.arange(1, S - 1, 2)
    yy, xx = np.meshgrid(c, c, indexing="ij")
    return yy.ravel(), xx.ravel()


def h1_map(S, pts, rng):
    """H1 diagram = pts.  Points born at BG1 are single-pixel peaks on every other pixel; any other point is a
    3 x 3 block (ring = birth, centre = death) with background between blocks.  Nothing touches the border."""
    pts = np.asarray(pts, F32).reshape(-1, 2)
    assert np.all(pts[:, 0] <= BG1) and np.all(pts[:, 0] < pts[:, 1])
    f = np.full((S, S), BG1, F32)
    single = bool(np.all(pts[:, 0] == BG1))
    ys, xs = _sites(S, 2 if single else 4)
    assert len(pts) <= len(ys), (len(pts), len(ys))
    sel = np.sort(rng.choice(len(ys), len(pts), replace=False))
    for (y, x), (b, d) in zip(zip(ys[sel], xs[sel]), pts):
        if not single:
            f[y - 1:y + 2, x - 1:x + 2] = b
        f[y, x] = d
    return f


def h0_map(S, pts, rng):
    """H0 diagram = pts (essential class included).  All deaths TOP0: single-pixel pits in a TOP0 plateau (the
    eldest pit is the essential class, paired with argmax = TOP0).  Otherwise the first point must be the
    essential (BG0, max death) and the others are 3 x 3 blocks (centre = birth, ring = death) on a BG0 background."""
    pts = np.asarray(pts, F32).reshape(-1, 2)
    if np.all(pts[:, 1] == TOP0):
        f = np.full((S, S), TOP0, F32)
        ys, xs = _sites(S, 2)
        assert len(pts) <= len(ys) and np.all(pts[:, 0] < TOP0)
        sel = np.sort(rng.choice(len(ys), len(pts), replace=False))
        f[ys[sel], xs[sel]] = pts[:, 0]
        return f
    f = np.full((S, S), BG0, F32)
    ess, rest = pts[0], pts[1:]
    assert ess[0] == BG0 and ess[1] == max([BG0] + list(rest[:, 1])), (ess, rest)
    assert np.all(rest[:, 0] > BG0) and np.all(rest[:, 0] < rest[:, 1])
    ys, xs = _sites(S, 4)
    assert len(rest) <= len(ys)
    sel = np.sort(rng.choice(len(ys), len(rest), replace=False))
    for (y, x), (b, d) in zip(zip(ys[sel], xs[sel]), rest):
        f[y - 1:y + 2, x - 1:x + 2] = d
        f[y, x] = b
    return f


def _grid_anchors(rng, k, births, deaths):
    g = np.array([(b, d) for b in births for d in deaths if d > b + 0.05], np.float64)
    assert k <= len(g), (k, len(g))
    return g[rng.choice(len(g), k, replace=False)]


def _jit(rng, a, s=0.01):
    return a + rng.uniform(-s, s, a.shape)


def design_points(rng, feat_d, n, m, kind):
    """(prediction points, ground-truth points), n and m of them, for h1_map / h0_map.

    cont    tie-free: min(n, m) anchors well apart (L-inf >= 0.08) shared by both sides with independent
            jitter of 0.01, the rest of the larger side near the diagonal -- a unique optimum by a wide margin;
    dyadic  values on a 1/16 grid drawn from a small pool: exact ties and duplicated points on both sides;
    binary  every point equal (two-valued maps)."""
    dense = max(n, m) > 150
    if kind == "binary":
        p = (BG1, F32(1.0)) if feat_d == 1 else (F32(0.5), TOP0)
        return np.tile(np.array(p, F32), (n, 1)), np.tile(np.array(p, F32), (m, 1))
    if feat_d == 1:
        if kind == "dyadic":
            if dense:
                pool = [(0.5, 0.5 + j / 16) for j in range(1, 9)]
            else:
                pool = [(b / 16, b / 16 + j / 16) for b in (3, 5, 8) for j in (2, 3, 5)]
            pool = np.array(pool)
            return tuple(pool[rng.integers(0, len(pool), c)].astype(F32) for c in (n, m))
        k = min(n, m)
        if dense:
            anc = np.stack([np.full(k, 0.5), 0.5 + 0.1 * rng.choice(np.arange(2, 12), k, replace=False)], 1)
        else:
            anc = _grid_anchors(rng, k, [0.1, 0.2, 0.3, 0.4], 0.6 + 0.1 * np.arange(12))
        out = []
        for c in (n, m):
            a = _jit(rng, anc)
            if dense:
                a[:, 0] = 0.5
                extra = np.stack([np.full(c - k, 0.5), 0.5 + rng.uniform(0.002, 0.02, c - k)], 1)
            else:
                a[:, 0] = np.minimum(a[:, 0], 0.5)
                eb = rng.uniform(0.05, 0.45, c - k)
                extra = np.stack([eb, eb + rng.uniform(0.01, 0.03, c - k)], 1)
            out.append(rng.permutation(np.concatenate([a, extra])).astype(F32))
        return tuple(out)
    # H0
    if dense or kind == "dyadic" and max(n, m) > 40:
        if kind == "dyadic":
            return tuple(np.stack([rng.integers(0, 15, c) / 16, np.ones(c)], 1).astype(F32) for c in (n, m))
        k = min(n, m)
        anc = 1.0 - 0.1 * rng.choice(np.arange(1, 10), k, replace=False)
        out = []
        for c in (n, m):
            b = np.concatenate([_jit(rng, anc), 1.0 - rng.uniform(0.002, 0.02, c - k)])
            out.append(np.stack([rng.permutation(b), np.ones(c)], 1).astype(F32))
        return tuple(out)
    # H0 blocks: the essential (BG0, max death) first, then n - 1 / m - 1 pits
    if kind == "dyadic":
        pool = np.array([(b / 16, b / 16 + j / 16) for b in (2, 4, 7) for j in (2, 3, 5)])
        rest = [pool[rng.integers(0, len(pool), c - 1)] for c in (n, m)]
    else:
        k = min(n, m) - 1
        anc = _grid_anchors(rng, k, [0.1, 0.2, 0.3, 0.4, 0.5], 0.7 + 0.1 * np.arange(12))
        rest = []
        for c in (n, m):
            eb = rng.uniform(0.05, 0.45, c - 1 - k)
            rest.append(rng.permutation(np.concatenate([_jit(rng, anc), np.stack([eb, eb + rng.uniform(0.01, 0.03, c - 1 - k)], 1)])))
    out = []
    for r in rest:
        r = r.astype(F32)
        out.append(np.concatenate([np.array([[BG0, max([BG0] + list(r[:, 1]))]], F32), r]))
    return tuple(out)


def build_map(S, feat_d, pts, rng):
    return h1_map(S, pts, rng) if feat_d == 1 else h0_map(S, pts, rng)


# ------------------------------------------------------------------ the float64 reference

_LIBM = ctypes.CDLL(ctypes.util.find_library("m"))
_LIBM.powf.argtypes, _LIBM.powf.restype = [ctypes.c_float, ctypes.c_float], ctypes.c_float
_POWF = np.frompyfunc(lambda x, q: _LIBM.powf(float(x), q), 2, 1)


def powq32(x, q):
    """tl_common.cuh powq in fp32: x * x for q = 2, else the C library's powf (numpy's float32 power is not powf)."""
    x = np.asarray(x, F32)
    if q == 2:
        return x * x
    if q == 1:
        return x.copy()
    return _POWF(x, float(q)).astype(F32)


def diag_cost(D, q, exact=False):
    """cost_diag of each point: fp32 L-inf to the diagonal, then powq (``exact``: the power in float64)."""
    D = np.asarray(D, F32).reshape(-1, 2)
    h = F32(0.5) * (D[:, 0] + D[:, 1])
    x = np.maximum(np.abs(D[:, 0] - h), np.abs(D[:, 1] - h))
    return x.astype(np.float64) ** q if exact else powq32(x, q).astype(np.float64)


def pair_cost(A, B, q, exact=False):
    """cost_pp of every (A[i], B[j])."""
    A = np.asarray(A, F32).reshape(-1, 2)
    B = np.asarray(B, F32).reshape(-1, 2)
    x = np.maximum(np.abs(A[:, None, 0] - B[None, :, 0]), np.abs(A[:, None, 1] - B[None, :, 1]))
    return x.astype(np.float64) ** q if exact else powq32(x, q).astype(np.float64)


def _square_lsa(Rp, Cp, q, exact, forbid):
    """Optimum of torch_topological's emd2 LP between Rp and Cp in its square assignment form: rows = Rp's points
    then one diagonal slot per Cp point, columns = Cp's points then one diagonal slot per Rp point.  A point may only
    use its own diagonal slot; diagonal slots pair at cost 0.  ``forbid``: (row, col or -1 for its diagonal)."""
    R, K = len(Rp), len(Cp)
    M = np.full((R + K, K + R), np.inf)
    M[:R, :K] = pair_cost(Rp, Cp, q, exact)
    M[np.arange(R), K + np.arange(R)] = diag_cost(Rp, q, exact)
    M[R + np.arange(K), np.arange(K)] = diag_cost(Cp, q, exact)
    M[R:, K:] = 0.0
    for r, k in forbid:
        M[r, K + r if k < 0 else k] = np.inf
    ri, ci = linear_sum_assignment(M)
    return float(M[ri, ci].sum())


def lsa_optimum(A, B, q, exact=False, forbid=(), reduce=True):
    """Optimal cost between prediction diagram A and ground truth B.  The smaller diagram is the rows; ``forbid``
    names (row, column or -1) in that orientation.  ``reduce`` keeps only each row's R cheapest columns by
    c(r, k) - diag(k) (exact, see the module docstring)."""
    A = np.asarray(A, F32).reshape(-1, 2)
    B = np.asarray(B, F32).reshape(-1, 2)
    Rp, Cp = (A, B) if len(A) < len(B) else (B, A)
    R, K = len(Rp), len(Cp)
    dc = diag_cost(Cp, q, exact)
    if R == 0:
        return float(dc.sum())
    keep = np.arange(K)
    if reduce and K > R:
        red = pair_cost(Rp, Cp, q, exact) - dc[None, :]
        for r, k in forbid:
            if k >= 0:
                red[r, k] = np.inf
        keep = np.unique(np.concatenate([np.argpartition(red[r], R - 1)[:R] for r in range(R)]))
    where = {int(k): i for i, k in enumerate(keep)}
    fb = [(r, where[k] if k >= 0 else -1) for r, k in forbid if k < 0 or k in where]
    dropped = np.ones(K, bool)
    dropped[keep] = False
    return _square_lsa(Rp, Cp[keep], q, exact, fb) + float(dc[dropped].sum())


def same_cost(a, b, A, B, q):
    """Two fp64 sums of the same fp32 entries, summed in different orders: equal to 1e-12 of the magnitude summed
    (every diagonal entry plus the optimum bounds it: a matched entry never exceeds its two diagonal entries)."""
    scale = diag_cost(A, q).sum() + diag_cost(B, q).sum() + abs(b)
    return abs(a - b) <= 1e-12 * max(scale, 1e-300)


def kernel_order(P, feat_d):
    """Order of the records the persistence kernels emit: raster order of the dying basin."""
    return np.argsort(P[:, 1] if feat_d == 1 else P[:, 0], kind="stable")


def unique_margin(A, B, q):
    """(second best - best) / best over assignments, float64 entries: each row's choice in the optimum is
    forbidden in turn.  Every other assignment changes some row's choice, so this bounds them all."""
    _, match = oracle.wasserstein(A, B, q)
    swp = len(A) < len(B)
    R = min(len(A), len(B))
    if R == 0:
        return np.inf
    if swp:
        choice = list(match)
    else:
        choice = [-1] * len(B)
        for i, j in enumerate(match):
            if j >= 0:
                choice[j] = i
    best = lsa_optimum(A, B, q, exact=True)
    alt = min(lsa_optimum(A, B, q, exact=True, forbid=[(r, int(choice[r]))]) for r in range(R))
    return (alt - best) / best


def map_reference(fp, ft, feat_d, q):
    """Diagrams in the kernels' order, the oracle's assignment and the optimal cost (checked against the LSA)."""
    P, T = oracle.cubical_pairs(fp, feat_d), oracle.cubical_pairs(ft, feat_d)
    P, T = P[kernel_order(P, feat_d)], T[kernel_order(T, feat_d)]
    A, B = fp.ravel()[P], ft.ravel()[T]
    cost, match = oracle.wasserstein(A, B, q)
    opt = lsa_optimum(A, B, q)
    assert same_cost(cost, opt, A, B, q), (cost, opt, len(A), len(B))
    return P, T, A, B, match, opt


def point_terms(A, B, match, q):
    """d cost / d (birth, death) of each prediction point (pair_gradient before the coefficient), float64."""
    A = A.astype(F32)
    gb = np.zeros(len(A))
    gd = np.zeros(len(A))
    for i, (b, d) in enumerate(A):
        j = match[i]
        if j < 0:
            h = F32(0.5) * (b + d)
            x = max(abs(b - h), abs(d - h))
            gg = q * float(x) ** (q - 1.0) if x > 0 else (1.0 if q == 1 else 0.0)
            s = 1.0 if d > b else (-1.0 if d < b else 0.0)
            gb[i], gd[i] = -0.5 * gg * s, 0.5 * gg * s
        else:
            xb, xd = b - B[j, 0], d - B[j, 1]
            ab, ad = abs(xb), abs(xd)
            dist = max(ab, ad)
            gg = q * float(dist) ** (q - 1.0) if dist > 0 else 0.0
            gb[i] = gg * np.sign(xb) if ab == dist else 0.0
            gd[i] = gg * np.sign(xd) if ad == dist else 0.0
    return gb, gd


def case_reference(pred, truth, feat_d, q, loss_r):
    """Loss, per-pixel gradient, per-pixel sum |terms| and term count of topo_loss (float64), per map (n, m, cost),
    and the per-pixel sum of |coefficient part| of the terms (the part proportional to S_b^(1/q - 1), before the
    loss_r term is subtracted: with loss_r the two may cancel inside one term)."""
    Bn, C, H, W = pred.shape
    lam = float(F32(LAMDA))  # the kernels take lamda as fp32
    maps = [map_reference(pred[b, c], truth[b, c], feat_d, q) for b in range(Bn) for c in range(C)]
    cost = np.array([r[5] for r in maps])
    S = []
    for b in range(Bn):
        s = F32(0)
        for c in range(C):
            s = F32(s + F32(cost[b * C + c]))
        S.append(s)
    Wb = [np.sqrt(s) if q == 2 else np.power(s, F32(1) / F32(q)) for s in S]
    acc = float(np.sum([float(w) for w in Wb])) / Bn
    grad = np.zeros(pred.size)
    absd = np.zeros(pred.size)
    absc = np.zeros(pred.size)
    cnt = np.zeros(pred.size, np.int64)
    reg = 0.0
    creg = lam / (Bn * C)
    for k, (P, T, A, B, match, _) in enumerate(maps):
        b = k // C
        coef = lam / Bn * (1.0 / q) * float(S[b]) ** (1.0 / q - 1.0) if S[b] > 0 else np.nan
        gb, gd = point_terms(A, B, match, q)
        gb, gd = gb * coef, gd * coef
        cb, cd = np.abs(gb), np.abs(gd)
        pers = A[:, 1].astype(np.float64) - A[:, 0].astype(np.float64)
        if loss_r:
            reg += float(np.sum(np.abs(pers) ** q))
            gr = np.where(pers != 0, q * np.abs(pers) ** (q - 1.0) * np.sign(pers) * creg, 0.0)
            gb, gd = gb - gr, gd + gr
        base = k * H * W
        for idx, t, tc in ((P[:, 0], gb, cb), (P[:, 1], gd, cd)):
            np.add.at(grad, base + idx, t)
            np.add.at(absd, base + idx, np.abs(t))
            np.add.at(absc, base + idx, tc)
            np.add.at(cnt, base + idx, 1)
    loss = acc + (reg / (Bn * C) if loss_r else 0.0)
    loss = float(F32(lam * loss))
    counts = [(len(r[0]), len(r[1]), r[5]) for r in maps]
    return (loss, grad.reshape(pred.shape), absd.reshape(pred.shape), cnt.reshape(pred.shape), counts,
            absc.reshape(pred.shape))


# ------------------------------------------------------------------ the cases

KC = K_COL_CACHE
SMALL_H1 = [[(0, 0), (1, 7), (9, 40), (0, 5)], [(5, 0), (7, 1), (40, 9), (1, 1)],
            [(8, 8), (8, 40), (40, 8), (9, 9)], [(12, 20), (20, 12), (8, 9), (9, 8)]]
SMALL_H0 = [[(1, 7), (9, 40), (7, 1), (1, 1)], [(8, 8), (8, 40), (40, 8), (9, 9)],
            [(12, 20), (20, 12), (8, 9), (9, 8)]]
# one image mixes all four branches (the tail scheduler's per-image bookkeeping); kColCache on both sides of it
LARGE_H1 = [[(3, KC + 1), (0, 5), (5, 7), (12, 20)], [(KC + 1, 3), (KC, 3), (3, KC), (8, 8)]]
LARGE_H0 = [[(3, KC + 1), (7, 5), (5, 7), (12, 20)], [(KC + 1, 3), (KC, 3), (3, KC), (8, 8)]]
N_HEAVY = K_HEAVY_SLOTS_MIN + 2
# (name, feat_d, q, S, kind, images, loss_r values, exact assignment, two-valued)
CASES = [
    ("branches_h1", 1, 2.0, 64, "cont", SMALL_H1, (False, True), True, False),
    ("branches_h0", 0, 2.0, 64, "cont", SMALL_H0, (False, True), True, False),
    ("branches_large_h1", 1, 2.0, 224, "cont", LARGE_H1, (False, True), True, False),
    ("branches_large_h0", 0, 2.0, 224, "cont", LARGE_H0, (False, True), True, False),
    ("ties_q1_h1", 1, 1.0, 64, "dyadic", [[(6, 4), (4, 6), (5, 5), (12, 30)], [(30, 12), (8, 8), (3, 9), (9, 3)]], (False,), True, False),
    ("ties_q2_h1", 1, 2.0, 64, "dyadic", [[(6, 4), (4, 6), (5, 5), (12, 30)], [(30, 12), (8, 8), (3, 9), (9, 3)]], (False,), True, False),
    ("ties_q1_h0", 0, 1.0, 64, "dyadic", [[(6, 4), (4, 6), (5, 5), (12, 30)], [(30, 12), (8, 8), (3, 9), (9, 3)]], (False,), True, False),
    ("ties_q2_h0", 0, 2.0, 64, "dyadic", [[(6, 4), (4, 6), (5, 5), (12, 30)], [(30, 12), (8, 8), (3, 9), (9, 3)]], (False,), True, False),
    ("ties_large_q1_h1", 1, 1.0, 224, "dyadic", [[(4, KC + 1), (6, 9)], [(KC + 1, 4), (9, 6)]], (False,), True, False),
    ("ties_large_q2_h1", 1, 2.0, 224, "dyadic", [[(4, KC + 1), (6, 9)], [(KC + 1, 4), (9, 6)]], (False,), True, False),
    ("q3", 1, 3.0, 64, "cont", [[(0, 5), (3, 6), (10, 14)], [(5, 0), (6, 3), (14, 10)]], (False, True), False, False),
    ("q3_h0", 0, 3.0, 64, "cont", [[(3, 6), (10, 14)], [(6, 3), (14, 10)]], (False,), False, False),
    ("q1.5", 1, 1.5, 64, "cont", [[(0, 5), (3, 6), (10, 14)], [(5, 0), (6, 3), (14, 10)]], (False, True), False, False),
    ("q1.5_h0", 0, 1.5, 64, "cont", [[(3, 6), (10, 14)], [(6, 3), (14, 10)]], (False,), False, False),
    ("q3_large", 1, 3.0, 224, "cont", [[(3, KC + 1)], [(2, 9)]], (False,), False, False),
    ("q1.5_large", 1, 1.5, 224, "cont", [[(KC + 1, 3)], [(9, 2)]], (False,), False, False),
    ("heavy_slots_swapped", 1, 2.0, 256, "cont",
     [[(9 + i % 8, 20 + i) for i in range(N_HEAVY)], [(9 + i % 5, 12 + i) for i in range(N_HEAVY)]], (False,), True, False),
]
BINARY = {  # prediction == ground truth except class 2 (image 0: more points, 1: fewer, 2: both > kSmallR)
    "binary_h1": 1, "binary_h0": 0,
}
BINARY_COUNTS = [[(5, 5), (3, 3), (9, 6)], [(4, 4), (7, 7), (2, 6)], [(6, 6), (1, 1), (20, 12)]]
for _name, _fd in BINARY.items():
    for _q in (1.0, 2.0):
        CASES.append((f"{_name}_q{int(_q)}", _fd, _q, 64, "binary", BINARY_COUNTS, (False, True), True, _fd == 1))
CASE_BY_NAME = {c[0]: c for c in CASES}


@functools.lru_cache(maxsize=None)
def case_maps(name):
    """pred, truth [B, C, S, S] of one case; every diagram checked against oracle.cubical_pairs."""
    _, feat_d, q, S, kind, images, _, _, _ = CASE_BY_NAME[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    C = len(images[0])
    pred = np.zeros((len(images), C, S, S), F32)
    truth = np.zeros_like(pred)
    for b, img in enumerate(images):
        for c, (n, m) in enumerate(img):
            P, T = design_points(rng, feat_d, n, m, kind)
            if kind == "binary" and n == m:  # the same map on both sides
                pred[b, c] = truth[b, c] = build_map(S, feat_d, P, rng)
            else:
                pred[b, c] = build_map(S, feat_d, P, rng)
                truth[b, c] = build_map(S, feat_d, T, rng)
            for f, want in ((pred[b, c], P), (truth[b, c], T)):
                got = f.ravel()[oracle.cubical_pairs(f, feat_d)]
                assert len(got) == len(want), (name, b, c, len(got), len(want))
                assert np.array_equal(got[np.lexsort(got.T[::-1])], want[np.lexsort(want.T[::-1])]), (name, b, c)
    return pred, truth


@functools.lru_cache(maxsize=None)
def case_ref(name, loss_r):
    _, feat_d, q, _, _, _, _, exact, _ = CASE_BY_NAME[name]
    pred, truth = case_maps(name)
    ref = case_reference(pred, truth, feat_d, q, loss_r)
    if not exact and not loss_r:  # unique optimum with float64 entries (module docstring)
        for b in range(pred.shape[0]):
            for c in range(pred.shape[1]):
                fp, ft = pred[b, c], truth[b, c]
                A = fp.ravel()[oracle.cubical_pairs(fp, feat_d)]
                Bd = ft.ravel()[oracle.cubical_pairs(ft, feat_d)]
                mg = unique_margin(A, Bd, q)
                assert mg > MARGIN, (name, b, c, mg)
    return ref


# ------------------------------------------------------------------ CPU tests

def test_constants_are_read_from_the_sources():
    assert 1 <= K_SMALL_R < 64 and K_COL_CACHE > K_SMALL_R and K_HEAVY_SLOTS_MIN >= 1 and K_MATCH_SLOTS >= K_HEAVY_SLOTS_MIN
    # the tail hands the persistence kernel's dynamic shared memory to match_one_map as its column cache
    assert K_SMALL_SMEM >= K_COL_CACHE * 8
    with open(os.path.join(CSRC, "ph_small.cuh")) as f:
        assert re.search(r"static_assert\(kSmallSmemBytes >= kColCache \* sizeof\(float2\)", f.read())
    with open(os.path.join(CSRC, "topoloss_api.cu")) as f:
        src = f.read()
    assert re.search(r"match_small_kernel<<<[^>]*tl::kColCache \* 8", src), "match_small_kernel's column cache changed"
    # the case with more heavy maps than match_kernel has CTAs needs a map size where the slots hit their floor
    assert heavy_slots(256, 1) < N_HEAVY * 2 and heavy_slots(256, 1) <= K_HEAVY_SLOTS_MIN + 1


@pytest.mark.parametrize("feat_d", [0, 1])
def test_gpu_cases_reach_every_path(feat_d):
    reached = {}
    for name, fd, q, S, kind, images, _, _, _ in CASES:
        if fd != feat_d:
            continue
        for img in images:
            for n, m in img:
                reached.setdefault(path_of(n, m), set()).add(name)
    main = {p for p, names in reached.items() if names & {f"branches_h{feat_d}", f"branches_large_h{feat_d}"}}
    assert required_paths(feat_d) <= main, sorted(required_paths(feat_d) - main)
    ties = {p[0] for p, names in reached.items() if any(n.startswith(("ties", "binary")) for n in names)}
    assert {"cached", "heavy"} <= ties and (feat_d == 0 or "uncached" in ties)
    # every branch at q = 3 and q = 1.5 (R0 needs H1)
    for q in (3.0, 1.5):
        got = set()
        for name, fd, qq, *_ in CASES:
            if qq == q:
                got |= {path_of(n, m)[0] for img in CASE_BY_NAME[name][5] for n, m in img}
        assert got >= {"R0", "cached", "uncached", "heavy"}, (q, got)
    # one image with more heavy maps than match_kernel's CTAs, swapped; one image that mixes all branches
    hv = CASE_BY_NAME["heavy_slots_swapped"]
    assert all(path_of(n, m) == ("heavy", "swapped") for n, m in hv[5][0])
    assert sum(1 for img in hv[5] for _ in img) > heavy_slots(hv[3], hv[1]) and len(hv[5][0]) > K_HEAVY_SLOTS_MIN
    assert {path_of(n, m)[0] for n, m in LARGE_H1[0]} == {"R0", "cached", "uncached", "heavy"}


def _random_diagrams(rng, n, m, levels):
    out = []
    for c in (n, m):
        if levels:
            b = rng.integers(0, levels, c) / levels
            d = b + rng.integers(1, levels, c) / levels
        else:
            b = rng.random(c)
            d = b + rng.random(c)
        out.append(np.stack([b, d], 1).astype(F32))
    return out


@pytest.mark.parametrize("q", [1.0, 2.0, 3.0, 1.5])
def test_oracle_assignment_is_optimal_under_lsa(q):
    """The oracle's Hungarian solver against scipy's LSA on the full square problem: tie-heavy and continuous
    diagrams, both orientations, empty sides."""
    rng = np.random.default_rng(int(q * 10))
    for t in range(60):
        n, m = int(rng.integers(0, 25)), int(rng.integers(0, 25))
        A, B = _random_diagrams(rng, n, m, (0, 3, 5, 8)[t % 4])
        if t % 5 == 0:  # duplicated points on both sides
            A = np.concatenate([A, A[: n // 2], B[: m // 3]]).astype(F32)
        cost, match = oracle.wasserstein(A, B, q)
        opt = lsa_optimum(A, B, q, reduce=False)
        assert same_cost(cost, opt, A, B, q), (t, cost, opt)
        # the matching the oracle reports has that cost
        dA, dB = diag_cost(A, q), diag_cost(B, q)
        used = match[match >= 0]
        assert len(set(used.tolist())) == len(used)
        direct = sum(pair_cost(A[i], B[j], q)[0, 0] if j >= 0 else dA[i] for i, j in enumerate(match))
        direct += dB[np.setdiff1d(np.arange(len(B)), used)].sum()
        assert same_cost(direct, opt, A, B, q)


@pytest.mark.parametrize("q", [1.0, 2.0, 3.0])
def test_reduction_matches_full_problem(q):
    """Keeping only each row's R cheapest columns leaves the optimum unchanged, with and without forbidden entries."""
    rng = np.random.default_rng(70 + int(q))
    for t in range(30):
        R = int(rng.integers(1, K_SMALL_R + 2))
        K = int(rng.integers(R + 1, 300))
        A, B = _random_diagrams(rng, R, K, (0, 4, 16)[t % 3])
        if t % 2:
            A, B = B, A
        full = lsa_optimum(A, B, q, reduce=False)
        red = lsa_optimum(A, B, q)
        assert same_cost(full, red, A, B, q), (t, full, red)
        fb = [(int(rng.integers(0, R)), int(rng.integers(-1, K)))]
        assert same_cost(lsa_optimum(A, B, q, forbid=fb, reduce=False), lsa_optimum(A, B, q, forbid=fb), A, B, q)


def test_builders_and_references():
    """Every case's maps have their designed diagrams; the reference's cost is the LSA optimum; q not in {1, 2}
    cases have a unique optimum; two-valued predictions are two-valued."""
    for name, feat_d, q, S, kind, images, loss_rs, exact, binary in CASES:
        pred, truth = case_maps(name)
        loss, grad, absd, cnt, counts, absc = case_ref(name, False)
        assert [(n, m) for n, m, _ in counts] == [nm for img in images for nm in img], name
        assert np.isfinite(loss) and np.all(np.isfinite(grad)), name
        assert np.all((absd > 0) <= (cnt > 0)) and np.all((absc > 0) <= (cnt > 0))
        if kind == "binary":
            assert all(len(np.unique(pred[b, c])) == 2 for b in range(pred.shape[0]) for c in range(pred.shape[1]))


# ------------------------------------------------------------------ GPU tests

ROUTES = {"fused": (), "no_fused_grad": ("OPT_NO_FUSED_GRAD",), "no_fused_match": ("OPT_NO_FUSED_MATCH",),
          "global": ("OPT_FORCE_GLOBAL_KERNEL",)}
BIT_IDENTICAL = ("fused", "no_fused_grad", "no_fused_match")


def _run(pred, truth, feat_d, q, loss_r, opts):
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    ids = [getattr(_lib, o) for o in opts]
    old = [L.tl_get_option(i) for i in ids]
    for i in ids:
        assert L.tl_set_option(i, 1) == 0
    try:
        p = torch.as_tensor(pred).cuda().requires_grad_(True)
        loss = tlb.topo_loss(p, torch.as_tensor(truth).cuda(), LAMDA, feat_d=feat_d, loss_q=q, loss_r=loss_r)
        loss.backward()
        torch.cuda.synchronize()
        tlb.check_status()
        return float(loss.detach()), p.grad.cpu().numpy().astype(np.float64)
    finally:
        for i, v in zip(ids, old):
            L.tl_set_option(i, v)


def _check_grad(got, ref, absd, absc, cnt, q, exact, what):
    bound = (cnt + 1) * EPS24 * absd + TINY
    if q not in (1.0, 2.0):  # the coefficient's uncertainty scales its own part of each term, not the sum with loss_r's
        bound += abs(1.0 / q - 1.0) * REL_COST * absc
    bad = np.abs(got - ref) > bound
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:5].tolist(), got[bad][:5], ref[bad][:5])
    assert np.all(got[absd == 0] == 0), what
    if exact:
        sel = (absd == 0) | (np.abs(ref) > bound)
        assert np.array_equal((got != 0)[sel], (ref != 0)[sel]), what


def _case_params():
    out = []
    for name, feat_d, q, S, kind, images, loss_rs, exact, binary in CASES:
        for loss_r in loss_rs:
            out.append(pytest.param(name, loss_r, id=f"{name}-r{int(loss_r)}"))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,loss_r", _case_params())
def test_loss_matching_routes(name, loss_r):
    _, feat_d, q, S, kind, images, _, exact, binary = CASE_BY_NAME[name]
    pred, truth = case_maps(name)
    want, ref, absd, cnt, counts, absc = case_ref(name, loss_r)
    routes = dict(ROUTES)
    if binary:
        routes["no_binary"] = ("OPT_NO_BINARY_PATH",)
    losses = {}
    for route, opts in routes.items():
        got, grad = _run(pred, truth, feat_d, q, loss_r, opts)
        losses[route] = got
        assert abs(got - want) <= REL_LOSS * abs(want), (name, route, got, want)
        _check_grad(grad, ref, absd, absc, cnt, q, exact, (name, route))
    assert len({losses[r] for r in BIT_IDENTICAL}) == 1, losses


@pytest.mark.gpu
def test_q1_cost_entries_are_exact():
    """q = 1: the device's powf(x, 1.0f) returns x, so the cost entries are bit-reproducible on the host.  One
    H1 point per map against an empty ground truth: the cost is one diagonal entry and the loss is exact."""
    rng = np.random.default_rng(5)
    deaths = np.array([[0.8137], [0.6071], [0.9533]], F32)
    pred = np.stack([h1_map(16, [(BG1, d[0])], rng) for d in deaths])[:, None]
    truth = np.full_like(pred, BG1)
    got, _ = _run(pred, truth, 1, 1.0, False, ())
    x = diag_cost(np.stack([np.full(3, BG1), deaths[:, 0]], 1), 1.0)
    want = float(F32(float(F32(LAMDA)) * (np.sum([float(F32(v)) for v in x]) / 3)))
    assert got == want, (got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ties_q1_h1", "ties_q2_h1", "ties_q1_h0", "binary_h1_q2", "q3", "q1.5_h0"])
def test_wasserstein_distance_matches_reference(name):
    """wasserstein_distance (match_kernel on every map) on the tie and swapped cases, diagrams in gudhi's order:
    value and gradient with respect to both diagrams."""
    import dilabhelmholtzoct_b200 as tlb
    _, feat_d, q, *_ = CASE_BY_NAME[name]
    pred, truth = case_maps(name)
    fp, ft = pred.reshape(-1, *pred.shape[2:]), truth.reshape(-1, *truth.shape[2:])
    Ps = [oracle.cubical_pairs(f, feat_d) for f in fp]
    Ts = [oracle.cubical_pairs(f, feat_d) for f in ft]
    As = [f.ravel()[P] for f, P in zip(fp, Ps)]
    Bs = [f.ravel()[T] for f, T in zip(ft, Ts)]

    def diagrams(pairs, pts):
        off = np.concatenate([[0], np.cumsum([len(p) for p in pairs])]).astype(np.int32)
        d = torch.as_tensor(np.concatenate(pts).reshape(-1, 2)).cuda().requires_grad_(True)
        pr = torch.as_tensor(np.concatenate(pairs).reshape(-1, 2)).cuda()
        return tlb.Diagrams(pr, d, torch.as_tensor(off).cuda(), off.tolist()), off

    D1, o1 = diagrams(Ps, As)
    D2, o2 = diagrams(Ts, Bs)
    w = torch.linspace(0.5, 2.0, len(fp), device="cuda")
    cost = tlb.wasserstein_distance(D1, D2, q)
    (cost * w).sum().backward()
    torch.cuda.synchronize()
    got = cost.detach().cpu().numpy().astype(np.float64)
    g1, g2 = D1.diagram.grad.cpu().numpy().astype(np.float64), D2.diagram.grad.cpu().numpy().astype(np.float64)
    wc = w.cpu().numpy().astype(np.float64)
    exact = q in (1.0, 2.0)
    for k, (A, B) in enumerate(zip(As, Bs)):
        want, match = oracle.wasserstein(A, B, q)
        opt = lsa_optimum(A, B, q)
        assert same_cost(want, opt, A, B, q)
        # one fp32 rounding of the fp64 optimum (q in {1, 2}) or the device powf (otherwise), plus the fp64 sum's
        # own order, which scales with the diagonal costs summed (see same_cost)
        scale = diag_cost(A, q).sum() + diag_cost(B, q).sum() + abs(opt)
        tol = (2 * EPS24 if exact else REL_COST) * abs(opt) + 1e-12 * scale
        assert abs(got[k] - opt) <= tol, (name, k, got[k], opt)
        gb, gd = point_terms(A, B, match, q)
        r1 = np.stack([gb, gd], 1) * float(F32(wc[k]))
        r2 = np.zeros((len(B), 2))
        for j in range(len(B)):  # ground-truth points: the diagonal term, or minus their match's
            h = F32(0.5) * (B[j, 0] + B[j, 1])
            x = max(abs(B[j, 0] - h), abs(B[j, 1] - h))
            gg = q * float(x) ** (q - 1.0) if x > 0 else (1.0 if q == 1 else 0.0)
            s = 1.0 if B[j, 1] > B[j, 0] else (-1.0 if B[j, 1] < B[j, 0] else 0.0)
            r2[j] = (-0.5 * gg * s, 0.5 * gg * s)
        for i, j in enumerate(match):
            if j >= 0:
                r2[j] = -np.array([gb[i], gd[i]])
        r2 *= float(F32(wc[k]))
        for got_g, ref_g in ((g1[o1[k]:o1[k + 1]], r1), (g2[o2[k]:o2[k + 1]], r2)):
            bound = 2 * EPS24 * np.abs(ref_g) + TINY
            assert np.all(np.abs(got_g - ref_g) <= bound), (name, k, got_g, ref_g)
            if exact:
                assert np.array_equal(got_g != 0, ref_g != 0), (name, k)
