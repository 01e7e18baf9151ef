"""Oracles for the Betti matching loss -- TEST INFRASTRUCTURE ONLY (the product package never imports this).

* ``image_pairs_literal`` / ``betti_matching_literal``: image persistence by a literal Z/2 reduction of the boundary
  matrix of the cubical complex of ``oracle.oracle_literal`` (same cells, cell order and pixel rules), and the Betti
  matching assembled from it;
* ``betti_matching``: the union-find restatement in ``tests/betti_oracle.c`` (fast enough for 256 x 256 maps), built
  on first use into the system's temporary directory with the compiler ``oracle/Makefile`` uses.

Parity with the upstream Betti-Matching-3D package is unpinned: it is not available here, and whether its cubical
complex follows the same convention is not verified.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.oracle_literal import _cells, _pixel_of, _top_cell

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "betti_oracle.c")
_DEPS = [_SRC, os.path.join(os.path.dirname(_HERE), "oracle", "topo_oracle.c")]
_LIB = None
# ---------------------------------------------------------------- image persistence and Betti matching
#
# Image persistence of H_d(F_t) -> H_d(G_t) for two filtrations of the same complex with f >= g cellwise (so that
# F_t is a subcomplex of G_t for every t), per Cohen-Steiner, Edelsbrunner, Harer and Morozov ("Persistent homology
# for kernels, images, and cokernels", SODA 2009) and Bauer and Schmahl ("Efficient computation of image
# persistence", SoCG 2023): reduce the boundary matrix with its COLUMNS in g's cell order and the lowest non-zero
# of each column taken in f's cell order.  A pivot (sigma, tau) is the image interval [f(sigma), g(tau)): sigma is a
# birth cell of the domain filtration, tau a death cell of the codomain one.  Intervals with f(sigma) >= g(tau) are
# empty and dropped.  With f == g this is the ordinary reduction of cubical_pairs_literal.

def _boundary(p: int, GW: int):
    Y, X = divmod(p, GW)
    out = []
    if X & 1:
        out += [p - 1, p + 1]
    if Y & 1:
        out += [p - GW, p + GW]
    return out


def _image_reduction(f: np.ndarray, g: np.ndarray):
    """Pivots ``(sigma, tau)`` (bitmap positions) of the image reduction, in g's order of tau, and the cells that
    are lowest in no column.  Also returns the two value grids and the cell dimensions."""
    valf, GH, GW = _cells(f)
    valg = _cells(g)[0]
    ncell = GH * GW
    Ys, Xs = np.divmod(np.arange(ncell), GW)
    dims = (Ys % 2) + (Xs % 2)
    vf, vg = valf.ravel(), valg.ravel()
    order_f = sorted(range(ncell), key=lambda p: (vf[p], dims[p], p))
    order_g = sorted(range(ncell), key=lambda p: (vg[p], dims[p], p))
    rank_f = np.empty(ncell, dtype=np.int64)
    for i, p in enumerate(order_f):
        rank_f[p] = i
    low_to_col, columns, pivots = {}, {}, []
    for tau in order_g:
        col = set(int(rank_f[q]) for q in _boundary(tau, GW))
        while col:
            j = low_to_col.get(max(col))
            if j is None:
                break
            col ^= columns[j]
        if col:
            lo = max(col)
            low_to_col[lo] = tau
            columns[tau] = col
            pivots.append((order_f[lo], tau))
    unpaired_rows = [order_f[i] for i in range(ncell) if i not in low_to_col]
    return pivots, unpaired_rows, valf, valg, dims, GH, GW


def image_pairs_literal(f, g, dim: int):
    """Image barcode of ``H_dim({f <= t}) -> H_dim({g <= t})`` for HxW maps with ``f >= g`` pixelwise.

    Returns ``(pairs, essential)``: ``pairs`` lists ``(birth_cell, death_cell, birth_pixel, death_pixel)`` of every
    non-empty interval ``[f(birth_cell), g(death_cell))``, in g's filtration order of the death cell (cells are
    bitmap positions in the (2H+1)x(2W+1) grid; pixels are chosen by gudhi's coface walk, the birth pixel in f and
    the death pixel in g).  ``essential`` is ``(birth_cell, birth_pixel)`` of the one infinite H0 interval, or
    ``None`` for ``dim == 1``.  ``image_pairs_literal(f, f, d)`` is ``cubical_pairs_literal(f)``'s barcode."""
    f = np.asarray(f)
    g = np.asarray(g)
    assert f.ndim == 2 and f.shape == g.shape and bool(np.all(f >= g))
    H, W = f.shape
    pivots, unpaired, valf, valg, dims, GH, GW = _image_reduction(f, g)
    vf, vg = valf.ravel(), valg.ravel()
    out = []
    for s, t in pivots:
        if dims[s] != dim or not (vf[s] < vg[t]):
            continue
        out.append((int(s), int(t), _pixel_of(_top_cell(s, valf, GH, GW), GW, W),
                    _pixel_of(_top_cell(t, valg, GH, GW), GW, W)))
    ess = None
    if dim == 0:
        # f-positive cells paired in no column: the one component of the filled rectangle (no H1 survives in g)
        vert = [p for p in unpaired if dims[p] == 0 and p not in {t for _, t in pivots}]
        assert len(vert) == 1, vert
        ess = (int(vert[0]), _pixel_of(_top_cell(vert[0], valf, GH, GW), GW, W))
    return out, ess


def betti_matching_literal(L, G, dim: int):
    """Betti matching of a prediction map ``L`` and a target map ``G`` (Stucki et al., ICML 2023) in homology
    dimension ``dim``, assembled from ``image_pairs_literal``.  With ``C = min(L, G)``:

    * the barcodes of L and G are the image barcodes of L -> L and G -> G;
    * an interval of L and one of G are matched when the image intervals of L -> C and G -> C born at their birth
      cells die at the same cell of C; the two essential H0 classes are always matched; the rest are unmatched.

    Returns a dict: ``matched`` int32 ``[M, 4]`` (pred creator, pred destroyer, target creator, target destroyer
    pixel), ``unmatched_pred`` / ``unmatched_target`` int32 ``[K, 2]``, and ``cost`` (float64) =
    sum over matched of (b_L - b_G)^2 + (d_L - d_G)^2 plus, per unmatched interval, (d - b)^2 / 2.
    Order: intervals by the bitmap position of their birth vertex (H0) or death square (H1) -- the cell that owns
    the interval in the pixel-graph merge tree; the H0 essential pair is the last matched row."""
    L = np.asarray(L, dtype=np.float32)
    G = np.asarray(G, dtype=np.float32)
    C = np.minimum(L, G)
    bar_l, ess_l = image_pairs_literal(L, L, dim)
    bar_g, ess_g = image_pairs_literal(G, G, dim)
    img_l, _ = image_pairs_literal(L, C, dim)
    img_g, _ = image_pairs_literal(G, C, dim)
    death_of_l = {s: t for s, t, _, _ in img_l}          # birth cell in L -> death cell in C
    birth_of_g = {t: s for s, t, _, _ in img_g}          # death cell in C -> birth cell in G
    g_by_birth = {s: (bp, dp) for s, _, bp, dp in bar_g}
    own = (lambda s, t: s) if dim == 0 else (lambda s, t: t)
    matched, up, partner_g = [], [], set()
    for s, t, bp, dp in sorted(bar_l, key=lambda r: own(r[0], r[1])):
        sg = birth_of_g.get(death_of_l.get(s, -1), -1)
        if sg in g_by_birth:
            matched.append((bp, dp) + g_by_birth[sg])
            partner_g.add(sg)
        else:
            up.append((bp, dp))
    ut = [(bp, dp) for s, t, bp, dp in sorted(bar_g, key=lambda r: own(r[0], r[1])) if s not in partner_g]
    if dim == 0:
        matched.append((ess_l[1], int(np.argmax(L)), ess_g[1], int(np.argmax(G))))
    lf, gf = L.ravel().astype(np.float64), G.ravel().astype(np.float64)
    cost = sum((lf[a] - gf[c]) ** 2 + (lf[b] - gf[d]) ** 2 for a, b, c, d in matched)
    cost += sum((lf[b] - lf[a]) ** 2 / 2 for a, b in up) + sum((gf[b] - gf[a]) ** 2 / 2 for a, b in ut)
    arr = lambda rows, k: np.array(rows, dtype=np.int32).reshape(-1, k)
    return {"matched": arr(matched, 4), "unmatched_pred": arr(up, 2), "unmatched_target": arr(ut, 2), "cost": float(cost)}


def _lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        h = hashlib.sha256(b"".join(open(p, "rb").read() for p in _DEPS)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"betti_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=os.path.dirname(so))
            os.close(fd)
            subprocess.check_call([cc, "-O2", "-fPIC", "-fopenmp", "-std=c11", "-shared", "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)  # atomic: concurrent test processes see a whole library or none
        L = ctypes.CDLL(so)
        fp, ip = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int32)
        L.to_betti_matching.argtypes = [fp, fp] + [ctypes.c_int] * 3 + [ip, ip, ip, ctypes.c_int, ip,
                                                                       ctypes.POINTER(ctypes.c_double)]
        L.to_betti_matching.restype = ctypes.c_int
        _LIB = L
    return _LIB


def betti_matching(pred, target, dim: int) -> dict:
    """Betti matching of one HxW prediction / target pair by union-find (``to_betti_matching``), in the format and
    order of ``betti_matching_literal``: ``matched`` [M, 4], ``unmatched_pred`` / ``unmatched_target`` [K, 2] int32
    pixel indices and the float64 ``cost``."""
    L = np.ascontiguousarray(pred, dtype=np.float32)
    G = np.ascontiguousarray(target, dtype=np.float32)
    if L.shape != G.shape or L.ndim != 2:
        raise ValueError("betti_matching: two HxW maps of one shape")
    H, W = L.shape
    cap = (H + 1) * (W + 1) + 2
    m = np.empty((cap, 4), dtype=np.int32)
    up = np.empty((cap, 2), dtype=np.int32)
    ut = np.empty((cap, 2), dtype=np.int32)
    cnt = np.zeros(3, dtype=np.int32)
    cost = ctypes.c_double(0.0)
    fptr = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    iptr = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    if _lib().to_betti_matching(fptr(L), fptr(G), H, W, int(dim), iptr(m), iptr(up), iptr(ut), cap, iptr(cnt),
                                ctypes.byref(cost)) != 0:
        raise RuntimeError("to_betti_matching failed")
    return {"matched": m[:cnt[0]].copy(), "unmatched_pred": up[:cnt[1]].copy(), "unmatched_target": ut[:cnt[2]].copy(),
            "cost": float(cost.value)}
