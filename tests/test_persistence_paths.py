"""The persistence kernels on every path they take, on both sides of every dispatch threshold, against the oracle.

One launch serves ``topo_loss``, ``persistence_pairs``, ``cubical_persistence``, the ``tda`` layer and
``topological_prior``.  Per map it picks a branch from the shape, the map pointer's alignment, the value count and
the number K of level-0 sub-basins (``ph_small.cuh``, ``ph_binary.cuh``, ``ph_kernel.cuh``, ``make_scratch`` /
``launch_ph`` in ``topoloss_api.cu``).  This file restates that choice as a path model whose thresholds are read
from the sources, restates level 0 (``pick``, cut at band borders) in numpy to know K for any map, and runs one GPU
case on each side of every threshold.

Path model (``path``).  A map takes:

* kernel: ``global`` (``H + 1`` or ``W + 1`` over ``kSmallMaxRow``, or ``2^22`` nodes or more), else the
  shared-memory kernel, ``single`` (one band: <= 65536 pixels for H1, <= 65535 vertices for H0) or ``multi``;
* two-valued H1 path (``binary``): taken with ``vec`` or ``scalar`` loads, or rejected by the value count (within
  the 8-trip probe, ``reject_values_probe``, or after it, ``reject_values_late``), the run count (``reject_runs``,
  more than ``r_cap`` runs) or the mask size (``reject_mask``); ``off`` under ``OPT_NO_BINARY_PATH``, for H0 and in
  the global kernel;
* front end: ``fast_one`` (H1, W % 4 == 0, 16-byte aligned, one band), ``inband`` (the same over several bands,
  each merged on its own by ``band_merge``), ``generic_one`` or ``generic_multi``; ``alias`` (H1 with N == 65536:
  the last pixel doubles as OUTSIDE), the bands and the last band's width;
* phase-0 loads (every map but ``fast_one``): ``vec`` when N % 4 == 0 and the map is 16-byte aligned, else ``scalar``;
* ``band_merge`` (``inband`` only): ``fits`` when every band's packed table fits, else ``nofit``;
* final table: ``packed`` 64-bit entries, ``smem128`` (128-bit in shared memory), ``global128``, or ``inband``
  (the bands' global table);
* emission: root pixels in shared memory as 16 or 32 bits or read from global memory (``rp``), the emitting-basin
  list in shared memory or not (``lst``), root values read from the map (``zmap``);
* ``kst``: the basin tables of ``topo_loss`` (``n_nodes / 4 + 2`` basins for multi-band maps) are exhausted, the
  status word says so and the loss is NaN.  ``persistence_pairs`` always has the worst-case tables.

The two-valued path and the merge path are enumerated apart: a rejected two-valued map takes the merge path its K
gives whatever the reason it was rejected.  ``FEASIBLE_MERGE`` / ``FEASIBLE_BINARY`` are the products of the axes
minus the rules in ``MERGE_RULES`` / ``BINARY_RULES``, each of which says why its combinations cannot happen.

Level-0 model (``level0``).  The sub-basins are the connected components of the graph in which every node is linked
to the far end of its ``pick``, when that lies in the node's band (H1 adds OUTSIDE, which is not a basin).  Designed
maps give a known K (``peaks_map`` / ``pits_map``), which a CPU test checks.

Maps.  H1: a ramp that rises towards the bottom row, with strict peaks on interior checkerboard sites.  H0: a ramp
that rises towards the bottom row and to the right, with pits on sites two pixels apart.  Two-valued maps: isolated
hi pixels (one run each).

Every GPU case asserts ``persistence_pairs`` against ``oracle.cubical_pairs`` bit for bit and, for each map batch,
``topo_loss`` and its gradient against ``oracle.topo_loss`` within ``REL`` under the fused tail, ``OPT_NO_FUSED_GRAD``
and ``OPT_NO_FUSED_MATCH`` (and ``OPT_NO_BINARY_PATH`` for two-valued maps).  Where the loss's tables run out, the
loss is NaN, ``check_status`` names the basin tables, and ``OPT_WORST_CASE_WORKSPACE`` gives the oracle's loss.
"""
import functools
import itertools
import os
import re
from collections import namedtuple

import numpy as np
import pytest
import torch
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dilabhelmholtzoct_b200", "csrc")

F32 = np.float32
REL = 1e-5     # the suite's loss / gradient tolerance (test_gpu_parity.py)
LAMDA = 0.1


# ------------------------------------------------------------------ constants and expressions of the sources

@functools.lru_cache(maxsize=None)
def _src(path):
    with open(path) as f:
        return f.read()


def _const(fname, name):
    text = _src(os.path.join(CSRC, fname))
    m = re.search(rf"constexpr\s+(?:int|size_t)\s+{name}\s*=\s*([^;,]+)[;,]", text)
    assert m, f"{name} not found in {fname}: update the path model"
    expr = re.sub(r"(\d+)u\b", r"\1", m.group(1).strip())
    assert re.fullmatch(r"[\d\s*+\-()<]+", expr), expr
    return int(eval(expr))  # digits and + - * << ( ) only, checked above


def _struct_bytes(fname, name):
    """Size of a ``struct __align__(16)`` of uint64_t / uint32_t fields."""
    m = re.search(rf"struct __align__\(16\) {name} \{{(.*?)\}};", _src(os.path.join(CSRC, fname)), re.S)
    assert m, f"struct {name} not found in {fname}"
    size = 0
    for ty, names in re.findall(r"(uint64_t|uint32_t)\s+([\w\s,]+);", m.group(1)):
        size += (8 if ty == "uint64_t" else 4) * len(names.split(","))
    return (size + 15) // 16 * 16


K_SMALL_MAX_ROW = _const("ph_small.cuh", "kSmallMaxRow")
K_SMALL_SMEM = _const("ph_small.cuh", "kSmallSmemBytes")
K_PH_THREADS = _const("ph_kernel.cuh", "kPhThreads")
K_RING = _const("ph_small.cuh", "kRing")
CROSS_EDGE = _struct_bytes("ph_small.cuh", "CrossEdge")
TENTRY = _struct_bytes("ph_small.cuh", "TEntry")
RING_BYTES = (K_PH_THREADS // 32) * K_RING * CROSS_EDGE   # the warps' staging rings
T_CAP_SMEM = K_SMALL_SMEM // TENTRY

# Every expression the model restates, verbatim: a change to any of them fails test_model_pins_match_the_sources.
PINS = {
    "ph_small.cuh": [
        "const bool fast = DIM == 1 && (W & 3) == 0 && H <= 16383 && (reinterpret_cast<uintptr_t>(g.f) & 15) == 0;",
        "const bool fast_one = fast && N <= 65536;",
        "if (!fast_one) {",
        "if ((N & 3) == 0 && (reinterpret_cast<uintptr_t>(g.f) & 15) == 0) {",
        "const int rowlen = DIM == 1 ? W : VW, n_rows = DIM == 1 ? H : H + 1;",
        "const bool alias = DIM == 1 && N == 65536;",
        "const int cols_per_band = alias ? rowlen : fast ? min(rowlen, (65535 / n_rows) & ~3) : min(rowlen, 65535 / n_rows);",
        "const bool one_band = !MULTI || cols_per_band >= rowlen;",
        "const bool inband = MULTI && fast && !one_band;",
        "const int n_ids_b = B.H * GWb + bw;",
        "const int Pb = 32 - __clz(n_ids_b), Gb = 32 - __clz(Kb + 1);",
        "const size_t ring_b = (size_t)(((Kb + 1) * 8 + 15) & ~15) + (size_t)(((Kb + 1) * 4 + 15) & ~15);",
        "const bool fits = Pb + Gb <= 32 && ring_b + (size_t)(kPhThreads / 32) * kRing * sizeof(CrossEdge) + "
        "(size_t)B.top_reserved <= (size_t)kSmallSmemBytes;",
        "bm.top_reserved = 4 * n_rows_all;",
        "if ((size_t)K + 2 > S.k_stride) {",
        "const int n_edge_ids = H * GW + W;",
        "const int Pbits = 32 - __clz(n_edge_ids), Gbits = 32 - __clz(K + 1);",
        "const size_t ring_off = (size_t)(((K + 1) * 8 + 15) & ~15) + (size_t)(((K + 1) * 4 + 15) & ~15);",
        "const bool packed = !inband && Pbits + Gbits <= 32 && ring_off + (size_t)(kPhThreads / 32) * kRing * "
        "sizeof(CrossEdge) <= (size_t)kSmallSmemBytes;",
        "const int t_cap_smem = kSmallSmemBytes / (int)sizeof(TEntry);",
        "const bool t_in_smem = !inband && K + 1 <= t_cap_smem;",
        "const size_t rp_off = ring_off + (size_t)(kPhThreads / 32) * kRing * sizeof(CrossEdge);",
        "const bool rp16 = (DIM == 1 ? N : NN) <= 65536;",
        "const bool rp_smem = packed && rp_off + (size_t)(K + 1) * (rp16 ? 2 : 4) <= (size_t)kSmallSmemBytes;",
        "const bool lst_smem = packed && (size_t)K * 2 <= (size_t)(kPhThreads / 32) * kRing * sizeof(CrossEdge);",
        "const bool z_in_map = fast && !MULTI;",
        "if (DIM == 1 && S.binary_path &&",
        "binary_h1_pairs(A.maps[set] + (size_t)map * N, H, W, smem, kSmallSmemBytes, A.ps, set, map, S.prof)",
        # pick (H1): bottom > right > left > top among the edges that carry the pixel's own value
        "if (r == H - 1) out = true;\n                else if (fd >= fp) { dr = 1; fo = fd; }\n"
        "                else if (c == W - 1) out = true;\n                else if (fr >= fp) { dc = 1; fo = fr; }\n"
        "                else if (c == 0) out = true;\n                else if (fl >= fp) { dc = -1; fo = fl; }\n"
        "                else if (r == 0) out = true;\n                else if (fu >= fp) { dr = -1; fo = fu; }\n"
        "                else none = true;",
        # pick (H0): the least (value, position) key among the vertex's edges
        "uint64_t k = g.make_ekey(g.vedge_val(r - 1, c), (uint32_t)(2 * c + (2 * r - 1) * GW));",
        "uint64_t k = g.make_ekey(g.vedge_val(r, c), (uint32_t)(2 * c + (2 * r + 1) * GW));",
        "uint64_t k = g.make_ekey(g.hedge_val(r, c - 1), (uint32_t)(2 * c - 1 + (2 * r) * GW));",
        "uint64_t k = g.make_ekey(g.hedge_val(r, c), (uint32_t)(2 * c + 1 + (2 * r) * GW));",
        "return (c2 < c0 || c2 >= c1) ? -1 : xl + dr * bw + dc;",
    ],
    "topoloss_api.cu": [
        "L.n_nodes = dim == 1 ? H * W + 1 : (H + 1) * (W + 1);",
        "L.small = (W + 1) <= tl::kSmallMaxRow && (H + 1) <= tl::kSmallMaxRow && (long long)L.n_nodes < (1ll << 22);",
        "size_t k_cap = (size_t)L.cap;",
        "if (L.n_nodes > 65537 && !opt(TL_OPT_WORST_CASE_WORKSPACE) && !with_sort) k_cap = (size_t)L.n_nodes / 4 + 2;",
        "L.k_stride = align_up(k_cap + 2, 64);",
        "const long long nn = dim == 1 ? (long long)H * W + 1 : (long long)(H + 1) * (W + 1);\n    return (int)(nn / 2 + 2);",
        "const bool single = dim == 1 ? (long long)H * W <= 65536 : (long long)(H + 1) * (W + 1) <= 65535;",
        "const bool use_small = L.small && !opt(TL_OPT_FORCE_GLOBAL_KERNEL);",
        "sa.binary_path = !opt(TL_OPT_NO_BINARY_PATH);",
    ],
    "ph_binary.cuh": [
        "const int nw = (W + 31) >> 5, n_words = H * nw;",
        "const int fixed = ((n_words * 6 + 15) & ~15);",
        "if (fixed + 3 * 64 > smem_bytes || n_words >= (1 << 22)) return 0;",
        "int r_cap = (smem_bytes - fixed) / 3;",
        "if (r_cap > 65535) r_cap = 65535;",
        "if (n_runs > r_cap) return 0;",
        "const bool vec = (W & 127) == 0 && (reinterpret_cast<uintptr_t>(f) & 15) == 0;",
        "const int per_trip = vec ? 4 : 1;",
        "const int n_it = (n_words + nwarp * per_trip - 1) / (nwarp * per_trip);",
        "const int it_probe = n_it < (vec ? 4 : 8) ? n_it : (vec ? 4 : 8);",
    ],
    # the Python entry points hand a contiguous view to the library as it is, storage offset included
    "../topological_loss.py": [
        "flat = maps.reshape(-1, H, W).contiguous()",
        "pred, truth = pred.contiguous(), truth.contiguous()",
    ],
}


# ------------------------------------------------------------------ path model

def _a16(x):
    return (x + 15) & ~15


def _align_up(x, a):
    return (x + a - 1) // a * a


def n_nodes(H, W, dim):
    return H * W + 1 if dim == 1 else (H + 1) * (W + 1)


def small_kernel(H, W, dim):
    return W + 1 <= K_SMALL_MAX_ROW and H + 1 <= K_SMALL_MAX_ROW and n_nodes(H, W, dim) < (1 << 22)


def single_band(H, W, dim):
    return H * W <= 65536 if dim == 1 else (H + 1) * (W + 1) <= 65535


def is_fast(H, W, dim, aligned16):
    return dim == 1 and W % 4 == 0 and H <= 16383 and aligned16


def bands(H, W, dim, aligned16):
    """(c0, width) of the bands the shared-memory kernel cuts the map into (node columns)."""
    rowlen, n_rows = (W, H) if dim == 1 else (W + 1, H + 1)
    if single_band(H, W, dim):
        return [(0, rowlen)]
    cols = min(rowlen, (65535 // n_rows) & ~3) if is_fast(H, W, dim, aligned16) else min(rowlen, 65535 // n_rows)
    return [(c0, min(rowlen, c0 + cols) - c0) for c0 in range(0, rowlen, cols)]


def k_stride(H, W, dim, api, options=()):
    nn = n_nodes(H, W, dim)
    k_cap = nn // 2 + 2
    if nn > 65537 and "OPT_WORST_CASE_WORKSPACE" not in options and api == "loss":
        k_cap = nn // 4 + 2
    return _align_up(k_cap + 2, 64)


def packed_fits(H, W, K):
    n_edge_ids = H * (2 * W + 1) + W
    return n_edge_ids.bit_length() + (K + 1).bit_length() <= 32 and \
        _a16((K + 1) * 8) + _a16((K + 1) * 4) + RING_BYTES <= K_SMALL_SMEM


def band_fits(H, W, dim, bw, Kb):
    n_ids_b = H * (2 * bw + 1) + bw
    ring_b = _a16((Kb + 1) * 8) + _a16((Kb + 1) * 4)
    top = 4 * (H if dim == 1 else H + 1)
    return n_ids_b.bit_length() + (Kb + 1).bit_length() <= 32 and ring_b + RING_BYTES + top <= K_SMALL_SMEM


def binary_r_cap(H, W):
    """(fits, r_cap) of the two-valued path's shared memory for an H x W mask."""
    n_words = H * ((W + 31) >> 5)
    fixed = (n_words * 6 + 15) & ~15
    if fixed + 3 * 64 > K_SMALL_SMEM or n_words >= (1 << 22):
        return False, 0
    return True, min((K_SMALL_SMEM - fixed) // 3, 65535)


def mono32(f):
    u = np.ascontiguousarray(f, F32).view(np.uint32).copy()
    u[u == 0x80000000] = 0
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def count_runs(hi):
    """Maximal horizontal runs of True pixels."""
    nxt = np.zeros_like(hi)
    nxt[:, :-1] = hi[:, 1:]
    return int((hi & ~nxt).sum())


def binary_outcome(f, aligned16):
    """What ``binary_h1_pairs`` does with map f (shared-memory kernel, H1, the path not switched off)."""
    H, W = f.shape
    ok, r_cap = binary_r_cap(H, W)
    if not ok:
        return "reject_mask"
    vec = W % 128 == 0 and aligned16
    nw, per_trip, nwarp = (W + 31) >> 5, 4 if vec else 1, K_PH_THREADS // 32
    n_words = H * nw
    n_it = (n_words + nwarp * per_trip - 1) // (nwarp * per_trip)
    probe_words = min(n_words, min(n_it, 4 if vec else 8) * nwarp * per_trip)
    m = mono32(f)
    ref = m[0, 0]
    word = np.arange(H)[:, None] * nw + np.arange(W)[None, :] // 32
    others = np.unique(m[m != ref])
    if len(np.unique(m[(word < probe_words) & (m != ref)])) > 1:
        return "reject_values_probe"
    if len(others) > 1:
        return "reject_values_late"
    if len(others) == 1 and count_runs(m == max(ref, others[0])) > r_cap:
        return "reject_runs"
    return "vec" if vec else "scalar"


Path = namedtuple("Path", "kernel binary front alias n_bands last_bw p0 merge table rp lst zmap kst")


def path(H, W, dim, K, aligned16=True, api="pairs", options=(), binary="reject_values_probe"):
    """Branch tuple of one map.  K: sub-basins per band (a list, as ``level0`` gives) or their total for a map of
    one band; ``binary``: ``binary_outcome`` of the map (H1, shared-memory kernel)."""
    Kb = list(K) if isinstance(K, (list, tuple)) else [K]
    K = sum(Kb)
    if not small_kernel(H, W, dim) or "OPT_FORCE_GLOBAL_KERNEL" in options:
        return Path("global", "off" if dim == 1 else None, *(None,) * 11)
    kernel = "single" if single_band(H, W, dim) else "multi"
    b = None
    if dim == 1:
        b = "off" if "OPT_NO_BINARY_PATH" in options else binary
        if b in ("vec", "scalar"):
            return Path(kernel, b, *(None,) * 11)
    N = H * W
    fast = is_fast(H, W, dim, aligned16)
    fast_one = fast and N <= 65536
    alias = dim == 1 and N == 65536
    bl = bands(H, W, dim, aligned16)
    one_band = kernel == "single" or len(bl) == 1
    inband = kernel == "multi" and fast and not one_band
    assert not (fast and not fast_one and one_band)
    front = "fast_one" if fast_one else "inband" if inband else "generic_one" if one_band else "generic_multi"
    if len(Kb) != len(bl):
        assert len(Kb) == 1 and not inband, "band_merge needs K per band"
    p0 = None if fast_one else ("vec" if N % 4 == 0 and aligned16 else "scalar")
    merge = None
    if inband:
        merge = "fits" if all(band_fits(H, W, dim, bw, k) for (_, bw), k in zip(bl, Kb)) else "nofit"
    head = (kernel, b, front, alias, len(bl), bl[-1][1], p0, merge)
    if K + 2 > k_stride(H, W, dim, api, options):
        return Path(*head, None, None, None, False, True)
    if inband:
        return Path(*head, "inband", None, None, False, False)
    if packed_fits(H, W, K):
        rp16 = (N if dim == 1 else n_nodes(H, W, 0)) <= 65536
        rp_off = _a16((K + 1) * 8) + _a16((K + 1) * 4) + RING_BYTES
        rp = ("smem16" if rp16 else "smem32") if rp_off + (K + 1) * (2 if rp16 else 4) <= K_SMALL_SMEM else "global"
        lst = "smem" if K * 2 <= RING_BYTES else "global"
        return Path(*head, "packed", rp, lst, fast_one, False)
    return Path(*head, "smem128" if K + 1 <= T_CAP_SMEM else "global128", None, None, fast_one, False)


def merge_tuple(dim, p):
    return (dim, p.kernel, p.front, p.alias, p.p0, p.merge, p.table, p.rp, p.lst, p.zmap, p.kst)


MERGE_AXES = [(0, 1), ("single", "multi"), ("fast_one", "inband", "generic_one", "generic_multi"), (False, True),
              (None, "vec", "scalar"), (None, "fits", "nofit"), (None, "packed", "smem128", "global128", "inband"),
              (None, "smem16", "smem32", "global"), (None, "smem", "global"), (False, True), (False, True)]

# (why the combinations cannot happen, predicate over (dim, kernel, front, alias, p0, merge, table, rp, lst, zmap, kst))
MERGE_RULES = [
    ("the fast front end needs H1 pixels in 128-bit quads", lambda d, k, f, a, p0, m, t, rp, l, z, s: d == 0 and f in ("fast_one", "inband")),
    ("fast_one / generic_one run in the single-band kernel, inband / generic_multi in the multi-band one",
     lambda d, k, f, a, p0, m, t, rp, l, z, s: (f in ("fast_one", "generic_one")) != (k == "single")),
    ("the OUTSIDE alias is H1 at N == 65536, which is one band", lambda d, k, f, a, p0, m, t, rp, l, z, s: a and (d == 0 or k != "single")),
    ("N == 65536 within kSmallMaxRow makes W a power of two >= 16, so a generic front end there means a misaligned map, "
     "whose phase 0 loads scalars", lambda d, k, f, a, p0, m, t, rp, l, z, s: a and f == "generic_one" and p0 == "vec"),
    ("phase 0 runs on every map but fast_one's", lambda d, k, f, a, p0, m, t, rp, l, z, s: (f == "fast_one") != (p0 is None)),
    ("an inband map is 16-byte aligned with W % 4 == 0, so N % 4 == 0: vector loads",
     lambda d, k, f, a, p0, m, t, rp, l, z, s: f == "inband" and p0 == "scalar"),
    ("band_merge runs on inband maps only", lambda d, k, f, a, p0, m, t, rp, l, z, s: (f == "inband") != (m is not None)),
    ("only multi-band maps get the typical-size basin tables (n_nodes > 65537)",
     lambda d, k, f, a, p0, m, t, rp, l, z, s: s and k != "multi"),
    ("a map whose basin tables ran out stops before the final table", lambda d, k, f, a, p0, m, t, rp, l, z, s: s == (t is not None)),
    ("inband maps keep the bands' global table", lambda d, k, f, a, p0, m, t, rp, l, z, s: t is not None and (f == "inband") != (t == "inband")),
    ("H0 maps of 65536 vertices have H + 1, W + 1 powers of two, so N is odd: scalar phase 0",
     lambda d, k, f, a, p0, m, t, rp, l, z, s: d == 0 and rp == "smem16" and k == "multi" and p0 == "vec"),
    ("a single band has Pbits <= 18, so the packed form fails only at K + 1 >= 2^14 > t_cap_smem",
     lambda d, k, f, a, p0, m, t, rp, l, z, s: k == "single" and t == "smem128"),
    ("the emission scratch goes with the packed table", 
     lambda d, k, f, a, p0, m, t, rp, l, z, s: (t == "packed") != (rp is not None) or (t == "packed") != (l is not None)),
    ("a packed table has K < 16298 basins, whose list fits the staging rings", lambda d, k, f, a, p0, m, t, rp, l, z, s: l == "global"),
    ("root pixels fit 16 bits on single-band maps, and of the multi-band ones only on H0 maps of 65536 vertices",
     lambda d, k, f, a, p0, m, t, rp, l, z, s: (rp == "smem16" and k != "single" and d == 1) or (rp == "smem32" and k == "single")),
    ("root values come from the map on fast_one maps that reach the table", lambda d, k, f, a, p0, m, t, rp, l, z, s: z != (f == "fast_one" and t is not None)),
]
FEASIBLE_MERGE = {t for t in itertools.product(*MERGE_AXES) if not any(rule(*t) for _, rule in MERGE_RULES)}

BINARY_AXES = [("single", "multi", "global"),
               ("vec", "scalar", "reject_values_probe", "reject_values_late", "reject_runs", "reject_mask", "off")]
BINARY_RULES = [
    ("the global-memory kernel has no two-valued path", lambda k, o: k == "global" and o != "off"),
    ("a single band's <= 65536 pixels need <= 4096 mask words: it always fits", lambda k, o: k == "single" and o == "reject_mask"),
    ("a single band has <= 32768 runs and r_cap == 65535 there", lambda k, o: k == "single" and o == "reject_runs"),
]
FEASIBLE_BINARY = {t for t in itertools.product(*BINARY_AXES) if not any(rule(*t) for _, rule in BINARY_RULES)}


# ------------------------------------------------------------------ level-0 model

def level0(f, dim, aligned16=True):
    """Sub-basins per band after level 0: numpy restatement of ``pick`` with links cut at band borders."""
    f = np.ascontiguousarray(f, F32)
    H, W = f.shape
    if dim == 1:
        R, C = np.mgrid[0:H, 0:W]
        fp = f
        fd = np.vstack([f[1:], f[-1:]])
        fr = np.hstack([f[:, 1:], f[:, -1:]])
        fl = np.hstack([f[:, :1], f[:, :-1]])
        fu = np.vstack([f[:1], f[:-1]])
        conds = [R == H - 1, fd >= fp, C == W - 1, fr >= fp, C == 0, fl >= fp, R == 0, fu >= fp]
        kind = np.select(conds, ["out", "d", "out", "r", "out", "l", "out", "u"], "none")
        dr = np.select([kind == "d", kind == "u"], [1, -1], 0)
        dc = np.select([kind == "r", kind == "l"], [1, -1], 0)
        n_rows, rowlen = H, W
    else:
        R, C = np.mgrid[0:H + 1, 0:W + 1]
        m = mono32(f).astype(np.uint64)
        GW = 2 * W + 1
        big = np.uint64(~np.uint64(0))

        def at(r, c):  # pixel value keys, +inf outside
            out = np.full(R.shape, big, np.uint64)
            ok = (r >= 0) & (r < H) & (c >= 0) & (c < W)
            out[ok] = m[r[ok], c[ok]]
            return out

        def vedge(i, j):  # v-edge (i, j): pixels (i, j-1), (i, j)
            return np.minimum(at(i, j - 1), at(i, j))

        def hedge(i, j):  # h-edge (i, j): pixels (i-1, j), (i, j)
            return np.minimum(at(i - 1, j), at(i, j))

        sh = np.uint64(32)
        cand = [
            (R > 0, (vedge(R - 1, C) << sh) | (2 * C + (2 * R - 1) * GW).astype(np.uint64), -1, 0),
            (R < H, (vedge(R, C) << sh) | (2 * C + (2 * R + 1) * GW).astype(np.uint64), 1, 0),
            (C > 0, (hedge(R, C - 1) << sh) | (2 * C - 1 + 2 * R * GW).astype(np.uint64), 0, -1),
            (C < W, (hedge(R, C) << sh) | (2 * C + 1 + 2 * R * GW).astype(np.uint64), 0, 1),
        ]
        best = np.full(R.shape, big, np.uint64)
        dr = np.zeros(R.shape, int)
        dc = np.zeros(R.shape, int)
        for ok, key, a, b in cand:
            take = ok & (key < best)
            best[take] = key[take]
            dr[take] = a
            dc[take] = b
        kind = np.full(R.shape, "x")
        n_rows, rowlen = H + 1, W + 1
    alias = dim == 1 and H * W == 65536
    out_node = n_rows * rowlen
    src = (R * rowlen + C).ravel()
    far = ((R + dr) * rowlen + (C + dc)).ravel()
    kind = kind.ravel()
    if dim == 1:
        far = np.where(kind == "out", out_node, far)
        if alias:
            far = np.where(far == H * W - 1, out_node, far)
        linked = kind != "none"
    else:
        linked = np.ones(src.shape, bool)
    cfar = np.where(far == out_node, -1, far % rowlen)
    Ks = []
    for c0, bw in bands(H, W, dim, aligned16):
        inb = (C.ravel() >= c0) & (C.ravel() < c0 + bw)
        ok = inb & linked & ((cfar == -1) | ((cfar >= c0) & (cfar < c0 + bw)))
        nodes = np.concatenate([src[inb], [out_node]]) if dim == 1 else src[inb]
        idx = np.full(out_node + 1, -1)
        idx[nodes] = np.arange(len(nodes))
        g = coo_matrix((np.ones(int(ok.sum())), (idx[src[ok]], idx[far[ok]])), shape=(len(nodes), len(nodes)))
        n_comp = connected_components(g, directed=True, connection="weak")[0]
        Ks.append(n_comp - (1 if dim == 1 else 0))
    return Ks


# ------------------------------------------------------------------ maps with a known K

def _ramp(H, W):
    """Rises strictly towards the bottom row, and within a row to the right: values in [0.25, 0.75)."""
    r = np.arange(H, dtype=np.float64)[:, None]
    c = np.arange(W, dtype=np.float64)[None, :]
    return (0.25 + 0.5 * (r + c / (W + 1)) / H).astype(F32)


def peaks_map(H, W, K, seed=0, cols=None):
    """H1: K strict peaks (values in [1, 2)) on interior checkerboard sites of the ramp.  Every other pixel links
    down (its lower neighbour is higher) or, on the last row, to OUTSIDE, and a peak is a strict maximum: the
    sub-basins are the K peaks with the column segments above them, in any band cut (links are vertical), so
    K(level 0) == K, and every peak is one H1 pair of the oracle."""
    rng = np.random.default_rng(seed)
    f = _ramp(H, W)
    ys, xs = np.nonzero((np.add.outer(np.arange(H), np.arange(W)) % 2 == 0))
    lo, hi = cols or (0, W)
    inner = (ys > 0) & (ys < H - 1) & (xs > 0) & (xs < W - 1) & (xs >= lo) & (xs < hi)
    ys, xs = ys[inner], xs[inner]
    assert K <= len(ys), (H, W, K, len(ys))
    sel = rng.choice(len(ys), K, replace=False)
    f[ys[sel], xs[sel]] = (1.0 + rng.random(K)).astype(F32)
    return f


def pits_sites(H, W, dim_bands):
    """Pixels (r, c) with r, c even: pairwise not 8-adjacent.  ``dim_bands``: the H0 bands.  Left out: a pit whose
    two vertex columns c, c + 1 straddle a band border, and a pit in row 0 at a band's first vertex column."""
    ys, xs = np.mgrid[0:H:2, 0:W:2]
    ys, xs = ys.ravel(), xs.ravel()
    starts = {c0 for c0, _ in dim_bands}
    keep = np.array([x + 1 not in starts and not (y == 0 and x in starts) for y, x in zip(ys, xs)], bool)
    return ys[keep], xs[keep]


def pits_map(H, W, P, aligned16=True, seed=0):
    """H0: P pits (values in [-2, -1)) on ``pits_sites`` of the ramp.

    K by hand, for pits that do not straddle a band border.  Vertex (r, c) takes the least of its <= 4 pixels; the
    ramp makes that an upper pixel for r >= 1, and the up edge carries the same value with the least bitmap
    position, so every such vertex links up.  Row 0 rises to the right, so its vertices link left, to the band's
    first vertex.  One basin per band so far.  A pit is below all of its 8 neighbours (sites are 2 apart), so its 4
    corners take its value; they link to each other (right / left along the top edge, up from the bottom two), and
    the vertices under the pit link up into it: one basin per pit.  Where a pit sits in row 0 its top corners cut
    the band's row-0 chain, whose right part then links into the pit: still one basin for the band's left part,
    unless the pit sits at the band's first vertex column, where the whole band would join it (no site is there).
    A pit that straddles a band border would be two basins (no site does).  Hence K = P + n_bands, and the oracle's H0 diagram holds P + 1 points (each pit dies where it meets the ramp, plus the
    essential class)."""
    rng = np.random.default_rng(seed)
    f = _ramp(H, W)
    ys, xs = pits_sites(H, W, bands(H, W, 0, aligned16))
    assert P <= len(ys), (H, W, P, len(ys))
    sel = rng.choice(len(ys), P, replace=False)
    f[ys[sel], xs[sel]] = (-2.0 + rng.random(P)).astype(F32)
    return f


def isolated_runs(H, W, runs, seed=0, interior=True):
    """Two-valued (0 / 1): ``runs`` isolated 1-pixels on checkerboard sites (odd r + c), each a run of its own."""
    rng = np.random.default_rng(seed)
    f = np.zeros((H, W), F32)
    ys, xs = np.nonzero(np.add.outer(np.arange(H), np.arange(W)) % 2 == 1)
    if interior:
        keep = (ys > 0) & (ys < H - 1) & (xs > 0) & (xs < W - 1)
        ys, xs = ys[keep], xs[keep]
    assert runs <= len(ys), (runs, len(ys))
    sel = rng.choice(len(ys), runs, replace=False) if runs < len(ys) else np.arange(len(ys))
    f[ys[sel], xs[sel]] = 1.0
    return f


def blobs_truth(H, W, n=4, seed=0):
    """Ground truth: a few 3 x 3 blocks of 1 on 0, off the border."""
    rng = np.random.default_rng(seed + 1000)
    f = np.zeros((H, W), F32)
    for _ in range(n):
        y, x = int(rng.integers(1, max(2, H - 4))), int(rng.integers(1, max(2, W - 4)))
        f[y:y + min(3, H - 1 - y), x:x + min(3, W - 1 - x)] = 1.0
    return f


# ------------------------------------------------------------------ thresholds in K, from the model

def k_first(pred, lo=0, hi=1 << 22):
    """The least K >= lo for which pred(K) holds (pred monotone)."""
    while lo < hi:
        mid = (lo + hi) // 2
        if pred(mid):
            hi = mid
        else:
            lo = mid + 1
    return lo


def k_packed_end(H, W):
    """Least K the packed table does not take."""
    return k_first(lambda K: not packed_fits(H, W, K))


def k_rp_end(H, W, dim):
    """Least K whose root pixels leave shared memory while the table is packed."""
    N = H * W if dim == 1 else n_nodes(H, W, 0)
    b = 2 if N <= 65536 else 4
    return k_first(lambda K: _a16((K + 1) * 8) + _a16((K + 1) * 4) + RING_BYTES + (K + 1) * b > K_SMALL_SMEM)


def k_band_fit_end(H, W, dim, bw):
    return k_first(lambda Kb: not band_fits(H, W, dim, bw, Kb))


# ------------------------------------------------------------------ GPU cases
#
# A case is one batch of maps of one shape and one base alignment; a map is (builder, args).  Its K comes from
# ``level0``, its branch from ``path``.  ``loss``: the batch also goes through topo_loss (as [n, 1] maps, with a
# two-valued ground truth); ``kst``: its loss runs out of basin tables.

TH = {}  # thresholds the cases sit on, recomputed from the model so that they follow the sources


def _th():
    if not TH:
        TH["pk256"] = k_packed_end(256, 256)             # fast_one / generic_one, 256 x 256
        TH["rp256"] = k_rp_end(256, 256, 1)
        TH["pk365"] = k_packed_end(364, 365)              # generic multi-band H1
        TH["ks364"] = k_stride(364, 365, 1, "loss")
        TH["rp259"] = k_rp_end(260, 257, 1)               # multi-band with Pbits == 18: packed, root pixels global
        TH["fit260"] = k_band_fit_end(256, 260, 1, 252)   # inband 256 x 260: bands 252 + 8
        TH["ks260"] = k_stride(256, 260, 1, "loss")
        TH["pk0"] = k_packed_end(254, 256)
        TH["rp0"] = k_rp_end(254, 256, 0)
    return TH


def _cases():
    t = _th()
    P, Q = "peaks", "pits"
    C = []

    def case(name, dim, H, W, maps, offset=0, loss=True, kst=False):
        C.append(dict(name=name, dim=dim, H=H, W=W, maps=maps, offset=offset, loss=loss, kst=kst))

    # ---- H1, one band: N = 65535 / 65536, fast_one / generic, alias, packed / root pixels global / 128-bit global
    k256 = [(P, 300), (P, t["rp256"] - 1), (P, t["rp256"]), (P, t["pk256"] - 1), (P, t["pk256"])]
    case("h1_256_fast_alias", 1, 256, 256, k256)
    case("h1_256_generic_alias", 1, 256, 256, k256, offset=1)
    case("h1_255x257_generic_scalar", 1, 255, 257, [(P, 300), (P, t["rp256"]), (P, t["pk256"])])
    case("h1_252x255_generic_vec", 1, 252, 255, [(P, 300), (P, t["rp256"]), (P, t["pk256"])])
    case("h1_252x256_fast", 1, 252, 256, [(P, 300), (P, t["rp256"]), (P, t["pk256"])])
    # ---- H1, several bands, generic: packed / 128-bit shared / global spill, vector and scalar phase 0
    k365 = [(P, t["pk365"] - 1), (P, t["pk365"]), (P, T_CAP_SMEM - 2), (P, T_CAP_SMEM - 1)]
    case("h1_364x365_generic_vec", 1, 364, 365, k365)
    case("h1_364x365_generic_scalar", 1, 364, 365, k365, offset=1)
    case("h1_260x257_generic_rp", 1, 260, 257, [(P, t["rp259"] - 1), (P, t["rp259"])])
    case("h1_260x257_generic_rp_scalar", 1, 260, 257, [(P, t["rp259"])], offset=1)
    # basin tables of topo_loss: K = k_stride - 2 fits, k_stride - 1 does not
    case("h1_364x365_tables_fit", 1, 364, 365, [(P, t["ks364"] - 2), (P, 100)])
    case("h1_364x365_tables_out", 1, 364, 365, [(P, t["ks364"] - 1), (P, 100)], kst=True)
    case("h1_364x365_tables_out_scalar", 1, 364, 365, [(P, t["ks364"] - 1), (P, 100)], offset=1, kst=True)
    # ---- H1, several bands, fast front end (bands 252 + 8): band_merge fits / not, with the loss's tables
    case("h1_256x260_inband", 1, 256, 260, [(P, 2000), (P, t["fit260"] - 1), ("peaks_bands", (t["fit260"], 100))])
    case("h1_256x260_inband_tables_fit", 1, 256, 260, [("peaks_bands", (t["fit260"] - 1, t["ks260"] - 2 - t["fit260"] + 1)),
                                                       (P, 100)])
    case("h1_256x260_inband_tables_out", 1, 256, 260, [("peaks_bands", (t["fit260"] - 1, t["ks260"] - 1 - t["fit260"] + 1)),
                                                       (P, 100)], kst=True)
    case("h1_256x260_inband_nofit_tables_out", 1, 256, 260, [("peaks_bands", (t["fit260"] + 2000, 600)), (P, 100)], kst=True)
    case("h1_256x260_generic_multi", 1, 256, 260, [(P, 2000)], offset=1)
    # ---- tall and wide maps at the row limit, and past it
    case("h1_4096x16_alias", 1, 4096, 16, [(P, 3000), (P, 100)])
    case("h1_4096x16_generic", 1, 4096, 16, [(P, 3000)], offset=1)
    case("h1_16x4096_alias", 1, 16, 4096, [(P, 3000), (P, 100)])
    case("h1_16x4096_generic", 1, 16, 4096, [(P, 3000)], offset=1)
    case("h1_4096x28_inband", 1, 4096, 28, [(P, 3000), (P, 100)])
    case("h1_4096x28_generic", 1, 4096, 28, [(P, 3000), (P, 100)], offset=1)
    case("h1_20x4096_inband", 1, 20, 4096, [(P, 3000), (P, 100)])
    case("h1_4097x8_global", 1, 4097, 8, [(P, 2000), (P, 100)])
    case("h1_8x4097_global", 1, 8, 4097, [(P, 2000), (P, 100)])
    # ---- 2^22 nodes: 1778 x 2359 (2^22 - 1 nodes, shared-memory kernel), 2047 x 2049 and 2048^2 (global kernel)
    case("h1_1778x2359_small", 1, 1778, 2359, [(P, 20000)], loss=False)
    case("h1_2047x2049_global", 1, 2047, 2049, [(P, 20000)], loss=False)
    case("h1_2048_global", 1, 2048, 2048, [(P, 20000)], loss=False)
    # ---- two-valued maps: runs at r_cap / r_cap + 1, mask size, a third value after the probe, vec / scalar
    case("bin_256x512_runs", 1, 256, 512, [("runs_all", (65535,)), ("runs_all", (65536,))])
    case("bin_256x512_runs_scalar", 1, 256, 512, [("runs_all", (65535,)), ("runs_all", (65536,))], offset=1)
    fit1188 = binary_r_cap(1188, 1024)[1]
    case("bin_1188x1024_runs", 1, 1188, 1024, [("runs", (fit1188,)), ("runs", (fit1188 + 1,))])
    case("bin_1189x1024_mask", 1, 1189, 1024, [("runs", (50,)), ("runs", (10,))])
    case("bin_256x256_vec", 1, 256, 256, [("runs", (200,)), ("third_last", (200,)), ("third_first", (200,))])
    case("bin_256x250_scalar", 1, 256, 250, [("runs", (200,)), ("third_last", (200,))])
    case("bin_256x512_third_last", 1, 256, 512, [("third_last", (5000,)), ("runs", (5000,))])
    # ---- H0: (H+1)(W+1) = 65535 (one band) / 65536 (bands 255 + 1), several bands, tables, the global kernel
    k0 = [(Q, 300), (Q, t["rp0"]), (Q, 16255)]
    case("h0_254x256_vec", 0, 254, 256, k0)
    case("h0_254x256_scalar", 0, 254, 256, k0, offset=1)
    case("h0_253x257_max", 0, 253, 257, [("pits_all", ())])
    case("h0_15x4092_max", 0, 15, 4092, [("pits_all", ()), (Q, 300)])
    case("h0_255x255_two_bands", 0, 255, 255, [(Q, 300), (Q, 3000)])
    k0m = [(Q, 4000), (Q, 11000), (Q, 16000)]   # packed, 128-bit shared, 128-bit global
    case("h0_364x364_multi", 0, 364, 364, k0m)
    case("h0_364x364_multi_scalar", 0, 364, 364, k0m, offset=1)
    case("h0_257x259_multi_rp", 0, 257, 259, [(Q, 13000)])
    case("h0_256x260_multi_rp", 0, 256, 260, [(Q, 13000)])
    case("h0_365x365_tables_out", 0, 365, 365, [("pits_all", ()), (Q, 100)], kst=True)
    case("h0_4096x16_tables_out", 0, 4096, 16, [("pits_all", ()), (Q, 100)], kst=True)
    case("h0_4096x16", 0, 4096, 16, [(Q, 3000), (Q, 100)])
    case("h0_16x4096", 0, 16, 4096, [(Q, 3000), (Q, 100)])
    case("h0_4097x8_global", 0, 4097, 8, [(Q, 2000), (Q, 100)])
    case("h0_2046x2048_small", 0, 2046, 2048, [(Q, 20000)], loss=False)
    case("h0_2047_global", 0, 2047, 2047, [(Q, 20000)], loss=False)
    return C


CASES = _cases()
CASE_BY_NAME = {c["name"]: c for c in CASES}


def build(spec, H, W, dim, aligned16, seed):
    kind, arg = spec
    if kind == "peaks":
        return peaks_map(H, W, arg, seed)
    if kind == "peaks_bands":  # H1 fast bands: (peaks in band 0, peaks in the others)
        k0, k1 = arg
        c1 = bands(H, W, 1, True)[0][1]
        f, g = peaks_map(H, W, k0, seed, (0, c1)), peaks_map(H, W, k1, seed + 1, (c1, W))
        return np.maximum(f, g)
    if kind == "pits":
        return pits_map(H, W, arg, aligned16, seed)
    if kind == "pits_all":
        ys, xs = np.mgrid[0:H:2, 0:W:2]
        f = _ramp(H, W)
        f[ys, xs] = (-2.0 + np.random.default_rng(seed).random(ys.shape)).astype(F32)
        return f
    if kind == "runs":
        return isolated_runs(H, W, arg[0], seed)
    if kind == "runs_all":
        f = isolated_runs(H, W, H * W // 2, seed, interior=False)
        ys, xs = np.nonzero(f)
        drop = H * W // 2 - arg[0]
        f[ys[:drop], xs[:drop]] = 0.0
        return f
    if kind in ("third_last", "third_first"):
        f = isolated_runs(H, W, arg[0], seed)
        if kind == "third_last":
            f[-1, -1] = 0.5
        else:
            f[0, 1] = 0.5
        return f
    raise ValueError(kind)


@functools.lru_cache(maxsize=None)
def case_maps(name):
    c = CASE_BY_NAME[name]
    return np.stack([build(s, c["H"], c["W"], c["dim"], c["offset"] == 0, 11 * i + 7) for i, s in enumerate(c["maps"])])


@functools.lru_cache(maxsize=None)
def case_paths(name):
    """Per map: K per band, and the paths of persistence_pairs and of topo_loss (default, and each option set)."""
    c = CASE_BY_NAME[name]
    H, W, dim, al = c["H"], c["W"], c["dim"], c["offset"] == 0
    out = []
    for f in case_maps(name):
        Ks = level0(f, dim, al) if small_kernel(H, W, dim) else [0]
        b = binary_outcome(f, al) if dim == 1 and small_kernel(H, W, dim) else "off"
        runs = {"pairs": path(H, W, dim, Ks, al, "pairs", (), b)}
        if c["loss"]:
            for opts in _loss_routes(name):
                runs[("loss",) + opts] = path(H, W, dim, Ks, al, "loss", opts, b)
            if c["kst"]:
                runs[("loss", "OPT_WORST_CASE_WORKSPACE")] = path(H, W, dim, Ks, al, "loss", ("OPT_WORST_CASE_WORKSPACE",), b)
        out.append((Ks, runs))
    return out


def _two_valued(name):
    return any(len(np.unique(f)) <= 2 for f in case_maps(name))


def _loss_routes(name):
    r = [(), ("OPT_NO_FUSED_GRAD",), ("OPT_NO_FUSED_MATCH",)]
    if CASE_BY_NAME[name]["dim"] == 1 and _two_valued(name) and small_kernel(CASE_BY_NAME[name]["H"], CASE_BY_NAME[name]["W"], 1):
        r.append(("OPT_NO_BINARY_PATH",))
    return r


def reached():
    merge, binary = {}, {}
    for c in CASES:
        for Ks, runs in case_paths(c["name"]):
            for run, p in runs.items():
                if p.kernel == "global" or p.binary not in ("vec", "scalar"):
                    if p.kernel != "global":
                        merge.setdefault(merge_tuple(c["dim"], p), []).append((c["name"], run))
                if c["dim"] == 1:
                    binary.setdefault((p.kernel, p.binary), []).append((c["name"], run))
    return merge, binary


# ------------------------------------------------------------------ CPU tests

def test_model_pins_match_the_sources():
    for fname, texts in PINS.items():
        src = _src(os.path.normpath(os.path.join(CSRC, fname)))
        for t in texts:
            assert t in src, f"{fname} no longer contains {t!r}: update the path model"
    assert CROSS_EDGE == 16 and TENTRY == 16
    assert (K_SMALL_MAX_ROW, K_PH_THREADS, K_RING) == (4097, 1024, 64)
    assert RING_BYTES == 32768 and T_CAP_SMEM == K_SMALL_SMEM // 16
    # the fast front end's H <= 16383 is implied by the row limit
    assert K_SMALL_MAX_ROW - 1 <= 16383
    # 4096 x 16 and 16 x 4096 hold 65536 pixels: one band, with the OUTSIDE alias.  At H = 4096 fast bands are 12
    # columns wide (4096 x 28: 12 + 12 + 4), generic ones 15; H0 at (H + 1)(W + 1) = 65536: bands of 255 + 1
    assert bands(4096, 16, 1, True) == [(0, 16)] and bands(16, 4096, 1, False) == [(0, 4096)]
    assert bands(4096, 28, 1, True) == [(0, 12), (12, 12), (24, 4)] and bands(4096, 28, 1, False) == [(0, 15), (15, 13)]
    assert bands(255, 255, 0, True) == [(0, 255), (255, 1)] and bands(4096, 16, 0, True) == [(0, 15), (15, 2)]


def test_thresholds_sit_where_the_model_puts_them():
    t = _th()
    # single band, Pbits == 18: the shared-memory budget ends the packed form before the 14 target bits do
    assert (256 * 513 + 256).bit_length() == 18 and t["pk256"] < 1 << 14 and t["pk256"] + 1 > T_CAP_SMEM
    assert t["rp256"] < t["pk256"] and path(256, 256, 1, t["rp256"]).rp == "global"
    assert path(256, 256, 1, t["rp256"] - 1).rp == "smem16" and path(256, 256, 1, t["pk256"]).table == "global128"
    # 364 x 365, Pbits == 19: 13 bits of basin id; then the 128-bit shared table, then the spill
    assert path(364, 365, 1, t["pk365"] - 1).table == "packed" and path(364, 365, 1, t["pk365"]).table == "smem128"
    assert path(364, 365, 1, T_CAP_SMEM - 1).table == "smem128" and path(364, 365, 1, T_CAP_SMEM).table == "global128"
    assert path(364, 365, 1, t["ks364"] - 2, api="loss").kst is False and path(364, 365, 1, t["ks364"] - 1, api="loss").kst
    assert not path(364, 365, 1, t["ks364"] - 1, api="pairs").kst
    assert binary_r_cap(1188, 1024) == (True, 85) and not binary_r_cap(1189, 1024)[0]
    assert binary_r_cap(256, 512) == (True, 65535)
    assert n_nodes(1778, 2359, 1) == (1 << 22) - 1 and small_kernel(1778, 2359, 1)
    assert n_nodes(2047, 2049, 1) == 1 << 22 and not small_kernel(2047, 2049, 1)
    assert n_nodes(2046, 2048, 0) == (1 << 22) - 1 and small_kernel(2046, 2048, 0) and not small_kernel(2047, 2047, 0)
    assert not small_kernel(4097, 8, 1) and small_kernel(4096, 16, 1)


@pytest.mark.parametrize("H,W", [(9, 12), (40, 52), (31, 33), (130, 600), (600, 130), (256, 256), (255, 257)])
def test_level0_model_on_peaks(H, W):
    rng = np.random.default_rng(H * W)
    for K in sorted({0, 1, 7, int(rng.integers(1, (H - 2) * (W - 2) // 2 + 1)), ((H - 2) * (W - 2) + 1) // 2}):
        f = peaks_map(H, W, K, seed=K)
        for al in (True, False):
            assert sum(level0(f, 1, al)) == K, (H, W, K, al, level0(f, 1, al))
        if H * W <= 70000:
            assert len(oracle.cubical_pairs(f, 1)) == K


@pytest.mark.parametrize("H,W", [(9, 12), (40, 52), (31, 33), (130, 600), (600, 130), (254, 256), (364, 364)])
def test_level0_model_on_pits(H, W):
    nb = len(bands(H, W, 0, True))
    n_sites = len(pits_sites(H, W, bands(H, W, 0, True))[0])
    for P in sorted({0, 1, 5, n_sites // 3, n_sites}):
        f = pits_map(H, W, P, seed=P)
        assert sum(level0(f, 0)) == P + nb, (H, W, P, nb, level0(f, 0))
        if H * W <= 70000:
            assert len(oracle.cubical_pairs(f, 0)) == P + 1


def test_feasible_sets_and_rules():
    assert all(any(rule(*t) for t in itertools.product(*MERGE_AXES)) for _, rule in MERGE_RULES)
    assert all(any(rule(*t) for t in itertools.product(*BINARY_AXES)) for _, rule in BINARY_RULES)
    # the model never produces a combination a rule calls impossible, over a wide sweep of shapes and K
    rng = np.random.default_rng(0)
    shapes = [(256, 256), (255, 257), (252, 255), (252, 256), (364, 365), (257, 259), (256, 260), (4096, 16),
              (16, 4096), (254, 256), (255, 255), (364, 364), (1778, 2359), (1188, 1024), (60, 60), (2, 65536 // 2)]
    for H, W in shapes:
        for dim in (0, 1):
            if not small_kernel(H, W, dim):
                continue
            for al in (True, False):
                nb = len(bands(H, W, dim, al))
                for K in list(rng.integers(0, n_nodes(H, W, dim) // 2, 40)) + [0, 8190, 8191, 12224, 13970, 14271,
                                                                              14272, 16297, 16298, 16383]:
                    if K > n_nodes(H, W, dim) // 2:  # more basins than the nodes can give
                        continue
                    Kb = [int(K) // nb] * nb
                    for api in ("pairs", "loss"):
                        p = path(H, W, dim, Kb, al, api)
                        assert merge_tuple(dim, p) in FEASIBLE_MERGE, (H, W, dim, al, K, api, p)


def test_gpu_cases_cover_every_feasible_branch():
    merge, binary = reached()
    assert set(merge) <= FEASIBLE_MERGE, sorted(set(merge) - FEASIBLE_MERGE, key=str)
    missing = FEASIBLE_MERGE - set(merge)
    assert not missing, "\n".join(map(str, sorted(missing, key=str)))
    assert set(binary) <= FEASIBLE_BINARY, sorted(set(binary) - FEASIBLE_BINARY, key=str)
    assert FEASIBLE_BINARY == set(binary), sorted(FEASIBLE_BINARY - set(binary), key=str)
    # global kernel reached naturally (no OPT_FORCE_GLOBAL_KERNEL in any case)
    kernels = {p.kernel for c in CASES for _, runs in case_paths(c["name"]) for p in runs.values()}
    assert kernels == {"single", "multi", "global"}


def test_cases_sit_on_their_thresholds():
    """Every designed map has the K it was built for, and each threshold has a case on either side of it."""
    t = _th()
    seen = {}
    for c in CASES:
        for spec, (Ks, runs) in zip(c["maps"], case_paths(c["name"])):
            if spec[0] == "peaks" and small_kernel(c["H"], c["W"], 1):
                assert sum(Ks) == spec[1], (c["name"], spec, Ks)
            if spec[0] == "pits" and small_kernel(c["H"], c["W"], 0):
                assert sum(Ks) >= spec[1], (c["name"], spec, Ks)
            seen.setdefault((c["H"], c["W"], c["dim"]), set()).add(sum(Ks))
        for (Ks, runs), f in zip(case_paths(c["name"]), case_maps(c["name"])):
            if c["kst"] and Ks[0] > 1000:
                assert runs[("loss",)].kst and not runs["pairs"].kst and not runs[("loss", "OPT_WORST_CASE_WORKSPACE")].kst
    s = seen[(256, 256, 1)]
    assert {t["rp256"] - 1, t["rp256"], t["pk256"] - 1, t["pk256"]} <= s
    assert {t["pk365"] - 1, t["pk365"], T_CAP_SMEM - 2, T_CAP_SMEM - 1, t["ks364"] - 2, t["ks364"] - 1} <= seen[(364, 365, 1)]
    assert {t["rp259"] - 1, t["rp259"]} <= seen[(260, 257, 1)]
    assert {t["ks260"] - 2, t["ks260"] - 1} <= seen[(256, 260, 1)]
    outcomes = {c["name"]: [r["pairs"].binary for _, r in case_paths(c["name"])] for c in CASES if c["name"].startswith("bin_")}
    assert outcomes["bin_256x512_runs"] == ["vec", "reject_runs"]
    assert outcomes["bin_256x512_runs_scalar"] == ["scalar", "reject_runs"]
    assert outcomes["bin_1188x1024_runs"] == ["vec", "reject_runs"]
    assert outcomes["bin_1189x1024_mask"] == ["reject_mask", "reject_mask"]
    assert outcomes["bin_256x256_vec"] == ["vec", "reject_values_late", "reject_values_probe"]


# ------------------------------------------------------------------ GPU tests

def _device_maps(maps, offset, shape):
    """The maps as a CUDA tensor of ``shape`` whose storage starts ``offset`` floats into its buffer."""
    flat = torch.zeros(maps.size + offset + 4, dtype=torch.float32, device="cuda")
    flat[offset:offset + maps.size] = torch.from_numpy(np.ascontiguousarray(maps).ravel()).cuda()
    t = flat[offset:offset + maps.size].view(*shape)
    assert t.is_contiguous() and t.data_ptr() % 16 == 4 * offset
    return flat, t


def _with_options(opts, fn):
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    ids = [getattr(_lib, o) for o in opts]
    old = [L.tl_get_option(i) for i in ids]
    for i in ids:
        assert L.tl_set_option(i, 1) == 0
    try:
        return fn()
    finally:
        for i, v in zip(ids, old):
            L.tl_set_option(i, v)


def _loss(maps, truth, dim, offset, backward=True):
    """topo_loss over [n, 1] maps whose kernel view is the H x W map (a non-square batch is passed as [n, 1, W, H]:
    the reference reads its flat buffer as W rows of H pixels, i.e. as our H x W maps)."""
    import dilabhelmholtzoct_b200 as tlb
    n, H, W = maps.shape
    shape = (n, 1, W, H)
    buf, p = _device_maps(maps, offset, shape)
    buf.requires_grad_(True)
    p = buf[offset:offset + maps.size].view(*shape)
    t = torch.from_numpy(truth.reshape(shape)).cuda()
    loss = tlb.topo_loss(p, t, LAMDA, feat_d=dim, loss_q=2)
    if not backward:  # (the backward would raise on the status of its own forward)
        torch.cuda.synchronize()
        return float(loss.detach()), None
    loss.backward()
    torch.cuda.synchronize()
    return float(loss.detach()), buf.grad[offset:offset + maps.size].cpu().numpy().reshape(maps.shape)


def _truth(name):
    c = CASE_BY_NAME[name]
    return np.stack([blobs_truth(c["H"], c["W"], 4, i) for i in range(len(c["maps"]))])


@functools.lru_cache(maxsize=None)
def _oracle_loss(name):
    c = CASE_BY_NAME[name]
    maps, truth = case_maps(name), _truth(name)
    n, H, W = maps.shape
    want, wgrad, _ = oracle.topo_loss(maps.reshape(n, 1, W, H), truth.reshape(n, 1, W, H), LAMDA, feat_d=c["dim"],
                                      loss_q=2, nthreads=os.cpu_count() or 1)
    return want, wgrad.reshape(maps.shape)


def _check_loss(name, got, grad, route):
    want, wgrad = _oracle_loss(name)
    assert abs(got - want) <= REL * abs(want) + 1e-12, (name, route, got, want)
    scale = np.abs(wgrad).max()
    if _two_valued(name):
        # a two-valued prediction has identical diagram points: which of them the matching takes is a tie, and the
        # kernels break it in their emission order, not the oracle's.  The gradient's values do not depend on it
        grad, wgrad = np.sort(grad.ravel()), np.sort(wgrad.ravel())
    assert np.abs(grad - wgrad).max() <= REL * scale + 1e-12, (name, route, np.abs(grad - wgrad).max(), scale)
    assert np.array_equal(grad != 0, wgrad != 0), (name, route, "critical pixels differ")


@pytest.fixture
def roomy_arena():
    """Maps with tens of thousands of pairs need more than the default pair arena (~N/5 records per map)."""
    from dilabhelmholtzoct_b200 import topological_loss as tlmod
    old = tlmod._ARENA_FACTOR
    tlmod.set_arena_factor(4.0)
    try:
        yield
    finally:
        tlmod._ARENA_FACTOR = old


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_persistence_paths(name, roomy_arena):
    import dilabhelmholtzoct_b200 as tlb
    c = CASE_BY_NAME[name]
    maps, dim, offset = case_maps(name), c["dim"], c["offset"]
    n, H, W = maps.shape
    _, dev = _device_maps(maps, offset, (n, H, W))
    got = [p.cpu().numpy() for p in tlb.persistence_pairs(dev, dim)]
    for k, f in enumerate(maps):
        want = oracle.cubical_pairs(f, dim)
        assert got[k].shape == want.shape and np.array_equal(got[k], want), (name, k, got[k].shape, want.shape)
    if not c["loss"] or n < 2:
        return
    truth = _truth(name)
    for opts in _loss_routes(name):
        tlb.check_status(sync=True)
        if any(runs[("loss",) + opts].kst for _, runs in case_paths(name)):
            # the loss's basin tables run out: NaN, a status naming them, and the oracle's loss with the worst case
            loss, _ = _with_options(opts, lambda: _loss(maps, truth, dim, offset, backward=False))
            assert np.isnan(loss), (name, opts, loss)
            with pytest.raises(RuntimeError, match="basin tables"):
                tlb.check_status(sync=True)
            opts = opts + ("OPT_WORST_CASE_WORKSPACE",)
        loss, grad = _with_options(opts, lambda: _loss(maps, truth, dim, offset))
        tlb.check_status(sync=True)
        _check_loss(name, loss, grad, opts)
