"""Edge shapes of the three fused kernels around the topological loss, against float64 references.

* F1 -- ``resample_kernel.cuh``: sigmoid + bilinear resample (align_corners=True), ``tlb.resample``;
* F3 -- the ``postprocess_*`` kernels: SAM's 256^2 -> T^2 -> crop -> original-size chain, ``tlb.postprocess_masks``;
* F2 -- ``dice_ce_kernel.cuh``: DiceCELoss(sigmoid=True), ``tlb.dice_ce_loss``.

References.  Bilinear resampling is separable and linear, so along each axis it is a dense float64 matrix built
from ATen's float32 taps and weights (``oracle.resample_oracle.axis_matrix``): F1 is ``Ay . sigmoid(X) . Ax^T``,
F3 is the same with ``A = A2 . A1[:r]`` per axis, and both backwards are ``Ay^T . G . Ax``.  F2's reference is
``oracle.dice_ce_oracle.dice_ce`` on float64 tensors with autograd.

Error bounds are per element, not relative to the largest entry (which hides a wrong value on a pixel with a
small gradient).  Every bilinear weight is non-negative, so an fp32 evaluation of an output is off by at most
``c * eps32 * (the same operation applied to |x|)``; for a gradient entry ``c * eps32 * (Ay^T |G| Ax)``.  ``c``
absorbs the rounding of the taps' products and of the sums (atomics make the order of the latter vary), see
the C_* constants below for how they were chosen.

The CPU part checks the float64 references against the fp32 oracle and PyTorch on the CPU, and checks with a
model of the kernels' host dispatch and capacity tests (constants read from the .cuh / .cu sources) that the
GPU case lists below reach every code path: a retuned constant that drops a path out of the suite fails here.
The GPU part (-m gpu) runs the cases, plus "fully overwritten, nothing past the end" checks through the C ABI.
"""
import ctypes
import math
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import resample_oracle as ro
from oracle.dice_ce_oracle import dice_ce

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dilabhelmholtzoct_b200", "csrc")

EPS = float(np.finfo(np.float32).eps)     # 2^-23
TINY = float(np.finfo(np.float32).tiny)   # smallest normal fp32: absolute floor for values that underflow

# c of the per-element bounds, calibrated once on a B200 (1000 W power limit; CUDA 12.9, torch 2.11) over the case
# lists of this file.  Largest c seen, kernel / torch-CUDA fp32 (same operation, its own rounding and sum order):
#   F1 forward 2.2 / 2.2, backward 1.4 / 1.4;  F3 forward 1.9 / 1.9, gather backward 1.8 / 5.7 (torch scatters),
#   scatter backward 5.3 / 1.0;  F2 gradient 4.1 with expf, 31 with the __expf intrinsic (saturated_60), loss 0.2.
# (Calibrated with F3's geometry rounded twice, the F3 forward needed c = 112 for kernel and torch alike: both round
# scale (dst + .5) - .5 once, see oracle.resample_oracle._axis_half_pixel.)  The constants leave about 2x of margin
# for the order of atomics; C_F2 = 8 is what separates expf from __expf.
C_F1 = 8            # F1 forward and backward
C_F3 = 8            # F3 forward (two rounded stages of 2 x 2 taps) and gather backward (<= kGK taps per axis)
C_F3_SCATTER = 16   # F3 scatter backward: a source pixel collects up to hundreds of shared / global atomics
C_TORCH = 32        # torch-CUDA fp32 against the same float64 reference: shows that it is the same operation
C_F2 = 8            # F2 loss and gradient
F2_SLICE_RTOL = 1e-5  # F2 gradient per (b, c) slice, relative to that slice's own largest entry


# ------------------------------------------------------------------ constants of the kernels, read from the source

def _int_expr(expr, known):
    expr = re.sub(r"[A-Za-z_]\w*", lambda m: str(known[m.group(0)]), expr.strip())
    assert re.fullmatch(r"[\d\s*+\-()/]+", expr), expr
    return int(eval(expr))  # digits and + - * / ( ) only, checked above


def _constexprs(name):
    """{name: value} of the ``constexpr int`` declarations of one CUDA source."""
    with open(os.path.join(CSRC, name)) as f:
        text = f.read()
    out = {}
    for decl in re.findall(r"constexpr\s+int\s+([^;]+);", text):
        for item in decl.split(","):
            k, v = item.split("=")
            out[k.strip()] = _int_expr(v, out)
    return out


def _grid_caps():
    """Grid caps of the host launchers in topoloss_api.cu (CTAs, or map lanes for the F3 gather)."""
    with open(os.path.join(CSRC, "topoloss_api.cu")) as f:
        src = f.read()
    pats = {
        "grid_for": r"int grid_for\(.*?cap = (\d+)ll \* (\d+);",
        "post_fwd": r"f_cap = (\d+)ll \* (\d+);",
        "gather_lanes": r"int lanes = \((\d+) \* (\d+) \+ classes - 1\) / classes;",
        "scatter": r"cap = (\d+)ll \* (\d+);\s*tl::postprocess_bwd_kernel<<<",
        "dice_ce": r"cap = (\d+)ll \* (\d+);\s*return \(int\)\(jobs",
    }
    caps = {}
    for k, p in pats.items():
        m = re.search(p, src, re.S)
        assert m, f"launcher of {k} not found in topoloss_api.cu: update the path model"
        caps[k] = int(m.group(1)) * int(m.group(2))
    return caps


K = {**_constexprs("resample_kernel.cuh"), **_constexprs("dice_ce_kernel.cuh")}
CAPS = _grid_caps()


# ------------------------------------------------------------------ model of the dispatch and capacity checks

def _hp(n_in, n_out):
    i0, i1, _, _ = ro._axis_half_pixel(n_in, n_out, fused=True)   # the kernels' fused multiply-add geometry
    return i0, i1


def _post_ranges(n_src, T, r, n_out):
    """post_out_range of every source index: first output and count of the outputs whose taps may reach it."""
    Y0, Y1 = _hp(r, n_out)
    a0, a1 = _hp(n_src, T)
    src_lo, src_hi = a0[Y0], a1[Y1]   # monotone in the output index
    s = np.arange(n_src)
    lo = np.searchsorted(src_hi, s, side="left")
    hi = np.searchsorted(src_lo, s, side="right") - 1
    return lo, np.where(hi >= lo, hi - lo + 1, 0)


def _span(lo, n):
    m = n > 0
    return (int((lo[m] + n[m] - 1).max() - lo[m].min() + 1), int(n.max())) if m.any() else (0, 0)


def _zero_fill_paths(n, tag):
    paths = set()
    if n % 4:
        paths.add(f"{tag}:zero_fill_tail")
    if (n >> 2) > CAPS["grid_for"] * 256:
        paths.add(f"{tag}:zero_fill_stride")
    return paths


def f3_paths(Hs, Ws, T, rh, rw, oh, ow, n):
    """Code paths tl_postprocess_forward / tl_postprocess_backward take for one geometry."""
    paths = set()
    ftx, fty = -(-ow // K["kFwdCols"]), -(-oh // K["kFwdRows"])
    if n * ftx * fty > CAPS["post_fwd"]:
        paths.add("post_fwd:tile_stride")
    ky, kx = 2.0 * oh * T / (Hs * rh) + 3.0, 2.0 * ow * T / (Ws * rw) + 3.0
    if ky <= K["kGK"] and kx <= K["kGK"]:
        gcy, gtx = -(-Hs // K["kGRows"]), -(-Ws // K["kGT_X"])
        lanes = min(n, max(1, -(-CAPS["gather_lanes"] // (gcy * gtx))))
        if n > lanes:
            paths.add("gather:map_stride")
        if gcy > 1:
            paths.add("gather:row_chunks")
        if Ws % K["kGT_X"]:
            paths.add("gather:partial_col_tile")
        if Hs != Ws:
            paths.add("gather:non_square")
        xlo, xn = _post_ranges(Ws, T, rw, ow)
        ylo, yn = _post_ranges(Hs, T, rh, oh)
        for c0 in range(0, Ws, K["kGT_X"]):
            cols, kxm = _span(xlo[c0:c0 + K["kGT_X"]], xn[c0:c0 + K["kGT_X"]])
            col_fit = cols <= K["kGWC"] and kxm <= K["kGK"]
            for r0 in range(0, Hs, K["kGTileRows"]):   # kGRows is a multiple of kGTileRows: chunks align
                rows, kym = _span(ylo[r0:r0 + K["kGTileRows"]], yn[r0:r0 + K["kGTileRows"]])
                fits = col_fit and rows <= K["kGWR"] and kym <= K["kGK"]
                paths.add("gather:staged" if fits else "gather:direct")
        return paths
    paths |= _zero_fill_paths(n * Hs * Ws, "scatter")
    ty, tx = -(-oh // K["kPostTileY"]), -(-ow // K["kPostTileX"])
    if n * ty * tx > CAPS["scatter"]:
        paths.add("scatter:tile_stride")

    def extents(n_src, r, n_out, tile):
        Y0, Y1 = _hp(r, n_out)
        a0, a1 = _hp(n_src, T)
        o0 = np.arange(0, n_out, tile)
        o1 = np.minimum(n_out, o0 + tile) - 1
        return a1[Y1[o1]] - a0[Y0[o0]] + 1

    win = np.outer(extents(Hs, rh, oh, K["kPostTileY"]), extents(Ws, rw, ow, K["kPostTileX"]))
    if (win <= K["kPostWin"]).any():
        paths.add("scatter:window")
    if (win > K["kPostWin"]).any():
        paths.add("scatter:global")
    return paths


def f1_paths(n, H, W, S):
    paths = _zero_fill_paths(n * H * W, "resample")
    if n * S * S > CAPS["grid_for"] * 256:
        paths.add("resample:grid_stride")
    return paths


def f2_paths(B, C, HW):
    tile = K["kDcThreads"] * K["kDcPix"]
    tiles = -(-HW // tile)
    paths = set()
    if B * tiles > CAPS["dice_ce"]:
        paths.add("dice_ce:job_stride")   # a CTA reuses its shared accumulators for a second job
    if HW % tile:
        paths.add("dice_ce:partial_tile")
    if C == K["kDcMaxC"]:
        paths.add("dice_ce:max_channels")
    return paths


REQUIRED_PATHS = {
    "post_fwd:tile_stride", "gather:staged", "gather:direct", "gather:map_stride", "gather:row_chunks",
    "gather:partial_col_tile", "gather:non_square", "scatter:window", "scatter:global", "scatter:tile_stride",
    "scatter:zero_fill_tail",
    "resample:grid_stride", "resample:zero_fill_tail", "resample:zero_fill_stride",
    "dice_ce:job_stride", "dice_ce:partial_tile", "dice_ce:max_channels",
}

# ------------------------------------------------------------------ the GPU cases

# F3: (name, Hs, Ws, T, rh, rw, oh, ow, n_maps, sparse grad_out)
F3_CASES = [
    ("callsite_256_maps", 256, 256, 1024, 992, 1024, 496, 512, 256, False),   # forward tile + gather map strides
    ("original_1024sq", 256, 256, 1024, 1024, 1024, 1024, 1024, 3, False),    # every gather tile: direct fallback
    ("portrait_crop", 256, 256, 1024, 1024, 720, 640, 450, 4, False),
    ("original_above_T", 256, 256, 1024, 768, 1024, 1536, 2048, 2, False),    # scatter, shared-memory window
    ("scatter_global", 1024, 16, 1024, 1024, 1024, 8, 1500, 2, False),        # scatter, window too large on some tiles
    ("out_1x1", 256, 256, 1024, 1024, 1024, 1, 1, 3, False),
    ("out_1xN", 64, 64, 256, 256, 200, 1, 300, 3, False),
    ("out_Nx1", 64, 64, 256, 200, 256, 300, 1, 3, False),
    ("src_300", 300, 300, 1024, 1000, 1024, 500, 512, 3, False),              # 2 row chunks, partial column tile
    ("src_520x200", 520, 200, 1024, 1024, 700, 333, 257, 2, False),           # 3 row chunks, non-square
    ("T_1000", 256, 256, 1000, 1000, 1000, 496, 512, 3, False),
    ("sparse_grad", 256, 256, 1024, 992, 1024, 496, 512, 4, True),            # the go == 0 skips
    ("upsample_small", 32, 32, 64, 64, 64, 700, 650, 2, False),
    ("odd_small", 41, 37, 256, 200, 256, 700, 650, 3, False),                 # scatter: zero-fill tail
]

# F1: (name, leading dims, H, W, S, sigmoid, logits)
F1_CASES = [
    ("S1", (3,), 37, 41, 1, True, "normal"),
    ("S2", (3,), 37, 41, 2, True, "normal"),
    ("S_H_minus_1", (3,), 40, 40, 39, True, "normal"),
    ("S_H", (3,), 40, 40, 40, True, "normal"),
    ("S_H_plain", (3,), 40, 40, 40, False, "normal"),
    ("upsample", (5,), 7, 9, 50, True, "normal"),
    ("upsample_plain", (5,), 7, 9, 50, False, "normal"),
    ("H_ne_W", (4,), 31, 77, 50, True, "normal"),
    ("map_1024sq", (2,), 1024, 1024, 50, True, "normal"),
    ("maps_896", (896,), 64, 64, 50, True, "normal"),                          # grid-stride, zero-fill stride
    ("lead_3d", (6,), 40, 44, 50, True, "normal"),
    ("lead_5d", (2, 2, 3), 40, 44, 50, True, "normal"),
    ("noncontiguous", (3,), 37, 41, 50, True, "noncontiguous"),
    ("logits_40", (3,), 33, 35, 50, True, "pm40"),
    ("logits_100", (3,), 33, 35, 50, True, "pm100"),
    ("logits_inf", (3,), 33, 35, 50, True, "pminf"),
]

# F2: (name, shape, targets, logits, upstream gradient)
F2_CASES = [
    ("C1", (2, 1, 50, 50), "binary", "normal", 1.0),
    ("C64", (2, 64, 33, 31), "binary", "normal", 1.0),
    ("HW1", (3, 5, 1, 1), "binary", "normal", 1.0),
    ("HW255", (3, 5, 15, 17), "binary", "normal", 1.0),
    ("HW2047", (3, 5, 23, 89), "binary", "normal", 1.0),
    ("HW2048", (3, 5, 32, 64), "binary", "normal", 1.0),
    ("HW2049", (3, 5, 2049), "binary", "normal", 1.0),
    ("callsite", (16, 14, 496, 512), "binary", "normal", 1.0),
    ("jobs_1280", (160, 2, 128, 128), "binary", "normal", 1.0),
    ("five_d", (2, 3, 4, 10, 12), "binary", "normal", -0.37),
    ("soft_targets", (2, 6, 40, 52), "soft", "normal", 1.0),
    ("multi_and_no_label", (2, 6, 40, 52), "multi", "normal", 2.5),
    ("saturated_15", (2, 6, 64, 64), "onehot_empty", "confident15", 1.0),
    ("saturated_30", (2, 6, 64, 64), "onehot_empty", "confident30", 1.0),
    ("saturated_60", (2, 6, 64, 64), "onehot_empty", "confident60", 1.0),
]


def _f3_case_paths():
    out = {}
    for name, Hs, Ws, T, rh, rw, oh, ow, n, _ in F3_CASES:
        for p in f3_paths(Hs, Ws, T, rh, rw, oh, ow, n):
            out.setdefault(p, name)
    return out


def covered_paths():
    """{path: first case that reaches it} over the three case lists."""
    out = _f3_case_paths()
    for name, lead, H, W, S, _, _ in F1_CASES:
        for p in f1_paths(math.prod(lead), H, W, S):
            out.setdefault(p, name)
    for name, shape, *_ in F2_CASES:
        for p in f2_paths(shape[0], shape[1], math.prod(shape[2:])):
            out.setdefault(p, name)
    return out


def test_constants_are_read_from_the_sources():
    for k in ("kGK", "kGWR", "kGWC", "kGRows", "kGT_X", "kGTileRows", "kPostWin", "kPostTileY", "kPostTileX",
              "kFwdCols", "kFwdRows", "kDcThreads", "kDcPix", "kDcMaxC"):
        assert K[k] > 0, k
    assert K["kGRows"] % K["kGTileRows"] == 0   # the model's tile loop assumes aligned row chunks
    assert set(CAPS) == {"grid_for", "post_fwd", "gather_lanes", "scatter", "dice_ce"}


def test_gpu_cases_reach_every_path():
    got = covered_paths()
    missing = REQUIRED_PATHS - set(got)
    assert not missing, f"no GPU case reaches {sorted(missing)}"


def test_path_model_examples():
    # the post-processing of the reference call site: the staged gather on every tile
    assert f3_paths(256, 256, 1024, 992, 1024, 496, 512, 6) == {"gather:staged"}
    # a 1024 x 1024 original: every tile beyond the staging buffers (direct-from-global gather)
    assert f3_paths(256, 256, 1024, 1024, 1024, 1024, 1024, 3) == {"gather:direct"}
    # up-sampling 32^2 -> 700 x 650: the scatter kernel, and every tile's window fits in shared memory
    p = f3_paths(32, 32, 64, 64, 64, 700, 650, 2)
    assert "scatter:window" in p and "scatter:global" not in p


# ------------------------------------------------------------------ CPU: float64 references against fp32 ones

def _np_units(got, ref, bnd):
    err = np.abs(got.astype(np.float64) - ref)
    with np.errstate(divide="ignore", invalid="ignore"):
        return float(np.nan_to_num(err / (EPS * bnd), nan=0.0).max())


@pytest.mark.parametrize("n_src,T,r,n_out", [(16, 64, 62, 31), (8, 32, 20, 33), (12, 24, 24, 7), (300, 1024, 1000, 500)])
def test_postprocess_axis_matrix_matches_fp32_oracle(n_src, T, r, n_out):
    A = ro.postprocess_axis_matrix(n_src, T, r, n_out)
    assert (A >= 0).all() and np.allclose(A.sum(1), 1.0, atol=1e-6)
    x = np.random.default_rng(n_src + r).standard_normal((2, n_src, 9)).astype(np.float32)
    Ax = ro.postprocess_axis_matrix(9, T, T // 2, 11)
    want = ro.postprocess(x, T, r, T // 2, n_out, 11)
    xd = x.astype(np.float64)
    assert _np_units(want, A @ xd @ Ax.T, A @ np.abs(xd) @ Ax.T) <= C_F3


@pytest.mark.parametrize("Hs,Ws,T,rh,rw,oh,ow", [(16, 20, 64, 62, 64, 31, 32), (8, 8, 32, 32, 20, 50, 33),
                                                 (12, 10, 24, 24, 24, 7, 9)])
def test_postprocess_reference_matches_pytorch_cpu(Hs, Ws, T, rh, rw, oh, ow):
    rng = np.random.default_rng(Hs * Ws + oh)
    x = (3.0 * rng.standard_normal((3, Hs, Ws))).astype(np.float32)
    g = rng.standard_normal((3, oh, ow)).astype(np.float32)
    Ay, Ax = ro.postprocess_axis_matrix(Hs, T, rh, oh), ro.postprocess_axis_matrix(Ws, T, rw, ow)
    t = torch.from_numpy(x).requires_grad_(True)
    y = F.interpolate(F.interpolate(t[None], (T, T), mode="bilinear", align_corners=False)[..., :rh, :rw],
                      (oh, ow), mode="bilinear", align_corners=False)[0]
    y.backward(torch.from_numpy(g))
    xd, gd = x.astype(np.float64), g.astype(np.float64)
    assert _np_units(y.detach().numpy(), Ay @ xd @ Ax.T, Ay @ np.abs(xd) @ Ax.T) <= C_TORCH
    assert _np_units(ro.postprocess(x, T, rh, rw, oh, ow), Ay @ xd @ Ax.T, Ay @ np.abs(xd) @ Ax.T) <= C_F3
    assert _np_units(t.grad.numpy(), Ay.T @ gd @ Ax, Ay.T @ np.abs(gd) @ Ax) <= C_TORCH


@pytest.mark.parametrize("H,W,S", [(9, 13, 5), (40, 40, 50), (7, 7, 1), (2, 3, 6), (31, 77, 50)])
def test_resample_reference_matches_fp32_oracle(H, W, S):
    rng = np.random.default_rng(H * W + S)
    x = (3.0 * rng.standard_normal((2, H, W))).astype(np.float32)
    g = rng.standard_normal((2, S, S)).astype(np.float32)
    Ay, Ax = ro.axis_matrix(H, S, True), ro.axis_matrix(W, S, True)
    assert (Ay >= 0).all() and np.allclose(Ay.sum(1), 1.0, atol=1e-6)
    xd, gd = x.astype(np.float64), g.astype(np.float64)
    for sig in (False, True):
        v = 1.0 / (1.0 + np.exp(-xd)) if sig else xd
        assert _np_units(ro.resample(x, S, sig), Ay @ v @ Ax.T, Ay @ np.abs(v) @ Ax.T) <= C_F1
        d = v * (1.0 - v) if sig else 1.0
        gbnd = Ay.T @ np.abs(gd) @ Ax * (v * (2.0 - v) if sig else 1.0)
        assert _np_units(ro.resample_backward(g, x, sig), (Ay.T @ gd @ Ax) * d, gbnd) <= C_F1
    if S == H == W:
        assert np.array_equal(ro.axis_matrix(H, S, True), np.eye(H))


def _f2_inputs(shape, targets, logits, seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    B, C = shape[:2]
    if logits == "normal":
        x = 3.0 * torch.randn(shape, generator=g)
    else:
        L = float(logits[len("confident"):])
        x = L * (1.0 + 0.1 * torch.rand(shape, generator=g))   # confident, saturated logits of either sign
    if targets == "binary":
        t = (torch.rand(shape, generator=g) < 0.3).float()
        t[:, -1] = 0.0                                         # a padded (empty) component mask
    elif targets == "soft":
        t = torch.rand(shape, generator=g)
        t = t / t.sum(1, keepdim=True)
        t[:, 0] *= (torch.rand(t[:, 0].shape, generator=g) < 0.5).float()   # some pixels with less than 1 in total
    elif targets == "multi":
        t = (torch.rand(shape, generator=g) < 0.4).float()     # several labels per pixel, some pixels with none
        t[:, 1] = 1.0                                          # an all-one channel
        t[:, -1] = 0.0
    else:  # onehot_empty: every pixel labelled by one of the first C // 2 channels, the rest empty
        lab = torch.randint(0, C // 2, (B, 1) + tuple(shape[2:]), generator=g)
        t = (torch.arange(C).view((1, C) + (1,) * (len(shape) - 2)) == lab).float()
    if logits != "normal":
        x = torch.where(t > 0, x, -x)                          # right and confident on every channel
    return x.to(device), t.to(device)


def f2_bounds(x, t, grad_scale, fp32_finish=False):
    """float64 reference loss and gradient of ``dice_ce(x, t) * grad_scale``, and their error bounds for c = 1.

    Loss: the Dice term of slice (b, c) is 1 - (2I + 1e-5) / (G + P + 1e-5) with I = sum s t, P = sum s,
    G = sum t, accumulated in fp32: relative errors of I, P, G move it by up to
    eps * (2I / den + (2I + 1e-5)(P + G) / den^2); the cross-entropy term of a pixel, ts (m + log S) - sum t x
    (m the largest logit, S the sum of exp(x - m), ts = sum t), loses eps * (ts (|m| + log S + E) + |sum t x|),
    where E = sum softmax |x - m| is the rounding of the exponents' arguments.  The kernel forms the ratio q and
    1 - q in float64; ``fp32_finish`` adds eps * (q + |1 - q|) for doing that in fp32 (PyTorch's fp32 evaluation).
    Gradient: w_dice (b - a t) s (1 - s) + w_ce (softmax ts - t) per element: the dice part is bounded by
    eps * w_dice (b + a t) s (the (1 - s) of an fp32 s near 1 is absolute, not relative), the CE part by
    eps * w_ce (softmax ts (1 + |x - m| + E) + t)."""
    xr = x.double().requires_grad_(True)
    td = t.double()
    want = dice_ce(xr, td)
    (grad_scale * want).backward()
    B, C = x.shape[:2]
    xd, td = xr.detach().reshape(B, C, -1), td.reshape(B, C, -1)
    HW = xd.shape[-1]
    s = torch.sigmoid(xd)
    I, P, G = (s * td).sum(-1), s.sum(-1), td.sum(-1)
    den = G + P + 1e-5
    q = (2 * I + 1e-5) / den
    dice_b = (2 * I / den + q * (P + G) / den + (q + (1 - q).abs() if fp32_finish else 0.0)).sum() / (B * C)
    m = xd.max(1, keepdim=True).values
    soft = torch.softmax(xd, 1)
    E = (soft * (xd - m).abs()).sum(1, keepdim=True)
    ts = td.sum(1, keepdim=True)
    lse = torch.logsumexp(xd, 1, keepdim=True)
    ce_b = (ts * (m.abs() + (lse - m) + E)).sum() + (td * xd).sum(1).abs().sum()
    loss_bound = dice_b + ce_b / (B * HW) + abs(float(want.detach()))   # the last term: the loss is returned in fp32
    g = abs(grad_scale)
    a, bb = (2.0 / den)[..., None], ((2 * I + 1e-5) / den ** 2)[..., None]
    grad_bound = g / (B * C) * (bb + a * td) * s + g / (B * HW) * (soft * ts * (1 + (xd - m).abs() + E) + td)
    return float(want.detach()), xr.grad.reshape(B, C, -1), float(abs(grad_scale) * loss_bound), grad_bound


def test_f2_bounds_hold_for_pytorch_cpu_fp32():
    """The F2 bounds are not tighter than fp32 arithmetic: PyTorch's own fp32 evaluation of the same loss
    meets them on the saturated and the mixed cases."""
    for name, shape, targets, logits, gs in F2_CASES:
        if math.prod(shape) > 100_000:
            continue
        x, t = _f2_inputs(shape, targets, logits, seed=7)
        xf = x.clone().requires_grad_(True)
        lf = dice_ce(xf, t)
        (gs * lf).backward()
        want, wgrad, lb, gb = f2_bounds(x, t, gs, fp32_finish=True)
        assert abs(float(lf.detach()) - want) <= C_F2 * EPS * lb + TINY, name
        B, C = shape[:2]
        err = (xf.grad.double().reshape(B, C, -1) - wgrad).abs()
        assert bool((err <= C_F2 * EPS * gb + TINY).all()), name


# ------------------------------------------------------------------ GPU helpers

def _units(got, ref, bnd, floor=0.0):
    """Smallest c with |got - ref| <= c * EPS * bnd + floor on every element (inf if an element with a zero
    bound is not exact); every output must be finite."""
    got = got.detach()
    assert bool(torch.isfinite(got).all()), "non-finite output"
    excess = ((got.double() - ref).abs() - floor).clamp_min(0.0)
    return float(torch.nan_to_num(excess / (EPS * bnd), nan=0.0, posinf=float("inf")).max())


def _torch_chain(x, T, rh, rw, oh, ow):
    m = F.interpolate(x, (T, T), mode="bilinear", align_corners=False)
    return F.interpolate(m[..., :rh, :rw], (oh, ow), mode="bilinear", align_corners=False)


def f3_units(case, seed=0):
    """c needed by the kernel's and by torch-CUDA's forward and backward for one F3 case."""
    import dilabhelmholtzoct_b200 as tlb
    name, Hs, Ws, T, rh, rw, oh, ow, n, sparse = case
    gen = torch.Generator(device="cuda").manual_seed(seed + Hs * 7 + ow)
    x = 3.0 * torch.randn((n, Hs, Ws), device="cuda", generator=gen)
    g = torch.randn((n, oh, ow), device="cuda", generator=gen)
    if sparse:
        g = g * (torch.rand((n, oh, ow), device="cuda", generator=gen) < 0.01)
    Ay = torch.from_numpy(ro.postprocess_axis_matrix(Hs, T, rh, oh, fused=True)).cuda()
    Ax = torch.from_numpy(ro.postprocess_axis_matrix(Ws, T, rw, ow, fused=True)).cuda()
    a = x.clone().requires_grad_(True)
    ya = tlb.postprocess_masks(a, (rh, rw), (oh, ow), padded_size=T)
    ya.backward(g)
    b = x.clone().requires_grad_(True)
    yb = _torch_chain(b[None], T, rh, rw, oh, ow)[0]
    yb.backward(g)
    xd, gd = x.double(), g.double()
    ref, bnd = Ay @ xd @ Ax.T, Ay @ xd.abs() @ Ax.T
    out = {"fwd": _units(ya, ref, bnd), "torch_fwd": _units(yb, ref, bnd)}
    del ref, bnd, ya, yb
    gref, gbnd = Ay.T @ gd @ Ax, Ay.T @ gd.abs() @ Ax
    out["bwd"], out["torch_bwd"] = _units(a.grad, gref, gbnd), _units(b.grad, gref, gbnd)
    out["scatter"] = not any(p.startswith("gather") for p in f3_paths(Hs, Ws, T, rh, rw, oh, ow, n))
    return out


def _f1_input(case, seed=0):
    name, lead, H, W, S, sig, logits = case
    gen = torch.Generator(device="cuda").manual_seed(seed + H * W + S)
    shape = tuple(lead) + (H, W)
    if logits == "noncontiguous":
        return (3.0 * torch.randn(shape[:-1] + (2 * W,), device="cuda", generator=gen))[..., ::2]
    x = 3.0 * torch.randn(shape, device="cuda", generator=gen)
    if logits.startswith("pm"):
        L = float(logits[2:])
        u = torch.rand(shape, device="cuda", generator=gen)
        x = torch.where(u < 0.3, torch.full_like(x, -L), torch.where(u < 0.6, torch.full_like(x, L), x))
    return x


def f1_units(case, seed=0):
    """c needed by the kernel's and by torch-CUDA's forward and backward for one F1 case."""
    import dilabhelmholtzoct_b200 as tlb
    name, lead, H, W, S, sig, logits = case
    x = _f1_input(case, seed)
    gen = torch.Generator(device="cuda").manual_seed(seed + 1)
    g = torch.randn(tuple(lead) + (S, S), device="cuda", generator=gen)
    a = x.clone().requires_grad_(True)   # clone() keeps the non-contiguous strides
    ya = tlb.resample(a, S, sigmoid=sig)
    ya.backward(g)
    assert ya.shape == tuple(lead) + (S, S) and a.grad.shape == x.shape
    b = x.detach().reshape(-1, H, W).clone().requires_grad_(True)
    yb = F.interpolate((torch.sigmoid(b) if sig else b)[None], size=(S, S), mode="bilinear", align_corners=True)[0]
    yb.backward(g.reshape(-1, S, S))
    Ay = torch.from_numpy(ro.axis_matrix(H, S, True)).cuda()
    Ax = torch.from_numpy(ro.axis_matrix(W, S, True)).cuda()
    xd, gd = x.detach().double().reshape(-1, H, W), g.double().reshape(-1, S, S)
    v = torch.sigmoid(xd) if sig else xd
    ref, bnd = Ay @ v @ Ax.T, Ay @ v.abs() @ Ax.T
    floor = TINY if sig else 0.0
    out = {"fwd": _units(ya.reshape(-1, S, S), ref, bnd, floor), "torch_fwd": _units(yb, ref, bnd, floor)}
    proj, pabs = Ay.T @ gd @ Ax, Ay.T @ gd.abs() @ Ax
    if sig:
        gref, gbnd = proj * v * (1.0 - v), pabs * v * (2.0 - v)   # s (1 - s), plus the absolute error of 1 - s
    else:
        gref, gbnd = proj, pabs
    out["bwd"] = _units(a.grad.reshape(-1, H, W), gref, gbnd, floor)
    out["torch_bwd"] = _units(b.grad, gref, gbnd, floor)
    if S == H == W and not sig:
        out["identity_exact"] = bool(torch.equal(ya, x))
    return out


def f2_units(case, seed=0):
    """c needed by the kernel's loss and gradient, and the largest per-(b, c)-slice relative gradient error."""
    import dilabhelmholtzoct_b200 as tlb
    name, shape, targets, logits, gs = case
    x, t = _f2_inputs(shape, targets, logits, seed=seed + sum(shape), device="cuda")
    want, wgrad, lb, gb = f2_bounds(x, t, gs)
    xg = x.clone().requires_grad_(True)
    loss = tlb.dice_ce_loss(xg, t)
    (gs * loss).backward()
    B, C = shape[:2]
    got = xg.grad.reshape(B, C, -1)
    assert bool(torch.isfinite(got).all()) and math.isfinite(float(loss.detach()))
    err = (got.double() - wgrad).abs()
    # per slice, relative to the slice's largest entry -- or to its fp32 resolution (its largest per-element bound)
    # where that is larger: on a channel that is right and saturated, s (1 - s) and softmax - t are below what fp32
    # resolves next to 1, in any fp32 evaluation
    scale = torch.maximum(wgrad.abs().amax(-1), C_F2 * EPS * gb.amax(-1) / F2_SLICE_RTOL)
    slice_rel = float(torch.nan_to_num(err.amax(-1) / scale, nan=0.0, posinf=float("inf")).max())
    return {"loss": max(0.0, abs(gs * float(loss.detach()) - gs * want) - TINY) / (EPS * lb) if lb > 0 else 0.0,
            "grad": _units(got, wgrad, gb, TINY), "slice_rel": slice_rel}


# ------------------------------------------------------------------ GPU tests

@pytest.mark.gpu
@pytest.mark.parametrize("case", F3_CASES, ids=[c[0] for c in F3_CASES])
def test_gpu_postprocess_edges(case):
    u = f3_units(case)
    assert u["fwd"] <= C_F3, u
    assert u["bwd"] <= (C_F3_SCATTER if u["scatter"] else C_F3), u
    assert u["torch_fwd"] <= C_TORCH and u["torch_bwd"] <= C_TORCH, u   # the reference is ATen's operation


@pytest.mark.gpu
@pytest.mark.parametrize("case", F1_CASES, ids=[c[0] for c in F1_CASES])
def test_gpu_resample_edges(case):
    u = f1_units(case)
    assert u["fwd"] <= C_F1 and u["bwd"] <= C_F1, u
    assert u["torch_fwd"] <= C_TORCH and u["torch_bwd"] <= C_TORCH, u
    assert u.get("identity_exact", True), "S = H = W without the sigmoid must return the input"


@pytest.mark.gpu
@pytest.mark.parametrize("case", F2_CASES, ids=[c[0] for c in F2_CASES])
def test_gpu_dice_ce_edges(case):
    u = f2_units(case)
    assert u["loss"] <= C_F2 and u["grad"] <= C_F2, u
    assert u["slice_rel"] <= F2_SLICE_RTOL, u


# ------------------------------------------------------------------ through the C ABI: every output element written,
# nothing written past the end.  Each output buffer is NaN-filled and followed by a guard region in the same
# allocation; afterwards no NaN may be left and the guard must be intact.

GUARD = 4096
SENTINEL = -12345.5


def _guarded(n, dtype=torch.float32):
    buf = torch.full((n + GUARD,), float("nan"), dtype=dtype, device="cuda")
    buf[n:] = SENTINEL
    return buf


def _check_guarded(buf, n, what):
    torch.cuda.synchronize()
    assert not bool(torch.isnan(buf[:n]).any()), f"{what}: output elements left unwritten"
    assert bool((buf[n:] == SENTINEL).all()), f"{what}: written past the end of the output"


@pytest.mark.gpu
@pytest.mark.parametrize("n,H,W,S,sig", [(3, 37, 41, 20, 1), (3, 37, 41, 50, 0), (2, 5, 3, 1, 1)])
def test_gpu_abi_resample_writes_every_output_once(n, H, W, S, sig):
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device="cuda").manual_seed(n * H + S)
    x = 3.0 * torch.randn((n, H, W), device="cuda", generator=gen)
    g = torch.randn((n, S, S), device="cuda", generator=gen)
    out = _guarded(n * S * S)
    _lib.check(L.tl_resample_forward(x.data_ptr(), n, H, W, S, sig, out.data_ptr(), st), "tl_resample_forward")
    _check_guarded(out, n * S * S, "tl_resample_forward")
    gin = _guarded(n * H * W)   # n * H * W % 4 == 3 for the first two: the zero fill's scalar tail
    _lib.check(L.tl_resample_backward(g.data_ptr(), x.data_ptr(), n, H, W, S, sig, gin.data_ptr(), st), "tl_resample_backward")
    _check_guarded(gin, n * H * W, "tl_resample_backward")
    a = x.clone().requires_grad_(True)
    y = F.interpolate((torch.sigmoid(a) if sig else a)[None], size=(S, S), mode="bilinear", align_corners=True)[0]
    y.backward(g)
    assert float((out[:n * S * S].view(n, S, S) - y).abs().max()) <= 1e-5
    assert float((gin[:n * H * W].view(n, H, W) - a.grad).abs().max()) <= 1e-5 * max(1.0, float(a.grad.abs().max()))


@pytest.mark.gpu
@pytest.mark.parametrize("Hs,Ws,T,rh,rw,oh,ow,n", [
    (72, 70, 256, 200, 230, 97, 115, 3),     # gather: crop (source pixels no output reads), partial column tile
    (41, 37, 256, 200, 256, 700, 650, 3),    # scatter: crop, zero-fill tail (n Hs Ws % 4 == 3)
    (256, 256, 1024, 1024, 1024, 1024, 1024, 1),  # gather, direct from global
])
def test_gpu_abi_postprocess_writes_every_output_once(Hs, Ws, T, rh, rw, oh, ow, n):
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device="cuda").manual_seed(Hs + ow)
    x = 3.0 * torch.randn((n, Hs, Ws), device="cuda", generator=gen)
    g = torch.randn((n, oh, ow), device="cuda", generator=gen)
    out = _guarded(n * oh * ow)
    _lib.check(L.tl_postprocess_forward(x.data_ptr(), n, Hs, Ws, T, rh, rw, oh, ow, out.data_ptr(), st), "tl_postprocess_forward")
    _check_guarded(out, n * oh * ow, "tl_postprocess_forward")
    gin = _guarded(n * Hs * Ws)
    _lib.check(L.tl_postprocess_backward(g.data_ptr(), n, Hs, Ws, T, rh, rw, oh, ow, gin.data_ptr(), st), "tl_postprocess_backward")
    _check_guarded(gin, n * Hs * Ws, "tl_postprocess_backward")
    b = x.clone().requires_grad_(True)
    y = _torch_chain(b[None], T, rh, rw, oh, ow)[0]
    y.backward(g)
    assert float((out[:n * oh * ow].view(n, oh, ow) - y).abs().max()) <= 1e-5 * max(1.0, float(y.abs().max()))
    assert float((gin[:n * Hs * Ws].view(n, Hs, Ws) - b.grad).abs().max()) <= 1e-5 * float(b.grad.abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,HW", [(3, 5, 2049), (2, 64, 1), (1, 1, 255)])
def test_gpu_abi_dice_ce_writes_every_output_once(B, C, HW):
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    x, t = _f2_inputs((B, C, HW), "binary", "normal", seed=B * C + HW, device="cuda")
    nb = ctypes.c_size_t(0)
    _lib.check(L.tl_dice_ce_workspace_bytes(B, C, ctypes.byref(nb)), "tl_dice_ce_workspace_bytes")
    n_ws = nb.value // 8
    ws = _guarded(n_ws, torch.float64)
    loss = _guarded(1)
    _lib.check(L.tl_dice_ce_forward(x.data_ptr(), t.data_ptr(), B, C, HW, ws.data_ptr(), loss.data_ptr(), st), "tl_dice_ce_forward")
    _check_guarded(loss, 1, "tl_dice_ce_forward")
    _check_guarded(ws, n_ws, "tl_dice_ce_forward workspace")
    gx = _guarded(B * C * HW)
    _lib.check(L.tl_dice_ce_backward(None, x.data_ptr(), t.data_ptr(), B, C, HW, ws.data_ptr(), gx.data_ptr(), st), "tl_dice_ce_backward")
    _check_guarded(gx, B * C * HW, "tl_dice_ce_backward")
    want, wgrad, _, _ = f2_bounds(x.cpu(), t.cpu(), 1.0)
    assert abs(float(loss[0]) - want) <= 1e-5 * abs(want)
    assert float((gx[:B * C * HW].cpu().double().view(B, C, -1) - wgrad).abs().max()) <= 1e-5 * float(wgrad.abs().max())
