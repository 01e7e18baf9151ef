"""CPU restatement of the step in front of the topological loss at the reference call site --
TEST INFRASTRUCTURE ONLY (same rules as the rest of oracle/).

    topo_loss(torch.sigmoid(masks.float()), gt_masks.float(), 0.1, feat_d=1, interp=50)
        /root/reference/octsam/models/training_utils.py:64
    F.interpolate(x, size=(interp, interp), mode='bilinear', align_corners=True)
        /root/reference/octsam/models/topological_loss.py:33-46

PARITY PINNED: the reference's implementation of this step is PyTorch itself (torch.sigmoid,
F.interpolate), importable in this container; tests/test_resample.py checks this restatement against it
on CPU, and tests/golden/resample_small.npz holds vectors generated from it (make_golden_resample.py).
Arithmetic in float32, following ATen's upsample_bilinear2d (align_corners=True).
"""
from __future__ import annotations

import numpy as np


def _axis(n_in: int, n_out: int):
    f32 = np.float32
    scale = f32(n_in - 1) / f32(n_out - 1) if n_out > 1 else f32(0)
    src = (scale * np.arange(n_out, dtype=np.float32)).astype(np.float32)
    i0 = src.astype(np.int64)
    i1 = i0 + (i0 < n_in - 1)
    l1 = (src - i0.astype(np.float32)).astype(np.float32)
    l0 = (f32(1) - l1).astype(np.float32)
    return i0, i1, l0, l1


def sigmoid(x):
    x = np.asarray(x, dtype=np.float32)
    return (np.float32(1) / (np.float32(1) + np.exp(-x, dtype=np.float32))).astype(np.float32)


def resample(x, size: int, apply_sigmoid: bool = False) -> np.ndarray:
    """[..., H, W] float32 -> [..., size, size]: bilinear(align_corners=True) of (sigmoid(x) | x)."""
    x = np.asarray(x, dtype=np.float32)
    H, W = x.shape[-2:]
    v = sigmoid(x) if apply_sigmoid else x
    y0, y1, ly0, ly1 = _axis(H, size)
    x0, x1, lx0, lx1 = _axis(W, size)
    ly0, ly1 = ly0[:, None], ly1[:, None]
    top = lx0 * v[..., y0, :][..., :, x0] + lx1 * v[..., y0, :][..., :, x1]
    bot = lx0 * v[..., y1, :][..., :, x0] + lx1 * v[..., y1, :][..., :, x1]
    return (ly0 * top + ly1 * bot).astype(np.float32)


def resample_backward(grad_out, x, apply_sigmoid: bool = False) -> np.ndarray:
    """Gradient of ``resample`` w.r.t. ``x`` (float64 accumulation, cast to float32)."""
    x = np.asarray(x, dtype=np.float32)
    g = np.asarray(grad_out, dtype=np.float64)
    H, W = x.shape[-2:]
    S = g.shape[-1]
    y0, y1, ly0, ly1 = _axis(H, S)
    x0, x1, lx0, lx1 = _axis(W, S)
    gin = np.zeros(x.shape, dtype=np.float64)
    flat = gin.reshape(-1, H, W)
    gf = g.reshape(-1, S, S)
    for (ys, wy) in ((y0, ly0), (y1, ly1)):
        for (xs, wx) in ((x0, lx0), (x1, lx1)):
            w = wy[:, None].astype(np.float64) * wx[None, :].astype(np.float64)
            for m in range(flat.shape[0]):
                np.add.at(flat[m], (ys[:, None].repeat(S, 1), xs[None, :].repeat(S, 0)), w * gf[m])
    if apply_sigmoid:
        s = sigmoid(x).astype(np.float64)
        gin *= s * (1.0 - s)
    return gin.astype(np.float32)


# ------------------------------------------------------------------ F3: SAM post-processing chain

def _axis_half_pixel(n_in: int, n_out: int, fused: bool = False):
    """ATen upsample_bilinear2d, align_corners=False: scale = in / out, src = max(0, scale (dst + .5) - .5).

    ``fused``: round ``scale (dst + .5) - .5`` once, as a fused multiply-add.  nvcc contracts it so in the F3
    kernels and in ATen's CUDA kernel; the two roundings of the default differ from it by one ulp of ``src`` at a
    few positions when ``scale`` is not a power of two."""
    f32 = np.float32
    scale = f32(n_in) / f32(n_out)
    half = np.arange(n_out, dtype=np.float32) + f32(0.5)
    if fused:  # the float64 product of two fp32 values and the subtraction of .5 are exact here
        src = (np.float64(scale) * half.astype(np.float64) - 0.5).astype(np.float32)
    else:
        src = (scale * half - f32(0.5)).astype(np.float32)
    src = np.maximum(src, f32(0)).astype(np.float32)
    i0 = src.astype(np.int64)
    i1 = i0 + (i0 < n_in - 1)
    l1 = (src - i0.astype(np.float32)).astype(np.float32)
    l0 = (f32(1) - l1).astype(np.float32)
    return i0, i1, l0, l1


def interpolate_half_pixel(x, out_h: int, out_w: int) -> np.ndarray:
    """F.interpolate(x, (out_h, out_w), mode='bilinear', align_corners=False) on [..., H, W] float32."""
    x = np.asarray(x, dtype=np.float32)
    H, W = x.shape[-2:]
    y0, y1, ly0, ly1 = _axis_half_pixel(H, out_h)
    x0, x1, lx0, lx1 = _axis_half_pixel(W, out_w)
    ly0, ly1 = ly0[:, None], ly1[:, None]
    top = lx0 * x[..., y0, :][..., :, x0] + lx1 * x[..., y0, :][..., :, x1]
    bot = lx0 * x[..., y1, :][..., :, x0] + lx1 * x[..., y1, :][..., :, x1]
    return (ly0 * top + ly1 * bot).astype(np.float32)


def postprocess(x, T: int, rh: int, rw: int, oh: int, ow: int) -> np.ndarray:
    """training_utils.py:57-59: upsample to T x T, crop to [rh, rw], resample to [oh, ow]."""
    return interpolate_half_pixel(interpolate_half_pixel(x, T, T)[..., :rh, :rw], oh, ow)


# ------------------------------------------------------------------ float64 references (dense weight matrices)
# Bilinear resampling is separable and linear: along one axis it is an [n_out, n_in] matrix whose row o holds
# the two tap weights of output o.  The taps and weights are ATen's float32 ones (_axis / _axis_half_pixel), so
# the matrix is exactly the operation the fp32 kernels compute; only the products and sums are done in float64.
# (Sampling positions computed in float64 would be a different operation: src moves by up to src * eps32.)

def axis_matrix(n_in: int, n_out: int, align_corners: bool, fused: bool = False) -> np.ndarray:
    """[n_out, n_in] float64 weights of one axis of F.interpolate(mode='bilinear') (``fused``: see _axis_half_pixel)."""
    i0, i1, l0, l1 = _axis(n_in, n_out) if align_corners else _axis_half_pixel(n_in, n_out, fused)
    m = np.zeros((n_out, n_in), dtype=np.float64)
    r = np.arange(n_out)
    np.add.at(m, (r, i0), l0.astype(np.float64))
    np.add.at(m, (r, i1), l1.astype(np.float64))
    return m


def postprocess_axis_matrix(n_src: int, T: int, r: int, n_out: int, fused: bool = False) -> np.ndarray:
    """[n_out, n_src] float64 weights of one axis of ``postprocess``: A2 . A1[:r] (up to T, crop to r, to n_out)."""
    return axis_matrix(r, n_out, False, fused) @ axis_matrix(n_src, T, False, fused)[:r]
