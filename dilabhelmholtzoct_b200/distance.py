"""Exact Euclidean distance transform and the Hausdorff distance-transform loss, batched, on the GPU.

``distance_transform_edt(mask)`` is ``scipy.ndimage.distance_transform_edt`` for every ``[H, W]`` map of a bool or
uint8 CUDA tensor (``tl_edt``).  ``hausdorff_dt_loss(masks, gt_masks, alpha)`` is the Hausdorff distance-transform
loss of Karimi & Salcudean (IEEE TMI 2020) per ``(b, c)`` map of decoder logits, differentiable with respect to the
logits (``tl_hausdorff_dt_*``).  Both transforms of each map (prediction and target, foreground and background) run
in the same kernels as the loss; nothing goes through the host.  ``surface_distances(pred, target)`` gives the
boundary metrics of mask pairs -- Hausdorff distance, percentile Hausdorff distance, ASSD and normalized surface Dice
-- from the same transform measured at surface pixels (``tl_surface_distances``).

There is no CPU path: the inputs must be CUDA tensors.
"""
from __future__ import annotations

import ctypes
import math
from typing import NamedTuple

import torch
from torch.autograd.function import once_differentiable

from . import _lib
from .topological_loss import _stream_ptr

MAX_DIM = 4096


def _check_hw(H: int, W: int, what: str) -> None:
    if not (1 <= H <= MAX_DIM and 1 <= W <= MAX_DIM):
        raise ValueError(f"{what}: H and W must each be in [1, {MAX_DIM}], got {H} x {W}")


class SurfaceDistances(NamedTuple):
    """Per-map surface-distance metrics of ``surface_distances``: float32, shape ``pred.shape[:-2]``."""
    hausdorff: torch.Tensor
    hausdorff_percentile: torch.Tensor
    assd: torch.Tensor
    nsd: torch.Tensor


def surface_distances(pred: torch.Tensor, target: torch.Tensor, percentile: float = 95.0,
                      tolerance: float = 1.0) -> SurfaceDistances:
    """Boundary metrics of every ``[H, W]`` map pair of ``pred`` and ``target`` (``[..., H, W]``, same shape, bool or
    uint8, CUDA; a nonzero pixel is foreground): the Hausdorff distance, its ``percentile``-th percentile (HD95 by
    default), the average symmetric surface distance and the normalized surface Dice at ``tolerance`` pixels.  No
    autograd, no host synchronisation.

    Per map, the surface ``S(M) = M & ~scipy.ndimage.binary_erosion(M)`` (cross structure, outside = 0) is the
    foreground pixels with a background or outside 4-neighbour.  ``d_pt`` is the exact Euclidean distance (unit
    spacing) from each pixel of ``S(pred)`` to the nearest pixel of ``S(target)``, ``sqrt(float64(s))`` of an integer
    ``s``; ``d_tp`` the same the other way.  In fp64, rounded to float32::

        hausdorff            = max(max d_pt, max d_tp)
        hausdorff_percentile = max(np.percentile(d_pt, q), np.percentile(d_tp, q))      # numpy's linear method
        assd                 = (sum d_pt + sum d_tp) / (|S(pred)| + |S(target)|)
        nsd                  = (#{d_pt <= tolerance} + #{d_tp <= tolerance}) / (|S(pred)| + |S(target)|)

    ``hausdorff``, ``hausdorff_percentile`` and ``nsd`` equal that numpy / scipy computation in float64 rounded to
    float32 bit for bit; ``assd`` sums in another order and is within one float32 ulp of it.  Both masks empty: all
    four are NaN (an all-zero padded mask pair; reduce with ``nanmean``).  One mask empty: ``hausdorff``,
    ``hausdorff_percentile`` and ``assd`` are ``+inf`` and ``nsd`` is 0.  By recollection this is monai's
    ``get_mask_edges`` with ``compute_hausdorff_distance``, ``compute_average_surface_distance(symmetric=True)`` and
    ``compute_surface_dice``; monai is not a dependency, so that parity is unpinned.

    ``percentile`` is in [0, 100], ``tolerance`` finite and >= 0, H and W each in [1, 4096].  About 16 bytes per pixel
    of scratch are taken from PyTorch's caching allocator for the duration of the call."""
    if not (torch.is_tensor(pred) and torch.is_tensor(target)):
        raise TypeError("pred and target must be tensors")
    if pred.dim() < 2 or pred.shape != target.shape:
        raise ValueError(f"expected two [..., H, W] tensors of the same shape, got {tuple(pred.shape)} and "
                         f"{tuple(target.shape)}")
    if not pred.is_cuda or not target.is_cuda:
        raise ValueError("surface_distances runs on a CUDA device only: there is no CPU fallback")
    if pred.device != target.device:
        raise ValueError(f"pred is on {pred.device}, target on {target.device}")
    for name, m in (("pred", pred), ("target", target)):
        if m.dtype not in (torch.bool, torch.uint8):
            raise ValueError(f"surface_distances expects a bool or uint8 {name}, got {m.dtype}")
    percentile, tolerance = float(percentile), float(tolerance)
    if not 0.0 <= percentile <= 100.0:
        raise ValueError(f"percentile must be in [0, 100], got {percentile}")
    if not (math.isfinite(tolerance) and tolerance >= 0.0):
        raise ValueError(f"tolerance must be finite and >= 0, got {tolerance}")
    H, W = int(pred.shape[-2]), int(pred.shape[-1])
    _check_hw(H, W, "surface_distances")
    n = pred.numel() // (H * W)
    dev = pred.device
    out = torch.empty((4, n), dtype=torch.float32, device=dev)
    if n > 0:
        p, t = (m.detach().contiguous() for m in (pred, target))
        p, t = (m.view(torch.uint8) if m.dtype == torch.bool else m for m in (p, t))
        L = _lib.lib()
        nb = ctypes.c_size_t(0)
        _lib.check(L.tl_surface_workspace_bytes(n, H, W, ctypes.byref(nb)), "tl_surface_workspace_bytes")
        with torch.cuda.device(dev):
            ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)  # per call: released to the caching allocator
            rc = L.tl_surface_distances(p.data_ptr(), t.data_ptr(), n, H, W, percentile, tolerance, ws.data_ptr(),
                                        ws.numel(), out.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_surface_distances")
    lead = pred.shape[:-2]
    return SurfaceDistances(*(o.view(lead) for o in out))


def distance_transform_edt(mask: torch.Tensor) -> torch.Tensor:
    """Exact Euclidean distance transform of every ``[H, W]`` map of ``mask`` (``[..., H, W]``, bool or uint8, CUDA;
    a nonzero pixel is a feature pixel).  Returns float32 of the same shape, without autograd: 0 at a zero pixel and,
    at a nonzero pixel, ``float32(sqrt(float64(s)))`` with ``s`` the exact integer squared distance (unit spacing,
    pixel centres) to the nearest zero pixel of the same map.

    On every map that has a zero pixel this equals ``scipy.ndimage.distance_transform_edt(m).astype(np.float32)`` bit
    for bit.  A map without a zero pixel gets ``+inf`` everywhere; scipy returns distances to a phantom pixel at
    ``(-1, -1)`` there instead.  No host synchronisation; 4 bytes per pixel of scratch are taken from PyTorch's caching
    allocator for the duration of the call."""
    if not torch.is_tensor(mask):
        raise TypeError("mask must be a tensor")
    if mask.dim() < 2:
        raise ValueError("distance_transform_edt expects [..., H, W] maps")
    if not mask.is_cuda:
        raise ValueError("distance_transform_edt runs on a CUDA device only: there is no CPU fallback")
    if mask.dtype not in (torch.bool, torch.uint8):
        raise ValueError(f"distance_transform_edt expects a bool or uint8 mask, got {mask.dtype}")
    H, W = int(mask.shape[-2]), int(mask.shape[-1])
    _check_hw(H, W, "distance_transform_edt")
    n = mask.numel() // (H * W)
    dev = mask.device
    out = torch.empty(mask.shape, dtype=torch.float32, device=dev)
    if n == 0:
        return out
    m = mask.detach().contiguous()
    if m.dtype == torch.bool:
        m = m.view(torch.uint8)
    L = _lib.lib()
    nb = ctypes.c_size_t(0)
    _lib.check(L.tl_edt_workspace_bytes(n, H, W, ctypes.byref(nb)), "tl_edt_workspace_bytes")
    with torch.cuda.device(dev):
        ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)  # per call: released to the caching allocator
        rc = L.tl_edt(m.data_ptr(), n, H, W, ws.data_ptr(), ws.numel(), out.data_ptr(), _stream_ptr(dev))
    _lib.check(rc, "tl_edt")
    return out


class _HausdorffDtFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, t, alpha):
        B, C, H, W = (int(d) for d in x.shape)
        n = B * C
        dev = x.device
        L = _lib.lib()
        ns, nc = ctypes.c_size_t(0), ctypes.c_size_t(0)
        _lib.check(L.tl_hausdorff_dt_workspace_bytes(n, H, W, ctypes.byref(ns), ctypes.byref(nc)),
                   "tl_hausdorff_dt_workspace_bytes")
        with torch.cuda.device(dev):
            state = torch.empty(ns.value, dtype=torch.uint8, device=dev)  # D per pixel: the backward reads it
            scratch = torch.empty(nc.value, dtype=torch.uint8, device=dev)  # per call, freed when the forward returns
            cost = torch.empty((B, C), dtype=torch.float32, device=dev)
            rc = L.tl_hausdorff_dt_forward(x.data_ptr(), t.data_ptr(), n, H, W, alpha, state.data_ptr(), state.numel(),
                                           scratch.data_ptr(), scratch.numel(), cost.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_hausdorff_dt_forward")
        ctx.save_for_backward(x, t, state)
        return cost

    @staticmethod
    @once_differentiable
    def backward(ctx, g_cost):
        x, t, state = ctx.saved_tensors
        B, C, H, W = (int(d) for d in x.shape)
        dev = x.device
        with torch.cuda.device(dev):
            gc = g_cost.to(device=dev, dtype=torch.float32).contiguous()
            grad = torch.empty_like(x)
            rc = _lib.lib().tl_hausdorff_dt_backward(x.data_ptr(), t.data_ptr(), B * C, H, W, state.data_ptr(),
                                                     state.numel(), gc.data_ptr(), grad.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_hausdorff_dt_backward")
        return grad, None, None


def hausdorff_dt_loss(masks: torch.Tensor, gt_masks: torch.Tensor, alpha: float = 2.0) -> torch.Tensor:
    """Hausdorff distance-transform loss (Karimi & Salcudean, IEEE TMI 2020) of every ``(b, c)`` map: float32
    ``[B, C]``, differentiable with respect to ``masks`` only.

    ``masks`` are float32 decoder logits ``[B, C, H, W]`` on CUDA; ``gt_masks`` has the same shape and any real or
    bool dtype, and is cast to float32 (as ``dice_ce_loss`` does).  Per map, with ``p = torch.sigmoid(x)`` (fp32)::

        P = p > 0.5,  T = t > 0.5
        F(M) = distance of each pixel to the nearest pixel of the other label of M   if M has both labels
             = 0 everywhere                                                           otherwise
        D    = F(P)^alpha + F(T)^alpha
        cost = (1 / HW) * sum_i (p_i - t_i)^2 * D_i

    accumulated in fp64 in a fixed order and rounded to fp32, so the cost is bit-identical from run to run; the
    gradient is ``(2 / HW) * (p - t) * D * p * (1 - p)``.  ``.mean()`` of the result is, by recollection (unpinned:
    monai is not a dependency), ``monai.losses.HausdorffDTLoss(alpha, include_background=True, sigmoid=True)`` with
    its default ``reduction="mean"``; the ``[B, C]`` form is its ``reduction="none"`` squeezed, including monai's rule
    that a map that is all foreground or all background gets a zero field.  The distance fields are exact
    (``distance_transform_edt``) and never leave the device.

    ``alpha`` must be finite and > 0; H and W must each be in [1, 4096].  A NaN logit makes that map's cost NaN.
    Neither the forward nor the backward synchronises the host.  The forward keeps D (4 bytes per pixel) for the
    backward, and takes 8 bytes per pixel of scratch from PyTorch's caching allocator for the duration of the call
    (about 1.8 GB at 64 x 14 x 496 x 512); nothing is kept between calls."""
    if not (torch.is_tensor(masks) and torch.is_tensor(gt_masks)):
        raise TypeError("masks and gt_masks must be tensors")
    if masks.dim() != 4 or masks.shape != gt_masks.shape:
        raise ValueError("expected two [B, C, H, W] tensors of the same shape")
    if not masks.is_cuda or not gt_masks.is_cuda:
        raise ValueError("hausdorff_dt_loss runs on a CUDA device only: there is no CPU fallback")
    if masks.device != gt_masks.device:
        raise ValueError(f"masks are on {masks.device}, gt_masks on {gt_masks.device}")
    if masks.dtype != torch.float32:
        raise ValueError(f"hausdorff_dt_loss expects float32 logits, got {masks.dtype}")
    if gt_masks.dtype.is_complex:
        raise ValueError(f"hausdorff_dt_loss expects a real or bool gt_masks, got {gt_masks.dtype}")
    alpha = float(alpha)
    if not (math.isfinite(alpha) and alpha > 0.0):
        raise ValueError(f"alpha must be finite and > 0, got {alpha}")
    B, C, H, W = (int(d) for d in masks.shape)
    _check_hw(H, W, "hausdorff_dt_loss")
    if B * C == 0:
        return masks.sum((2, 3))  # empty, still attached to autograd
    return _HausdorffDtFn.apply(masks.contiguous(), gt_masks.detach().to(torch.float32).contiguous(), alpha)
