"""Betti matching loss for 2-D maps, batched, on the GPU.

The Wasserstein cost (``topo_loss``, ``wasserstein_distance``) matches persistence diagrams by value only: a
predicted blob at C can pay for a target blob at B anywhere in the image.  Betti matching (Stucki et al., ICML 2023,
"Topologically faithful image segmentation via induced matching of persistence barcodes") matches a predicted
feature to a target feature only when both persist in the comparison image ``C = min(pred, target)``, through the
induced matchings of the two inclusions into it.  ``betti_matching(pred, target, dim)`` computes, for every pair of
``[H, W]`` maps, the matching and its cost, differentiable with respect to both maps (``tl_betti_*``).

The complex, filtration and pixel rules are those of ``cubical_persistence`` (T-construction, sublevel filtration,
exact cell order); maps are read as H rows of W pixels.  The cost is squared Euclidean distance between matched
diagram points plus squared distance to the diagonal, ``(d - b)^2 / 2``, for unmatched ones.  Parity with the
upstream Betti-Matching-3D package is unpinned: that package is not available here, and whether its cubical complex
follows the same convention is not verified.

There is no CPU path: the inputs must be float32 CUDA tensors.
"""
from __future__ import annotations

import ctypes
from typing import List

import torch
from torch.autograd.function import once_differentiable

from . import _lib
from .diagrams import _stream_ptr


class BettiMatching:
    """Betti matchings of ``n`` prediction / target map pairs.

    * ``cost``: float32 ``[n]``, per map ``sum_matched (b_p - b_t)^2 + (d_p - d_t)^2 + sum_unmatched (d - b)^2 / 2``,
      attached to autograd (prediction and target);
    * ``matched``: int32 ``[M, 4]``, (pred creator, pred destroyer, target creator, target destroyer) flat pixel
      indices into the map (``x[i].ravel()``);
    * ``unmatched_pred`` / ``unmatched_target``: int32 ``[K, 2]``, (creator, destroyer);
    * ``*_offsets``: int32 ``[n + 1]`` on the device; ``host_*_offsets``: the same as Python lists.  Map ``i`` owns
      rows ``offsets[i]`` .. ``offsets[i + 1] - 1`` of each record tensor.

    Within a map, records follow the pixel-graph node that owns the prediction (for ``unmatched_target``: target)
    interval -- H0: its birth vertex, H1: its destroyer pixel -- in raster order; for H0 the essential pair
    (global minimum -> argmax) is the map's last matched row.
    """
    __slots__ = ("cost", "matched", "unmatched_pred", "unmatched_target", "matched_offsets", "pred_offsets",
                 "target_offsets", "host_matched_offsets", "host_pred_offsets", "host_target_offsets")

    def __init__(self, cost, matched, unmatched_pred, unmatched_target, offsets: torch.Tensor, host: List[List[int]]):
        self.cost, self.matched, self.unmatched_pred, self.unmatched_target = cost, matched, unmatched_pred, unmatched_target
        self.matched_offsets, self.pred_offsets, self.target_offsets = offsets[0], offsets[1], offsets[2]
        self.host_matched_offsets, self.host_pred_offsets, self.host_target_offsets = (list(h) for h in host)

    def __len__(self) -> int:
        return len(self.host_matched_offsets) - 1

    def __repr__(self) -> str:
        return (f"BettiMatching(n={len(self)}, matched={self.host_matched_offsets[-1]}, "
                f"unmatched_pred={self.host_pred_offsets[-1]}, unmatched_target={self.host_target_offsets[-1]}, "
                f"device={self.cost.device})")


def _grad_rows(t: torch.Tensor) -> torch.Tensor:
    """The upstream gradient as a contiguous float32 vector on an 8-byte boundary (as ``diagrams._rows``): autograd
    can hand a backward a slice that starts 4 bytes into its storage, and such a one is copied."""
    t = t.to(dtype=torch.float32).contiguous()
    return t if t.data_ptr() % 8 == 0 else t.clone()


class _BettiFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, H, W, dim):
        n = pred.shape[0]
        dev = pred.device
        L = _lib.lib()
        nb = ctypes.c_size_t(0)
        _lib.check(L.tl_betti_workspace_bytes(n, H, W, dim, ctypes.byref(nb)), "tl_betti_workspace_bytes")
        with torch.cuda.device(dev):
            ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
            cost = torch.empty(n, dtype=torch.float32, device=dev)
            meta = torch.empty(3 * (n + 1) + 1, dtype=torch.int32, device=dev)  # offsets[3][n + 1], then the status word
            st = _stream_ptr(dev)
            _lib.check(L.tl_betti_compute(pred.data_ptr(), target.data_ptr(), n, H, W, dim, ws.data_ptr(), ws.numel(),
                                          cost.data_ptr(), meta.data_ptr(), meta[3 * (n + 1):].data_ptr(), st),
                       "tl_betti_compute")
            # the one host synchronisation: the record counts size the outputs, and the status comes with them
            host = meta.cpu()
            status = int(host[3 * (n + 1)])
            if status:
                why = "; ".join(msg for bit, msg in _lib.STATUS_BITS.items() if status & bit)
                raise RuntimeError(f"betti_matching: status {status}: {why}")
            host_off = host[:3 * (n + 1)].contiguous()
            M, Kp, Kt = (int(host_off[k * (n + 1) + n]) for k in range(3))
            offsets = meta[:3 * (n + 1)].view(3, n + 1)
            matched = torch.empty((M, 4), dtype=torch.int32, device=dev)
            up = torch.empty((Kp, 2), dtype=torch.int32, device=dev)
            ut = torch.empty((Kt, 2), dtype=torch.int32, device=dev)
            _lib.check(L.tl_betti_gather(n, H, W, dim, ws.data_ptr(), ws.numel(), offsets.data_ptr(), host_off.data_ptr(),
                                         M, Kp, Kt, matched.data_ptr() if M else None, up.data_ptr() if Kp else None,
                                         ut.data_ptr() if Kt else None, st), "tl_betti_gather")
        ctx.save_for_backward(pred, target, offsets, matched, up, ut)
        ctx.meta = (n, H, W, M, Kp, Kt)
        ctx.mark_non_differentiable(matched, up, ut, offsets, host_off)
        return cost, matched, up, ut, offsets, host_off

    @staticmethod
    @once_differentiable
    def backward(ctx, g_cost, *_unused):
        pred, target, offsets, matched, up, ut = ctx.saved_tensors
        n, H, W, M, Kp, Kt = ctx.meta
        want_t = ctx.needs_input_grad[1]
        dev = pred.device
        with torch.cuda.device(dev):
            gp = torch.empty((n, H, W), dtype=torch.float32, device=dev)
            gt = torch.empty((n, H, W), dtype=torch.float32, device=dev) if want_t else None
            gc = _grad_rows(g_cost)
            rc = _lib.lib().tl_betti_backward(pred.data_ptr(), target.data_ptr(), n, H, W, offsets.data_ptr(),
                                              matched.data_ptr() if M else None, M, up.data_ptr() if Kp else None, Kp,
                                              ut.data_ptr() if Kt else None, Kt, gc.data_ptr(), gp.data_ptr(),
                                              gt.data_ptr() if want_t else None, _stream_ptr(dev))
        _lib.check(rc, "tl_betti_backward")
        return gp, gt, None, None, None


def betti_matching(pred: torch.Tensor, target: torch.Tensor, dim: int, superlevel: bool = False) -> BettiMatching:
    """Betti matching of every ``[H, W]`` map pair of ``pred`` and ``target`` (``[..., H, W]``, float32, CUDA, equal
    shapes) in homology dimension ``dim`` (0 or 1).  Maps are numbered in ``x.reshape(-1, H, W)`` order.

    ``cost`` is differentiable with respect to both inputs (the target gets a gradient only when it requires one);
    as a loss term, use e.g. ``betti_matching(prob, gt, 1).cost.mean()``.  ``superlevel=True`` negates both maps, so
    the comparison image is the pixelwise maximum of the originals; the gradient is negated accordingly.

    The call synchronises the host with the device once, to read the record counts (they size the outputs)
    together with the status word: a map holding a NaN raises ``RuntimeError`` here.  The backward makes no
    synchronisation.
    """
    for t, what in ((pred, "pred"), (target, "target")):
        if not torch.is_tensor(t):
            raise TypeError(f"{what} must be a tensor")
        if not t.is_cuda:
            raise ValueError(f"betti_matching: {what} must be on a CUDA device: there is no CPU fallback")
        if t.dtype != torch.float32:
            raise ValueError(f"betti_matching expects float32 maps, {what} is {t.dtype}")
    if pred.dim() < 2 or pred.shape != target.shape:
        raise ValueError(f"betti_matching expects [..., H, W] maps of one shape, got {tuple(pred.shape)} and "
                         f"{tuple(target.shape)}")
    if pred.device != target.device:
        raise ValueError("betti_matching: pred and target are on different devices")
    if dim not in (0, 1):
        raise ValueError(f"dim must be 0 or 1 on 2-D maps, got {dim}")
    if superlevel:
        pred, target = -pred, -target
    H, W = int(pred.shape[-2]), int(pred.shape[-1])
    P = pred.reshape(-1, H, W).contiguous()
    T = target.reshape(-1, H, W).contiguous()
    n = P.shape[0]
    if n == 0:
        z = torch.zeros(0, dtype=torch.int32, device=pred.device)
        off = torch.zeros((3, 1), dtype=torch.int32, device=pred.device)
        return BettiMatching(torch.zeros(0, dtype=torch.float32, device=pred.device), z.view(0, 4), z.view(0, 2),
                             z.view(0, 2), off, [[0], [0], [0]])
    cost, matched, up, ut, offsets, host_off = _BettiFn.apply(P, T, H, W, int(dim))
    host = host_off.view(3, n + 1).tolist()
    return BettiMatching(cost, matched, up, ut, offsets, host)
