"""Topological prior loss for 2-D maps, batched, on the GPU.

``topo_loss``, ``wasserstein_distance`` and ``betti_matching`` compare a prediction with a ground-truth map.  The
topological prior of Clough et al. ("Explicit topological priors for deep-learning based image segmentation using
persistent homology", IPMI 2019; TPAMI 2022) needs no target: it asks each map for a given number of features in one
homology dimension, e.g. one component and no holes for the mask of one structure, and none at all for an empty
(padded) mask.  ``topological_prior(x, dim, betti)`` computes it for every ``[H, W]`` map of ``x``, differentiable with
respect to ``x`` (``tl_prior_*``).

Per map, with D the diagram ``cubical_persistence(x, dim, superlevel)`` returns (same pairs, same order) and
``p = |death - birth|`` of each record (fp32), ranked by p descending with ties broken by position in D::

    cost = sum_{rank < betti} (1 - p^2) + sum_{rank >= betti} p^2 + max(0, betti - |D|)

A missing interval counts as persistence 0 (1 each, no gradient), as TopologyLayer's ``TopKBarcodeLengths`` pads.
Parity with Clough et al.'s published code is unpinned: that code is not available here; the formula above is the
definition implemented.

There is no CPU path: the input must be a float32 CUDA tensor.
"""
from __future__ import annotations

import ctypes
import numbers

import torch
from torch.autograd.function import once_differentiable

from . import _lib
from .diagrams import _stream_ptr
from .topological_loss import _scratch, _status_ring

_INT32_MAX = 2 ** 31 - 1


class _PriorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, maps, betti, H, W, dim):
        n = maps.shape[0]
        dev = maps.device
        L = _lib.lib()
        ns, nc = ctypes.c_size_t(0), ctypes.c_size_t(0)
        _lib.check(L.tl_prior_workspace_bytes(n, H, W, dim, ctypes.byref(ns), ctypes.byref(nc)), "tl_prior_workspace_bytes")
        ring = _status_ring(dev)
        ring.poll()
        with torch.cuda.device(dev):
            state = torch.empty(ns.value, dtype=torch.uint8, device=dev)  # sorted records + thresholds: the backward reads it
            scratch = _scratch(nc.value, dev)
            cost = torch.empty(n, dtype=torch.float32, device=dev)
            _lib.check(L.tl_prior_forward(maps.data_ptr(), n, H, W, dim, betti.data_ptr(), state.data_ptr(), state.numel(),
                                          scratch.data_ptr(), scratch.numel(), cost.data_ptr(), _stream_ptr(dev)),
                       "tl_prior_forward")
            # a NaN map or an exhausted arena: the costs are NaN now, and the next call (or check_status) raises
            ring.post(state, dev, "topological_prior")
        ctx.save_for_backward(maps)
        ctx.state = state
        ctx.meta = (n, H, W, dim)
        return cost

    @staticmethod
    @once_differentiable
    def backward(ctx, g_cost):
        (maps,) = ctx.saved_tensors
        n, H, W, dim = ctx.meta
        dev = maps.device
        with torch.cuda.device(dev):
            gc = g_cost.to(dtype=torch.float32).contiguous()
            grad = torch.empty((n, H, W), dtype=torch.float32, device=dev)
            rc = _lib.lib().tl_prior_backward(maps.data_ptr(), n, H, W, dim, ctx.state.data_ptr(), ctx.state.numel(),
                                              gc.data_ptr(), grad.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_prior_backward")
        return grad, None, None, None, None


def _check_betti(betti, lead: torch.Size):
    """The host-side checks of ``betti``: an int, or an integer tensor (CPU or CUDA) that broadcasts to ``lead``.
    Values are checked for the int and a CPU tensor only: reading a CUDA tensor would synchronise."""
    if isinstance(betti, numbers.Integral) and not isinstance(betti, bool):
        if betti < 0:
            raise ValueError(f"topological_prior: betti must be >= 0, got {betti}")
        return min(int(betti), _INT32_MAX)
    if torch.is_tensor(betti):
        t = betti
    else:
        try:
            t = torch.as_tensor(betti)
        except (TypeError, ValueError, RuntimeError) as e:
            raise ValueError(f"topological_prior: betti must be an int, a sequence of ints or an integer tensor ({e})")
    if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
        raise ValueError(f"topological_prior: betti must hold integers, got {t.dtype}")
    if not (t.is_cuda or t.device.type == "cpu"):
        raise ValueError(f"topological_prior: betti must be on the CPU or on the maps' device, got {t.device}")
    try:
        shape = torch.broadcast_shapes(t.shape, lead)
    except RuntimeError:
        shape = None
    if shape != lead:
        raise ValueError(f"topological_prior: betti of shape {tuple(t.shape)} does not broadcast to the map shape "
                         f"{tuple(lead)}")
    if not t.is_cuda and t.numel() and int(t.min()) < 0:
        raise ValueError("topological_prior: betti must be >= 0")
    return t


def _betti_vector(betti, lead: torch.Size, n: int, dev) -> torch.Tensor:
    """A checked ``betti`` -> int32 ``[n]`` on ``dev``, without a host synchronisation (a negative value in a CUDA
    tensor makes that map's cost NaN on the device)."""
    if isinstance(betti, int):
        return torch.full((n,), betti, dtype=torch.int32, device=dev)
    t = betti.to(torch.int64)
    if t.is_cuda:
        if t.device != dev:
            raise ValueError(f"topological_prior: betti is on {t.device}, the maps on {dev}")
        return t.clamp(-1, _INT32_MAX).to(torch.int32).expand(lead).reshape(n).contiguous()
    host = t.clamp(max=_INT32_MAX).to(torch.int32).expand(lead).reshape(n).contiguous()
    return host.pin_memory().to(dev, non_blocking=True)  # asynchronous: a pageable source would synchronise


def topological_prior(x: torch.Tensor, dim: int, betti, superlevel: bool = False) -> torch.Tensor:
    """Topological prior loss of every ``[H, W]`` map of ``x`` (``[..., H, W]``, float32, CUDA) in homology dimension
    ``dim`` (0 or 1): float32 ``[n]``, maps numbered in ``x.reshape(-1, H, W)`` order, differentiable with respect
    to ``x``.

    ``betti`` is the wanted number of features per map: an int, a sequence or an integer tensor (CPU or ``x``'s
    device) that broadcasts to ``x.shape[:-2]``.  Per map, the ``betti`` most persistent intervals of the map's
    diagram (ranked by ``p = |death - birth|`` descending, ties by position in the diagram, as a stable sort) are
    pushed towards persistence 1 and every other interval towards 0::

        cost = sum_{rank < betti} (1 - p^2) + sum_{rank >= betti} p^2 + max(0, betti - |D|)

    where D is the diagram ``cubical_persistence(x, dim, superlevel)`` returns (sublevel filtration, pixels as top
    cells, the H0 essential class paired with the argmax) and a missing interval counts as persistence 0.  On
    probability maps use ``superlevel=True`` (the filtration of ``-x``): ``dim=0, betti=1`` asks for one foreground
    component, ``dim=1, betti=0`` for no holes, ``dim=0, betti=0`` for an empty mask.  Squares and sums are fp64, the
    result is rounded to fp32 and is bit-identical from run to run.

    Neither the forward nor the backward synchronises the host with the device.  A map holding a NaN (or an
    exhausted pair arena) makes every cost of the call NaN and raises ``RuntimeError`` at the next call or at
    ``check_status()``; a negative entry of a CUDA ``betti`` makes that map's cost NaN.  Host-side ``betti`` values
    are checked at once.  Parity with Clough et al.'s published code is unpinned (it is not available here).
    """
    if not torch.is_tensor(x):
        raise TypeError("x must be a tensor")
    if x.dim() < 2:
        raise ValueError("topological_prior expects [..., H, W] maps")
    if dim not in (0, 1):
        raise ValueError(f"dim must be 0 or 1 on 2-D maps, got {dim}")
    lead = x.shape[:-2]
    betti = _check_betti(betti, lead)
    if not x.is_cuda:
        raise ValueError("topological_prior runs on a CUDA device only: there is no CPU fallback")
    if x.dtype != torch.float32:
        raise ValueError(f"topological_prior expects float32 maps, got {x.dtype}")
    H, W = int(x.shape[-2]), int(x.shape[-1])
    n = 1
    for d in lead:
        n *= int(d)
    b = _betti_vector(betti, lead, n, x.device)
    if n == 0:
        return x.reshape(0, H * W).sum(1)  # empty, still attached to autograd
    if superlevel:
        x = -x
    maps = x.reshape(n, H, W).contiguous()
    return _PriorFn.apply(maps, b, H, W, int(dim))
