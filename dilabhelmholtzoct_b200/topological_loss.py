"""Drop-in replacement for the reference's topological loss.

Mirrors ``topo_loss`` of ``/root/reference/octsam/models/topological_loss.py:11-96`` -- same name,
positional order, keyword names and defaults -- as called from the SAM fine-tuning step
(``/root/reference/octsam/models/training_utils.py:64`` and ``:375``)::

    train_loss += topo_loss(torch.sigmoid(masks.float()), gt_masks.float(), 0.1, feat_d=1, interp=50)

The arithmetic (cubical persistence, diagram matching, loss, gradient scatter) runs in
``libtopoloss.so`` -- hand-written sm_100a CUDA kernels behind the C ABI of ``include/topoloss.h``.
There is no CPU path, no PyTorch fallback and no multi-backend dispatch: tensors must live on a
CUDA device and the library must be built, otherwise the call raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Sequence, Tuple

import torch
import torch.nn.functional as F
from torch.autograd.function import once_differentiable

from . import _lib


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


_SCRATCH = {}        # (device index, stream handle) -> uint8 tensor, grown on demand
_ARENA_FACTOR = float(os.environ.get("TL_ARENA_FACTOR", "1.0"))


def set_arena_factor(factor: float) -> None:
    """Scale the pair arena of every later call (1.0 = room for ~H*W/5 pairs per map; see
    ``tl_workspace_bytes``).  Raise it when ``check_status`` reports an exhausted arena."""
    global _ARENA_FACTOR
    _ARENA_FACTOR = max(1.0, float(factor))


def _buffers(B: int, C: int, H: int, W: int, feat_d: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
    """(state, scratch) for one tl_forward: ``state`` is fresh (tl_backward reads it), ``scratch`` is one
    cached buffer per (device, stream) -- calls on one stream run one after the other."""
    ns, nc = ctypes.c_size_t(0), ctypes.c_size_t(0)
    _lib.check(_lib.lib().tl_workspace_bytes(B, C, H, W, feat_d, ctypes.byref(ns), ctypes.byref(nc)), "tl_workspace_bytes")
    state = torch.empty(int(ns.value * _ARENA_FACTOR), dtype=torch.uint8, device=device)
    return state, _scratch(nc.value, device)


def _scratch(nbytes: int, device) -> torch.Tensor:
    """The cached scratch buffer of (device, current stream), grown to at least ``nbytes``: a scratch is only live
    inside one call, and calls on one stream run one after the other."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    scratch = _SCRATCH.get(key)
    if scratch is None or scratch.numel() < nbytes:
        scratch = _SCRATCH[key] = torch.empty(nbytes, dtype=torch.uint8, device=device)
    return scratch


class _StatusRing:
    """Deferred check of the device status word: every forward copies it (4 bytes, asynchronously) into a
    pinned slot; the next call into this module looks at the slots whose copy has finished and raises if a
    kernel reported an overflow or a NaN map.  The loss of that call is already NaN, so nothing is silent."""
    SLOTS = 64

    def __init__(self):
        self.host = torch.zeros(self.SLOTS, dtype=torch.int32).pin_memory()
        self.events = [None] * self.SLOTS
        self.ops = ["topo_loss"] * self.SLOTS  # the op whose status word each slot holds (named in the error)
        self.next = 0

    def post(self, state: torch.Tensor, device, op: str = "topo_loss") -> None:
        i = self.next
        self.next = (i + 1) % self.SLOTS
        if self.events[i] is not None:
            self.events[i].synchronize()
            self._raise_if_set(i)
        self.host[i:i + 1].copy_(state[16:20].view(torch.int32), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(device))
        self.events[i] = ev
        self.ops[i] = op

    def _raise_if_set(self, i: int) -> None:
        v = int(self.host[i])
        self.events[i] = None
        self.host[i] = 0
        if v:
            why = "; ".join(msg for bit, msg in _lib.STATUS_BITS.items() if v & bit)
            raise RuntimeError(f"{self.ops[i]}: an earlier call reported status {v}: {why} (its loss was NaN)")

    def poll(self, sync: bool = False) -> None:
        for i, ev in enumerate(self.events):
            if ev is not None and (sync or ev.query()):
                if sync:
                    ev.synchronize()
                self._raise_if_set(i)


_STATUS = {}


def _status_ring(device) -> _StatusRing:
    r = _STATUS.get(device.index)
    if r is None:
        r = _STATUS[device.index] = _StatusRing()
    return r


def check_status(sync: bool = True) -> None:
    """Raise if any earlier ``topo_loss`` or ``topological_prior`` call on this process reported a device-side
    problem (``sync=True`` waits for the outstanding status copies first)."""
    for ring in _STATUS.values():
        ring.poll(sync)


class _TopoLossFn(torch.autograd.Function):
    """forward = tl_forward, backward = tl_backward (analytic backward of the reference's autograd
    graph: MulBackward / MeanBackward / PowBackward / POT ValFunction / CdistBackward /
    IndexBackward, i.e. what ``train_loss.backward()`` at training_utils.py:66 runs for this loss).

    When the prediction requires a gradient the forward is ``tl_forward_backward``: the gradient for an
    upstream gradient of 1 is written in the tail of the persistence launch (by SMs that have run out of
    persistence work), and ``backward`` only scales it -- a kernel that returns at once when the upstream
    gradient is exactly 1, the case of ``(seg_loss + topo_loss).backward()``."""

    @staticmethod
    def forward(ctx, pred, truth, lamda, feat_d, loss_q, loss_r, global_batch):
        B, C, H, W = pred.shape
        dev = pred.device
        ring = _status_ring(dev)
        ring.poll()
        want_grad = bool(ctx.needs_input_grad[0])
        with torch.cuda.device(dev):
            state, scratch = _buffers(B, C, H, W, feat_d, dev)
            loss = torch.empty((), dtype=torch.float32, device=dev)
            args = (pred.data_ptr(), truth.data_ptr(), B, C, H, W, feat_d, float(loss_q), float(lamda),
                    int(bool(loss_r)), int(global_batch), state.data_ptr(), state.numel(), scratch.data_ptr(),
                    scratch.numel(), loss.data_ptr())
            ctx.grad = None
            if want_grad:
                ctx.grad = torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
                rc = _lib.lib().tl_forward_backward(*args, ctx.grad.data_ptr(), _stream_ptr(dev))
            else:
                rc = _lib.lib().tl_forward(*args, _stream_ptr(dev))
            _lib.check(rc, "tl_forward")
            ring.post(state, dev)
        ctx.ws = state  # header + bookkeeping + pair arena (a second backward over a retained graph reads it)
        ctx.args = (B, C, H, W, feat_d, float(loss_q), float(lamda), int(bool(loss_r)), int(global_batch))
        ctx.pred_meta = (pred.dtype, dev)
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        B, C, H, W, feat_d, q, lamda, loss_r, gb = ctx.args
        dtype, dev = ctx.pred_meta
        _status_ring(dev).poll()
        with torch.cuda.device(dev):
            g = grad_out.to(device=dev, dtype=torch.float32).contiguous()
            # the gradient the forward wrote is handed over (not kept: autograd's AccumulateGrad copies a buffer
            # somebody else still holds, a 2 x 235 MB pass at the headline shape)
            grad_pred, ctx.grad = ctx.grad, None
            if grad_pred is not None:
                rc = _lib.lib().tl_scale_gradient(g.data_ptr(), grad_pred.data_ptr(), grad_pred.numel(), _stream_ptr(dev))
                _lib.check(rc, "tl_scale_gradient")
            else:  # a second backward over a retained graph: from the pairs
                grad_pred = torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
                rc = _lib.lib().tl_backward(g.data_ptr(), ctx.ws.data_ptr(), ctx.ws.numel(), B, C, H, W, feat_d, q,
                                            lamda, loss_r, gb, grad_pred.data_ptr(), _stream_ptr(dev))
                _lib.check(rc, "tl_backward")
        return grad_pred, None, None, None, None, None, None


def _check_inputs(pred_obj, true_obj, feat_d):
    if not (torch.is_tensor(pred_obj) and torch.is_tensor(true_obj)):
        raise TypeError("pred_obj and true_obj must be tensors")
    if pred_obj.shape != true_obj.shape:
        raise ValueError(f"pred_obj {tuple(pred_obj.shape)} and true_obj {tuple(true_obj.shape)} differ in shape")
    if pred_obj.dim() != 4:
        raise ValueError("expected [B, C, H, W] maps (topological_loss.py:17-18 with two spatial dims)")
    if not pred_obj.is_cuda or not true_obj.is_cuda:
        raise ValueError("topo_loss runs on a CUDA device only: there is no CPU fallback")
    if pred_obj.dtype != torch.float32 or true_obj.dtype != torch.float32:
        raise ValueError("topo_loss expects float32 maps (the reference call site passes .float())")
    if feat_d not in (0, 1):
        # feat_d = 2 (the reference default) selects no diagram on 2-D maps and crashes in
        # WassersteinDistance; anything outside [0, 2] crashes in batch_iter (SURVEY.md 8a row A4)
        raise ValueError("feat_d must be 0 or 1 for 2-D maps (the reference call site uses feat_d=1)")


def _canonical(pred, truth) -> Tuple[torch.Tensor, torch.Tensor]:
    """Reproduce the nesting that ``.squeeze()`` + CubicalComplex.forward + batch_iter produce
    (topological_loss.py:62-75): with B == 1 every channel becomes its own 'image'."""
    B, C, H, W = pred.shape
    if H < 2 or W < 2:
        raise ValueError("maps must be at least 2x2 (a size-1 spatial dim is squeezed away by the reference)")
    if B == 1 and C == 1:
        raise ValueError("B == C == 1: the reference crashes here (batch_iter on a flat list)")
    if B == 1:
        pred, truth = pred.reshape(C, 1, H, W), truth.reshape(C, 1, H, W)
    pred, truth = pred.contiguous(), truth.contiguous()
    if H != W:
        # CubicalComplex passes ``dimensions=x.shape`` to gudhi un-reversed, and gudhi's FIRST dimension is the
        # fastest-varying one [UPSTREAM-RECALL, SURVEY.md 8a row A3a]: for H != W the reference computes the
        # persistence of the same flat buffer read as W rows of H pixels.  Flat indices -- hence where the
        # gradient lands -- are unchanged, so the drop-in is a view (autograd undoes it).
        lead = pred.shape[:2]
        pred, truth = pred.view(*lead, W, H), truth.view(*lead, W, H)
    return pred, truth


def topo_loss(pred_obj, true_obj, lamda, interp=0, feat_d=2, loss_q=2, loss_r=False):
    """Topological loss, forward step (signature of topological_loss.py:11-12).

    Args:
        pred_obj (torch.Tensor): prediction, ``[B, C, H, W]`` float32 on a CUDA device
        true_obj (torch.Tensor): ground truth, same shape
        lamda (float): strength of topological regularisation; ``0.0`` returns the float ``0.0``
        interp (int): side of the bilinear down-sample applied to both inputs (0 = none)
        feat_d (int): homology dimension to use (0 or 1 on 2-D maps)
        loss_q (int): exponent of the Wasserstein loss
        loss_r (bool): add the total-persistence regulariser of the prediction

    Returns:
        0-d float32 tensor on ``pred_obj.device`` attached to autograd.
    """
    if lamda == 0.0:  # topological_loss.py:30-31
        return 0.0
    _check_inputs(pred_obj, true_obj, feat_d)
    if interp != 0:  # topological_loss.py:33-46
        size = (interp,) * 2
        pred_obj = F.interpolate(pred_obj, size=size, mode="bilinear", align_corners=True)
        true_obj = F.interpolate(true_obj, size=size, mode="bilinear", align_corners=True)
    pred, truth = _canonical(pred_obj, true_obj.detach())
    return _TopoLossFn.apply(pred, truth, lamda, feat_d, loss_q, loss_r, 0)


class _ResampleFn(torch.autograd.Function):
    """tl_resample_forward / tl_resample_backward: ``F.interpolate(torch.sigmoid(x) if sig else x,
    size=(S, S), mode="bilinear", align_corners=True)`` as one gather (SURVEY.md 8f, row F1)."""

    @staticmethod
    def forward(ctx, x, S, sig):
        lead, (H, W) = x.shape[:-2], x.shape[-2:]
        n = 1
        for d in lead:
            n *= int(d)
        dev = x.device
        with torch.cuda.device(dev):
            out = torch.empty(tuple(lead) + (S, S), dtype=torch.float32, device=dev)
            rc = _lib.lib().tl_resample_forward(x.data_ptr(), n, H, W, S, int(sig), out.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_resample_forward")
        ctx.save_for_backward(x)
        ctx.meta = (n, H, W, S, int(sig))
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        n, H, W, S, sig = ctx.meta
        dev = x.device
        with torch.cuda.device(dev):
            g = g.to(dtype=torch.float32).contiguous()
            gin = torch.empty_like(x)
            rc = _lib.lib().tl_resample_backward(g.data_ptr(), x.data_ptr(), n, H, W, S, sig, gin.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_resample_backward")
        return gin, None, None


def resample(x: torch.Tensor, size: int, sigmoid: bool = False) -> torch.Tensor:
    """``F.interpolate(torch.sigmoid(x) if sigmoid else x, size=(size, size), mode="bilinear",
    align_corners=True)`` for ``[..., H, W]`` float32 CUDA tensors, fused (the sigmoid is taken of the
    <= 4 size^2 source pixels the outputs read, not of the whole map); differentiable."""
    if not x.is_cuda or x.dtype != torch.float32:
        raise ValueError("resample expects a float32 CUDA tensor (there is no CPU fallback)")
    if x.dim() < 2 or size < 1:
        raise ValueError("resample expects [..., H, W] and size >= 1")
    return _ResampleFn.apply(x.contiguous(), int(size), bool(sigmoid))


class _PostprocessFn(torch.autograd.Function):
    """tl_postprocess_forward / tl_postprocess_backward (SURVEY.md 8f, row F3)."""

    @staticmethod
    def forward(ctx, x, T, rh, rw, oh, ow):
        lead, (Hs, Ws) = x.shape[:-2], x.shape[-2:]
        n = 1
        for d in lead:
            n *= int(d)
        dev = x.device
        with torch.cuda.device(dev):
            out = torch.empty(tuple(lead) + (oh, ow), dtype=torch.float32, device=dev)
            rc = _lib.lib().tl_postprocess_forward(x.data_ptr(), n, Hs, Ws, T, rh, rw, oh, ow, out.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_postprocess_forward")
        ctx.meta = (tuple(x.shape), n, Hs, Ws, T, rh, rw, oh, ow)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        shape, n, Hs, Ws, T, rh, rw, oh, ow = ctx.meta
        dev = g.device
        with torch.cuda.device(dev):
            g = g.to(dtype=torch.float32).contiguous()
            gin = torch.empty(shape, dtype=torch.float32, device=dev)
            rc = _lib.lib().tl_postprocess_backward(g.data_ptr(), n, Hs, Ws, T, rh, rw, oh, ow, gin.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_postprocess_backward")
        return gin, None, None, None, None, None


def postprocess_masks(pred_masks: torch.Tensor, reshaped_input_size, original_size, padded_size: int = 1024) -> torch.Tensor:
    """The SAM post-processing of the reference training step (training_utils.py:57-59) as one gather::

        masks = F.interpolate(pred_masks, (1024, 1024), mode="bilinear", align_corners=False)
        masks = masks[..., :reshaped_input_size[0], :reshaped_input_size[1]]
        masks = F.interpolate(masks, original_size, mode="bilinear", align_corners=False)

    ``pred_masks`` is ``outputs.pred_masks.squeeze(2)``, ``[..., 256, 256]`` float32 on a CUDA device.  The
    ``[..., 1024, 1024]`` intermediate is never written; differentiable (the backward accumulates each
    output tile's 16-tap footprint in shared memory)."""
    if not pred_masks.is_cuda or pred_masks.dtype != torch.float32:
        raise ValueError("postprocess_masks expects a float32 CUDA tensor (there is no CPU fallback)")
    rh, rw = int(reshaped_input_size[0]), int(reshaped_input_size[1])
    oh, ow = int(original_size[0]), int(original_size[1])
    return _PostprocessFn.apply(pred_masks.contiguous(), int(padded_size), rh, rw, oh, ow)


class _DiceCeFn(torch.autograd.Function):
    """tl_dice_ce_forward / tl_dice_ce_backward (SURVEY.md 8f, row F2)."""

    @staticmethod
    def forward(ctx, x, t):
        B, C = int(x.shape[0]), int(x.shape[1])
        HW = 1
        for d in x.shape[2:]:
            HW *= int(d)
        dev = x.device
        L = _lib.lib()
        nb = ctypes.c_size_t(0)
        _lib.check(L.tl_dice_ce_workspace_bytes(B, C, ctypes.byref(nb)), "tl_dice_ce_workspace_bytes")
        with torch.cuda.device(dev):
            ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
            loss = torch.empty((), dtype=torch.float32, device=dev)
            rc = L.tl_dice_ce_forward(x.data_ptr(), t.data_ptr(), B, C, HW, ws.data_ptr(), loss.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_dice_ce_forward")
        ctx.save_for_backward(x, t, ws)
        ctx.meta = (B, C, HW)
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, t, ws = ctx.saved_tensors
        B, C, HW = ctx.meta
        dev = x.device
        with torch.cuda.device(dev):
            g = g.to(device=dev, dtype=torch.float32).contiguous()
            gx = torch.empty_like(x)
            rc = _lib.lib().tl_dice_ce_backward(g.data_ptr(), x.data_ptr(), t.data_ptr(), B, C, HW, ws.data_ptr(),
                                                gx.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_dice_ce_backward")
        return gx, None


def dice_ce_loss(masks: torch.Tensor, gt_masks: torch.Tensor) -> torch.Tensor:
    """``monai.losses.DiceCELoss(sigmoid=True)(masks, gt_masks)`` -- the reference's ``seg_loss``
    (training_utils.py:32, :62; monai 1.3.0 defaults: Dice with ``smooth_nr = smooth_dr = 1e-5`` averaged over
    (b, c), plus ``CrossEntropyLoss`` over the channel axis with the masks as class probabilities) -- as one
    fused reduction: the two ``[B, C, H, W]`` tensors are read once in the forward and once in the backward.
    ``masks`` are the decoder's logits (float32, CUDA); the gradient flows to ``masks`` only."""
    if not (torch.is_tensor(masks) and torch.is_tensor(gt_masks)):
        raise TypeError("masks and gt_masks must be tensors")
    if masks.shape != gt_masks.shape or masks.dim() < 3:
        raise ValueError("expected two [B, C, ...] tensors of the same shape")
    if not masks.is_cuda or not gt_masks.is_cuda:
        raise ValueError("dice_ce_loss runs on a CUDA device only: there is no CPU fallback")
    if masks.dtype != torch.float32:
        raise ValueError("dice_ce_loss expects float32 logits")
    return _DiceCeFn.apply(masks.contiguous(), gt_masks.detach().to(torch.float32).contiguous())


def topo_loss_from_logits(masks, gt_masks, lamda, interp=0, feat_d=2, loss_q=2, loss_r=False):
    """The reference call site as ONE call (training_utils.py:64 / :375)::

        topo_loss(torch.sigmoid(masks.float()), gt_masks.float(), lamda, interp=..., feat_d=...)

    ``masks`` are the mask decoder's logits ``[B, C, H, W]``, ``gt_masks`` the ground truth.  With
    ``interp != 0`` the sigmoid and both bilinear down-samples (topological_loss.py:33-46) run as fused
    gathers: only the source pixels that survive the down-sample are read, and the backward writes the
    dense logit gradient once.  Same value and gradient as the two-step form up to fp32 rounding of the
    resample (tests/test_resample.py).
    """
    if lamda == 0.0:  # topological_loss.py:30-31
        return 0.0
    if not (torch.is_tensor(masks) and torch.is_tensor(gt_masks)):
        raise TypeError("masks and gt_masks must be tensors")
    if masks.shape != gt_masks.shape or masks.dim() != 4:
        raise ValueError("expected two [B, C, H, W] tensors of the same shape")
    if not masks.is_cuda or not gt_masks.is_cuda:
        raise ValueError("topo_loss runs on a CUDA device only: there is no CPU fallback")
    if feat_d not in (0, 1):
        raise ValueError("feat_d must be 0 or 1 for 2-D maps (the reference call site uses feat_d=1)")
    H, W = masks.shape[-2:]
    if interp == 0 and H != W:  # nothing to resample; H != W as the reference sees such maps, see _canonical
        pred, truth = torch.sigmoid(masks.float()), gt_masks.detach().float()
    else:
        S = int(interp) if interp != 0 else H
        pred = resample(masks.float(), S, sigmoid=True)
        truth = resample(gt_masks.detach().float(), S, sigmoid=False)
    pred, truth = _canonical(pred, truth)
    return _TopoLossFn.apply(pred, truth, lamda, feat_d, loss_q, loss_r, 0)


_COPY_STREAMS = {}


def pack_mask_bits(true_host: torch.Tensor) -> torch.Tensor:
    """{0, 1} masks ``[B, C, H, W]`` (any dtype, host) -> pinned ``uint8 [B, C, H, W // 8]``, 8 pixels per byte in
    ``numpy.packbits`` order: the form ``topo_loss_from_host(..., truth_packed=True)`` takes.  W must be a multiple
    of 8."""
    if true_host.dim() != 4 or true_host.shape[-1] % 8:
        raise ValueError("expected [B, C, H, W] with W a multiple of 8")
    import numpy as np
    bits = np.packbits(true_host.cpu().numpy() != 0, axis=-1)
    return torch.from_numpy(bits).pin_memory()


def topo_loss_from_host(pred_host, true_host, lamda, interp=0, feat_d=2, loss_q=2, loss_r=False, *,
                        device=None, chunks=4, want_grad=True, truth_packed=False):
    """``topo_loss`` for inputs that live in pinned HOST memory: forward + backward with the
    host->device copies pipelined against the kernels.  ``true_host`` may be ``uint8``: one-hot / component
    masks are {0, 1} (the reference builds them on the CPU, training_utils.py:413, :432), so they can cross
    PCIe as bytes and be widened on the device (5 instead of 8 bytes per pixel and step) -- or, with
    ``truth_packed=True``, as BITS: ``uint8 [B, C, H, W // 8]`` from ``pack_mask_bits`` (4.125 bytes per pixel).

    The batch is cut into at most ``chunks`` groups of whole images (one wave of the persistence kernel each when
    ``chunks`` allows it); group i+1 is copied on a side stream
    while group i runs ``tl_forward`` / ``tl_backward`` (with ``B_global = B`` so the partial losses
    add up to ``lamda * mean_b W_b`` and gradients carry ``1/B``).  Returns ``(loss, grad_pred)``:
    a 0-d device tensor and the ``[B, C, H, W]`` device gradient of the (resampled, if ``interp``)
    prediction, or ``None`` when ``want_grad`` is false.  Same semantics as ``topo_loss(...)``
    followed by ``.backward()``.
    """
    if lamda == 0.0:
        return 0.0, None
    if interp != 0:
        raise ValueError("topo_loss_from_host takes maps at their final resolution (interp=0)")
    if truth_packed:
        if (pred_host.dim() != 4 or pred_host.shape[-1] % 8 or true_host.dtype != torch.uint8
                or tuple(true_host.shape) != tuple(pred_host.shape[:-1]) + (pred_host.shape[-1] // 8,)):
            raise ValueError("truth_packed: expected uint8 [B, C, H, W // 8] next to a [B, C, H, W] prediction, W % 8 == 0")
    elif pred_host.shape != true_host.shape or pred_host.dim() != 4:
        raise ValueError("expected two [B, C, H, W] tensors of the same shape")
    if pred_host.dtype != torch.float32 or true_host.dtype not in (torch.float32, torch.uint8):
        raise ValueError("topo_loss expects a float32 prediction and float32 (or uint8 {0, 1}) ground truth")
    if pred_host.is_cuda or true_host.is_cuda:
        raise ValueError("topo_loss_from_host takes HOST tensors (use topo_loss for device tensors)")
    if not (pred_host.is_pinned() and true_host.is_pinned()):
        raise ValueError("topo_loss_from_host needs pinned host tensors (tensor.pin_memory()): a pageable "
                         "source makes the copies synchronous and the copy / kernel overlap disappears")
    if feat_d not in (0, 1):
        raise ValueError("feat_d must be 0 or 1 for 2-D maps (the reference call site uses feat_d=1)")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    B, C, H, W = pred_host.shape
    if H < 2 or W < 2 or (B == 1 and C == 1):
        raise ValueError("unsupported shape (see topo_loss)")
    orig_shape = None
    if B == 1:  # the reference's .squeeze() quirk: every channel is its own image
        orig_shape = (B, C, H, W)
        pred_host, true_host = pred_host.reshape(C, 1, H, W), true_host.reshape(C, 1, H, -1)
        B, C = C, 1
    # H != W: the reference reads the same flat buffer as W rows of H pixels (see _canonical)
    Hk, Wk = (W, H) if H != W else (H, W)
    L = _lib.lib()
    # The persistence kernel runs one prediction map per SM at a time, so a group of `sms // C` images is one
    # full wave: finer groups would only add partly filled waves.  `chunks` caps the number of groups.
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    per = max(1, sms // C)
    chunks = max(1, min(int(chunks), B))
    if chunks >= (B + per - 1) // per:
        bounds = list(range(0, B, per)) + [B]
    else:
        bounds = [(i * B) // chunks for i in range(chunks + 1)]
    chunks = len(bounds) - 1
    ring = _status_ring(dev)
    ring.poll()
    with torch.cuda.device(dev):
        cur = torch.cuda.current_stream(dev)
        side = _COPY_STREAMS.get(dev.index)
        if side is None:
            side = _COPY_STREAMS[dev.index] = torch.cuda.Stream(device=dev)
        side.wait_stream(cur)
        pred = torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
        truth = torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
        truth_u8 = torch.empty(tuple(true_host.shape), dtype=torch.uint8, device=dev) if true_host.dtype == torch.uint8 else None
        grad = torch.empty((B, C, H, W), dtype=torch.float32, device=dev) if want_grad else None
        parts = torch.empty((chunks,), dtype=torch.float32, device=dev)
        events = []
        with torch.cuda.stream(side):  # nothing but copies on this stream: PCIe stays busy back to back
            for i in range(chunks):
                a, b = bounds[i], bounds[i + 1]
                pred[a:b].copy_(pred_host[a:b], non_blocking=True)
                (truth_u8 if truth_u8 is not None else truth)[a:b].copy_(true_host[a:b], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(side)
                events.append(ev)
        # forward and backward of a group run back to back on this stream, so ONE state buffer (sized for the
        # largest group) and the cached scratch serve every group
        state, scratch = _buffers(max(bounds[i + 1] - bounds[i] for i in range(chunks)), C, Hk, Wk, feat_d, dev)
        for i in range(chunks):
            a, b = bounds[i], bounds[i + 1]
            cur.wait_event(events[i])
            if truth_packed:          # {0, 1} masks travelled as bits
                _lib.check(L.tl_unpack_mask_bits(truth_u8[a:b].data_ptr(), truth[a:b].data_ptr(), (b - a) * C * H * W,
                                                 cur.cuda_stream), "tl_unpack_mask_bits")
            elif truth_u8 is not None:  # ... as bytes: widen them on the device
                truth[a:b].copy_(truth_u8[a:b])
            args = (pred[a:b].data_ptr(), truth[a:b].data_ptr(), b - a, C, Hk, Wk, feat_d, float(loss_q),
                    float(lamda), int(bool(loss_r)), B, state.data_ptr(), state.numel(),
                    scratch.data_ptr(), scratch.numel(), parts[i:].data_ptr())
            if want_grad:  # loss and gradient of the group in one launch sequence
                rc = L.tl_forward_backward(*args, grad[a:b].data_ptr(), cur.cuda_stream)
            else:
                rc = L.tl_forward(*args, cur.cuda_stream)
            _lib.check(rc, "tl_forward")
        ring.post(state, dev)  # the last group's status; the loss carries a NaN for any group
        loss = parts.sum()
        for t in (pred, truth, truth_u8, state):  # allocated on this stream, last used here or on the copy stream
            if t is not None:
                t.record_stream(side)
    if grad is not None and orig_shape is not None:
        grad = grad.reshape(orig_shape)
    return loss, grad


# ---------------------------------------------------------------- inner boundaries (parity tests)

def persistence_pairs(maps: torch.Tensor, dim: int, reference_shape_order: bool = False) -> List[torch.Tensor]:
    """CubicalComplex(dim=2, superlevel=False) on ``[..., H, W]`` maps: per map an int32 ``[K, 2]``
    tensor of (creator, destroyer) flat pixel indices in gudhi's emission order; for ``dim == 0`` the
    essential class, paired with ``argmax``, comes last (torch_topological
    CubicalComplex._extract_generators_and_diagrams; reference call topological_loss.py:62).

    By default the map is the image it looks like (H rows of W pixels).  ``reference_shape_order=True``
    reproduces what torch_topological computes for H != W, where gudhi receives ``dimensions=x.shape``
    un-reversed and reads the flat buffer as W rows of H pixels (see ``_canonical``); flat indices are the
    same in both readings, and for square maps the flag changes nothing."""
    if not maps.is_cuda or maps.dtype != torch.float32:
        raise ValueError("persistence_pairs expects float32 CUDA maps")
    H, W = maps.shape[-2:]
    if reference_shape_order:
        H, W = W, H
    flat = maps.reshape(-1, H, W).contiguous()
    n = flat.shape[0]
    L = _lib.lib()
    cap = L.tl_max_pairs(H, W, dim)
    if cap < 0:
        _lib.check(cap, "tl_max_pairs")
    dev = maps.device
    with torch.cuda.device(dev):
        nb = ctypes.c_size_t(0)
        _lib.check(L.tl_pairs_workspace_bytes(n, H, W, dim, ctypes.byref(nb)), "tl_pairs_workspace_bytes")
        ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
        pairs = torch.empty((n, cap, 2), dtype=torch.int32, device=dev)
        counts = torch.empty((n,), dtype=torch.int32, device=dev)
        rc = L.tl_persistence_pairs(flat.data_ptr(), n, H, W, dim, ws.data_ptr(), ws.numel(), pairs.data_ptr(),
                                    cap, counts.data_ptr(), _stream_ptr(dev))
    _lib.check(rc, "tl_persistence_pairs")
    cnt = counts.cpu().tolist()
    return [pairs[i, :c].clone() for i, c in enumerate(cnt)]


def wasserstein_cost(D1: Sequence[torch.Tensor], D2: Sequence[torch.Tensor], q: float = 2.0):
    """Per diagram pair: the ``ot.emd2`` value WassersteinDistance(q) sums (before the 1/q root,
    topological_loss.py:78-82) and, for every row of D1[k], the matched row of D2[k] or -1."""
    assert len(D1) == len(D2) and len(D1) > 0
    dev = D1[0].device
    if dev.type != "cuda":
        raise ValueError("wasserstein_cost expects CUDA tensors")
    n1 = [int(d.shape[0]) for d in D1]
    n2 = [int(d.shape[0]) for d in D2]
    off1 = torch.tensor([0] + list(torch.tensor(n1).cumsum(0).tolist()), dtype=torch.int32, device=dev)
    off2 = torch.tensor([0] + list(torch.tensor(n2).cumsum(0).tolist()), dtype=torch.int32, device=dev)
    A = torch.cat([d.reshape(-1, 2).float() for d in D1] + [torch.zeros((1, 2), device=dev)]).contiguous()
    Bm = torch.cat([d.reshape(-1, 2).float() for d in D2] + [torch.zeros((1, 2), device=dev)]).contiguous()
    L = _lib.lib()
    nb = ctypes.c_size_t(0)
    _lib.check(L.tl_wasserstein_workspace_bytes(len(D1), max(n1), max(n2), ctypes.byref(nb)), "tl_wasserstein_workspace_bytes")
    with torch.cuda.device(dev):
        ws = torch.empty(max(nb.value, 1), dtype=torch.uint8, device=dev)
        cost = torch.empty(len(D1), dtype=torch.float64, device=dev)
        match = torch.full((sum(n1) + 1,), -2, dtype=torch.int32, device=dev)
        rc = L.tl_wasserstein(A.data_ptr(), off1.data_ptr(), Bm.data_ptr(), off2.data_ptr(), len(D1), max(n1), max(n2),
                              float(q), ws.data_ptr(), ws.numel(), cost.data_ptr(), match.data_ptr(), _stream_ptr(dev))
    _lib.check(rc, "tl_wasserstein")
    o = off1.cpu().tolist()
    return cost, [match[o[k]:o[k + 1]] for k in range(len(D1))]
