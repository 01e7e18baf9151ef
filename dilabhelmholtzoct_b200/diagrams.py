"""Differentiable cubical persistence diagrams and Wasserstein distances, batched, on the GPU.

The fused ``topo_loss`` runs one fixed composition (sublevel filtration, one homology dimension, q-Wasserstein
with the L-inf ground metric, batch mean, ``lamda``).  These ops expose its pieces so that other compositions --
a superlevel filtration, H0 and H1 together, per-class weights, another reduction, logged diagrams -- stay on the
device:

* ``cubical_persistence(x, dim)`` -- the persistence pairs and diagram of every ``[H, W]`` map of ``x`` in one
  batched call (``tl_diagrams_compute`` / ``tl_diagrams_gather``), packed by map; the diagram is attached to
  autograd (``tl_diagrams_backward`` scatters its gradient into the critical pixels);
* ``wasserstein_distance(D1, D2, q)`` -- per pair of maps the ``ot.emd2`` value torch_topological's
  ``WassersteinDistance`` sums (``tl_wasserstein``), differentiable with respect to both diagrams
  (``tl_wasserstein_backward``);
* ``total_persistence(D, p)`` -- per map the sum of ``|death - birth|^p`` (plain torch).

There is no CPU path: the inputs must be float32 CUDA tensors.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence

import torch
from torch.autograd.function import once_differentiable

from . import _lib


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _rows(t: torch.Tensor) -> torch.Tensor:
    """A [P, 2] float32 tensor the library may read as 8-byte pairs: contiguous and 8-byte aligned.  Autograd can hand
    a backward a contiguous gradient that starts 4 bytes into its storage (a slice of a concatenation); that one is
    copied."""
    t = t.to(dtype=torch.float32).contiguous()
    return t if t.data_ptr() % 8 == 0 else t.clone()


class Diagrams:
    """Persistence diagrams of ``n`` maps, packed by map: map ``i`` owns rows ``host_offsets[i]`` ..
    ``host_offsets[i + 1] - 1``.

    * ``pairs``: int32 ``[P, 2]``, (creator, destroyer) flat pixel indices into the map (``x[i].ravel()``);
    * ``diagram``: float32 ``[P, 2]``, (birth, death) = the map's values at those pixels, attached to autograd;
    * ``offsets``: int32 ``[n + 1]`` on the device;
    * ``host_offsets``: the same offsets as a Python list.
    """
    __slots__ = ("pairs", "diagram", "offsets", "host_offsets")

    def __init__(self, pairs: torch.Tensor, diagram: torch.Tensor, offsets: torch.Tensor, host_offsets: List[int]):
        self.pairs, self.diagram, self.offsets, self.host_offsets = pairs, diagram, offsets, list(host_offsets)

    def __len__(self) -> int:
        return len(self.host_offsets) - 1

    @property
    def counts(self) -> List[int]:
        """Pairs per map."""
        o = self.host_offsets
        return [o[i + 1] - o[i] for i in range(len(o) - 1)]

    def split(self) -> List[torch.Tensor]:
        """The diagram of each map, as views of ``diagram`` (gradients flow back through them)."""
        o = self.host_offsets
        return [self.diagram[o[i]:o[i + 1]] for i in range(len(o) - 1)]

    def __repr__(self) -> str:
        return f"Diagrams(n={len(self)}, P={self.host_offsets[-1]}, device={self.diagram.device})"


class _CubicalFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, maps, H, W, dim):
        n = maps.shape[0]
        dev = maps.device
        L = _lib.lib()
        nb = ctypes.c_size_t(0)
        _lib.check(L.tl_diagrams_workspace_bytes(n, H, W, dim, ctypes.byref(nb)), "tl_diagrams_workspace_bytes")
        with torch.cuda.device(dev):
            ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
            meta = torch.empty(n + 2, dtype=torch.int32, device=dev)  # offsets[n + 1], then the status word
            st = _stream_ptr(dev)
            _lib.check(L.tl_diagrams_compute(maps.data_ptr(), n, H, W, dim, ws.data_ptr(), ws.numel(), meta.data_ptr(),
                                             meta[n + 1:].data_ptr(), st), "tl_diagrams_compute")
            # the one host synchronisation: the pair count sizes the outputs, and the status comes with it
            host = meta.cpu()
            status = int(host[n + 1])
            if status:
                why = "; ".join(msg for bit, msg in _lib.STATUS_BITS.items() if status & bit)
                raise RuntimeError(f"cubical_persistence: status {status}: {why}")
            host_off = host[:n + 1]
            P = int(host_off[n])
            offsets = meta[:n + 1]
            pairs = torch.empty((P, 2), dtype=torch.int32, device=dev)
            diagram = torch.empty((P, 2), dtype=torch.float32, device=dev)
            _lib.check(L.tl_diagrams_gather(maps.data_ptr(), n, H, W, dim, ws.data_ptr(), ws.numel(), offsets.data_ptr(),
                                            host_off.data_ptr(), P, pairs.data_ptr(), diagram.data_ptr(), st),
                       "tl_diagrams_gather")
        ctx.save_for_backward(pairs, offsets)
        ctx.meta = (n, H, W, P)
        ctx.mark_non_differentiable(pairs, offsets, host_off)
        return diagram, pairs, offsets, host_off

    @staticmethod
    @once_differentiable
    def backward(ctx, g_diagram, _g_pairs, _g_offsets, _g_host):
        pairs, offsets = ctx.saved_tensors
        n, H, W, P = ctx.meta
        dev = offsets.device
        with torch.cuda.device(dev):
            grad = torch.empty((n, H, W), dtype=torch.float32, device=dev)
            g = _rows(g_diagram) if P else None
            rc = _lib.lib().tl_diagrams_backward(pairs.data_ptr() if P else None, offsets.data_ptr(),
                                                 g.data_ptr() if P else None, P, n, H, W, grad.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_diagrams_backward")
        return grad, None, None, None


def cubical_persistence(x: torch.Tensor, dim: int, superlevel: bool = False,
                        reference_shape_order: bool = False) -> Diagrams:
    """Persistence pairs and diagrams of homology dimension ``dim`` (0 or 1) of every ``[H, W]`` map of ``x``
    (``[..., H, W]``, float32, CUDA), as torch_topological's ``CubicalComplex`` computes them through gudhi:
    pixels are the top cells, sublevel filtration, pairs in gudhi's emission order, for ``dim == 0`` the
    essential class last, paired with the map's ``argmax``.  Maps are numbered in ``x.reshape(-1, H, W)`` order.

    ``superlevel=True`` is torch_topological's ``x = -x``: the pairs and values of ``-x``, with the gradient
    negated accordingly.  ``reference_shape_order`` has the meaning it has in ``persistence_pairs``: for
    ``H != W`` the flat buffer is read as ``W`` rows of ``H`` pixels, as the reference does.

    The call synchronises the host with the device once, to read the number of pairs (it sizes the outputs)
    together with the status word: a map holding a NaN, or more pairs than the workspace holds, raises
    ``RuntimeError`` here.  The backward makes no synchronisation.
    """
    if not torch.is_tensor(x):
        raise TypeError("x must be a tensor")
    if not x.is_cuda:
        raise ValueError("cubical_persistence runs on a CUDA device only: there is no CPU fallback")
    if x.dtype != torch.float32:
        raise ValueError("cubical_persistence expects float32 maps")
    if x.dim() < 2:
        raise ValueError("cubical_persistence expects [..., H, W] maps")
    if dim not in (0, 1):
        raise ValueError(f"dim must be 0 or 1 on 2-D maps, got {dim}")
    if superlevel:
        x = -x
    H, W = int(x.shape[-2]), int(x.shape[-1])
    if reference_shape_order:
        H, W = W, H
    maps = x.reshape(-1, H, W).contiguous()
    diagram, pairs, offsets, host_off = _CubicalFn.apply(maps, H, W, int(dim))
    return Diagrams(pairs, diagram, offsets, host_off.tolist())


def _nonempty(t: torch.Tensor) -> torch.Tensor:
    """The library takes a valid pointer for an empty diagram set too."""
    return _rows(t) if t.numel() else torch.zeros((1, 2), dtype=torch.float32, device=t.device)


class _WassersteinFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, d1, d2, off1, off2, rows1, rows2, q):
        n = off1.shape[0] - 1
        dev = d1.device
        L = _lib.lib()
        nb = ctypes.c_size_t(0)
        _lib.check(L.tl_wasserstein_workspace_bytes(n, rows1, rows2, ctypes.byref(nb)), "tl_wasserstein_workspace_bytes")
        with torch.cuda.device(dev):
            a, b = _nonempty(d1), _nonempty(d2)
            ws = torch.empty(max(nb.value, 1), dtype=torch.uint8, device=dev)
            cost = torch.empty(n, dtype=torch.float64, device=dev)
            match = torch.empty(d1.shape[0] + 1, dtype=torch.int32, device=dev)
            rc = L.tl_wasserstein(a.data_ptr(), off1.data_ptr(), b.data_ptr(), off2.data_ptr(), n, rows1, rows2, float(q),
                                  ws.data_ptr(), ws.numel(), cost.data_ptr(), match.data_ptr(), _stream_ptr(dev))
        _lib.check(rc, "tl_wasserstein")
        ctx.save_for_backward(a, b, off1, off2, match)
        ctx.meta = (n, float(q), d1.shape[0], d2.shape[0])
        return cost.float()  # the emd2 value cast back to the diagrams' dtype, as POT does

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        a, b, off1, off2, match = ctx.saved_tensors
        n, q, P1, P2 = ctx.meta
        want1, want2 = ctx.needs_input_grad[0] and P1 > 0, ctx.needs_input_grad[1] and P2 > 0
        dev = a.device
        g1 = torch.empty((P1, 2), dtype=torch.float32, device=dev) if want1 else None
        g2 = torch.empty((P2, 2), dtype=torch.float32, device=dev) if want2 else None
        if want1 or want2:
            with torch.cuda.device(dev):
                gc = g.to(dtype=torch.float32).contiguous()
                rc = _lib.lib().tl_wasserstein_backward(a.data_ptr(), off1.data_ptr(), b.data_ptr(), off2.data_ptr(), n, q,
                                                        match.data_ptr(), gc.data_ptr(), g1.data_ptr() if want1 else None,
                                                        g2.data_ptr() if want2 else None, _stream_ptr(dev))
            _lib.check(rc, "tl_wasserstein_backward")
        if ctx.needs_input_grad[0] and g1 is None:
            g1 = torch.zeros((P1, 2), dtype=torch.float32, device=dev)
        if ctx.needs_input_grad[1] and g2 is None:
            g2 = torch.zeros((P2, 2), dtype=torch.float32, device=dev)
        return g1, g2, None, None, None, None, None


def _max_rows(host_offsets: Sequence[int]) -> int:
    return max((host_offsets[i + 1] - host_offsets[i] for i in range(len(host_offsets) - 1)), default=0)


def _check_packed(d: torch.Tensor, what: str) -> None:
    if not d.is_cuda:
        raise ValueError(f"wasserstein_distance: {what} must be on a CUDA device (there is no CPU fallback)")
    if d.dtype != torch.float32 or d.dim() != 2 or d.shape[1] != 2:
        raise ValueError(f"wasserstein_distance: {what} must be a float32 [P, 2] diagram")


def _wasserstein_packed(d1: torch.Tensor, off1: torch.Tensor, host_off1: Sequence[int], d2: torch.Tensor,
                        off2: torch.Tensor, host_off2: Sequence[int], q: float = 2.0) -> torch.Tensor:
    """``wasserstein_distance`` on packed diagrams: ``d1`` ``[P1, 2]`` with device offsets ``off1`` (int32,
    ``[n + 1]``, on d1's device) and their host copy ``host_off1``, likewise ``d2``.  The device offsets must hold
    the values of the host lists; that is not checked here (it would take a synchronisation): callers build both
    from one source (``Diagrams``, ``_pack``)."""
    _check_packed(d1, "D1")
    _check_packed(d2, "D2")
    n = len(host_off1) - 1
    for off, host, d, what in ((off1, host_off1, d1, "off1"), (off2, host_off2, d2, "off2")):
        if not torch.is_tensor(off) or off.dtype != torch.int32 or off.device != d.device or off.dim() != 1 \
                or off.shape[0] != len(host) or not off.is_contiguous():
            raise ValueError(f"wasserstein_distance: {what} must be a contiguous int32 [{len(host)}] tensor on {d.device}")
    if n != len(host_off2) - 1:
        raise ValueError(f"wasserstein_distance: {n} diagrams against {len(host_off2) - 1}")
    if host_off1[-1] != d1.shape[0] or host_off2[-1] != d2.shape[0]:
        raise ValueError("wasserstein_distance: offsets disagree with the diagrams' row counts")
    if not q > 0:
        raise ValueError("wasserstein_distance: q must be positive")
    if n == 0:
        return torch.zeros(0, dtype=torch.float32, device=d1.device)
    return _WassersteinFn.apply(d1, d2, off1, off2, _max_rows(host_off1), _max_rows(host_off2),
                                float(q))


def wasserstein_distance(D1: Diagrams, D2: Diagrams, q: float = 2) -> torch.Tensor:
    """Per pair of maps ``k``: the optimal-transport cost between ``D1``'s and ``D2``'s diagram of map ``k`` with
    the L-inf ground metric raised to ``q`` and the diagonal as a sink -- the ``ot.emd2`` value torch_topological's
    ``WassersteinDistance(q=q)`` adds up, before its ``1/q`` root.  Returns float32 ``[n]`` (the fp64 optimum cast
    to fp32), differentiable with respect to both diagrams; no gradient is computed for a side that does not
    require one.  Empty diagrams, on either side or both, are fine.  No host synchronisation."""
    if not (isinstance(D1, Diagrams) and isinstance(D2, Diagrams)):
        raise TypeError("wasserstein_distance takes two Diagrams (from cubical_persistence)")
    return _wasserstein_packed(D1.diagram, D1.offsets, D1.host_offsets, D2.diagram, D2.offsets, D2.host_offsets, q)


def total_persistence(D: Diagrams, p: float = 2) -> torch.Tensor:
    """Per map, the sum of ``|death - birth|^p`` over its finite points (torch_topological's
    ``total_persistence``, batched): float32 ``[n]``, differentiable, no host synchronisation."""
    n = len(D)
    dev = D.diagram.device
    pers = D.diagram[:, 1] - D.diagram[:, 0]
    pers = torch.where(torch.isfinite(pers), pers, torch.zeros_like(pers)).abs().pow(p)
    ids = torch.repeat_interleave(torch.arange(n, device=dev), D.offsets[1:] - D.offsets[:-1], output_size=int(D.host_offsets[-1]))
    return torch.zeros(n, dtype=pers.dtype, device=dev).index_add(0, ids, pers)


def _as_device_offsets(host_offsets: Sequence[int], device) -> torch.Tensor:
    """int32 device offsets from a host list without a synchronising copy (pinned source, asynchronous copy)."""
    return torch.tensor(list(host_offsets), dtype=torch.int32).pin_memory().to(device, non_blocking=True)


def _pack(diagrams: Sequence[torch.Tensor]) -> "tuple[torch.Tensor, torch.Tensor, List[int]]":
    """``[K_i, 2]`` diagrams -> (``[sum K_i, 2]`` rows in order, device offsets, host offsets).  Diagrams that are
    consecutive row slices of one tensor (what ``Diagrams.split`` and the compatibility layer hand out) become one
    view of it instead of a copy, so the backward does not build one full-size gradient per slice."""
    host = [0]
    for d in diagrams:
        if d.dim() != 2 or d.shape[1] != 2:
            raise ValueError("diagrams must be [K, 2]")
        host.append(host[-1] + int(d.shape[0]))
    dev = diagrams[0].device
    base: Optional[torch.Tensor] = diagrams[0]._base
    packed = None
    if base is not None and base.dim() == 2 and base.shape[1] == 2 and base.is_contiguous():
        row0 = (diagrams[0].storage_offset() - base.storage_offset()) // 2
        ok = all(d._base is base and (d.shape[0] <= 1 or d.stride() == (2, 1)) and (d.shape[0] == 0 or d.stride(1) == 1)
                 and d.storage_offset() - base.storage_offset() == 2 * (row0 + host[i]) for i, d in enumerate(diagrams))
        if ok and row0 + host[-1] <= base.shape[0]:
            packed = base.narrow(0, row0, host[-1])
    if packed is None:
        packed = torch.cat([d.to(torch.float32) for d in diagrams]) if diagrams else torch.zeros((0, 2), device=dev)
    return packed, _as_device_offsets(host, dev), host
