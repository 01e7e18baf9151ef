"""torch_topological-compatible layer over the batched GPU ops of ``diagrams.py``.

``CubicalComplex``, ``PersistenceInformation``, ``batch_iter``, ``WassersteinDistance`` and ``total_persistence``
behave like the torch_topological classes of the same names that the reference's ``topological_loss.py``
imports, so a loss written against torch_topological ports by changing its imports::

    from dilabhelmholtzoct_b200.tda import CubicalComplex, WassersteinDistance, batch_iter, total_persistence

What differs is where the work runs: ``CubicalComplex`` computes all maps of its input in one batched call per
homology dimension on the GPU (torch_topological calls gudhi once per map on the CPU), and ``WassersteinDistance``
solves all diagram pairs of one call in one launch (instead of one ``ot.emd2`` per pair).  Only 2-D maps and the
L-inf ground metric (``p=inf``, torch_topological's default) are supported; anything else raises.
"""
from __future__ import annotations

import itertools
import math
from collections import namedtuple

import torch

from .diagrams import _pack, _wasserstein_packed, cubical_persistence


class PersistenceInformation(namedtuple("PersistenceInformation", ["pairing", "diagram", "dimension"], defaults=[None])):
    """Persistence information of one map and homology dimension: ``pairing`` (int64 ``[K, 4]``: creator row,
    creator column, destroyer row, destroyer column), ``diagram`` (float32 ``[K, 2]``: birth, death) and
    ``dimension``."""
    __slots__ = ()


def nesting_level(x) -> int:
    """How many times one can recurse into ``x`` while still obtaining lists (a PersistenceInformation is a leaf)."""
    if not isinstance(x, list):
        return 0
    if len(x) == 0:
        return 1
    return max(nesting_level(y) for y in x) + 1


def batch_iter(x, dim=None):
    """Iterate over a batch of persistence information: per batch element, its PersistenceInformation objects
    (only those of homology dimension ``dim`` when given), the channels of a ``[B][C]`` nesting chained."""
    level = nesting_level(x)
    if level <= 2:
        def handler(y):
            return y
    else:
        handler = itertools.chain.from_iterable
    if dim is not None:
        for first in x:
            yield [*filter(lambda y: y.dimension == dim, handler(first))]
    else:
        for first in x:
            yield handler(first)


def total_persistence(D, p=2, **kwargs):
    """Sum of ``|death - birth|^p`` over the finite points of one diagram ``[K, 2]``."""
    persistence = torch.diff(D)
    persistence = persistence[torch.isfinite(persistence)]
    return persistence.abs().pow(p).sum()


class CubicalComplex(torch.nn.Module):
    """Cubical persistence of ``[..., H, W]`` float32 CUDA maps with at most two leading dimensions.

    ``forward(x)`` returns what torch_topological's ``CubicalComplex(superlevel, dim)`` returns: for one map
    ``[PersistenceInformation(dim 0), PersistenceInformation(dim 1)]``, for ``[N, H, W]`` a list of those, for
    ``[B, C, H, W]`` a list of lists.  ``diagram`` of each is a slice of one packed autograd tensor per homology
    dimension; ``pairing`` holds coordinates with respect to the map's shape.  For ``H != W`` the maps are read
    the way the reference reads them (gudhi receives ``dimensions=x.shape`` un-reversed, see
    ``persistence_pairs(..., reference_shape_order=True)``)."""

    def __init__(self, superlevel=False, dim=None):
        super().__init__()
        self.superlevel = superlevel
        self.dim = dim

    def forward(self, x):
        if self.dim is not None and self.dim != 2:
            raise ValueError(f"CubicalComplex: only 2-D complexes (dim=2) are supported, got dim={self.dim}")
        if not torch.is_tensor(x) or x.dim() < 2:
            raise ValueError("CubicalComplex expects [..., H, W] maps")
        lead = tuple(x.shape[:-2])
        if len(lead) > 2:  # the exception torch_topological raises here
            raise RuntimeError("unsupported number of leading dimensions (at most two: [B, C, H, W])")
        h, w = int(x.shape[-2]), int(x.shape[-1])
        n = 1
        for s in lead:
            n *= int(s)
        per_map = [[None, None] for _ in range(n)]
        for d in (0, 1):
            D = cubical_persistence(x, d, superlevel=self.superlevel, reference_shape_order=True)
            p = D.pairs.long()
            pairing = torch.stack((p[:, 0] // w, p[:, 0] % w, p[:, 1] // w, p[:, 1] % w), 1)
            o = D.host_offsets
            for i in range(n):
                per_map[i][d] = PersistenceInformation(pairing=pairing[o[i]:o[i + 1]], diagram=D.diagram[o[i]:o[i + 1]],
                                                       dimension=d)
        if len(lead) == 0:
            return per_map[0]
        if len(lead) == 1:
            return per_map
        B, C = lead
        return [per_map[b * C:(b + 1) * C] for b in range(B)]


class WassersteinDistance(torch.nn.Module):
    """q-Wasserstein distance between the diagrams of two batches of PersistenceInformation with the L-inf ground
    metric: ``(sum over the pairs of zip(X, Y) of the ot.emd2 cost) ** (1 / q)``, summed in float32 in zip order
    like torch_topological's ``total_cost +=``.  All pairs go to one ``wasserstein_distance`` launch."""

    def __init__(self, p=torch.inf, q=1):
        super().__init__()
        if not (isinstance(p, (int, float)) and math.isinf(p) and p > 0):
            raise ValueError(f"WassersteinDistance: only the L-inf ground metric (p=inf) is supported, got p={p}")
        self.p = p
        self.q = q

    def forward(self, X, Y):
        pairs = list(zip(X, Y))
        if not pairs:
            raise ValueError("WassersteinDistance: no diagram pairs (torch_topological fails on this input too)")
        d1, off1, h1 = _pack([a.diagram for a, _ in pairs])
        d2, off2, h2 = _pack([b.diagram for _, b in pairs])
        cost = _wasserstein_packed(d1, off1, h1, d2, off2, h2, self.q)
        parts = cost.unbind(0)
        total_cost = parts[0]
        for c in parts[1:]:
            total_cost = total_cost + c
        return total_cost.pow(1.0 / self.q)
