#!/usr/bin/env python
"""Forward + backward time of the topological prior loss at the C2 shape (64 x 14 maps of 256 x 256, superlevel), for
dim 0 with betti 1 (one component per mask) and dim 1 with betti 0 (no holes), next to the same loss composed in torch
and to the fused Wasserstein topo_loss, on the same inputs, on one GPU:

  prior_d0_b1 / prior_d1_b0        topological_prior(pred, dim, betti, superlevel=True).mean(); backward
  composed_d0_b1 / composed_d1_b0  cubical_persistence + two stable sorts + the formula in torch (fp64 terms); backward
  fused                            topo_loss(pred, truth, 0.1, feat_d=1); backward

Each form is warmed up, then timed step by step with CUDA events around forward + backward (the composed form
synchronises the host once inside the step: the events include that).  The forms run interleaved, one step of each
per round.  The card's name and power limit are read in the same run, and the largest cost and gradient differences
between each prior and its composed form are reported.

    python scripts/prior_probe.py [--steps 10] [--warmup 3] [--out FILE.json]
"""
from __future__ import annotations

import argparse
import itertools
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import dilabhelmholtzoct_b200 as tlb  # noqa: E402
from dilabhelmholtzoct_b200.synthetic import make_batch  # noqa: E402
from scripts.tda_probe import card, fused  # noqa: E402


def composed_cost(x, dim, betti):
    """The prior from the composable ops: one host sync (cubical_persistence), a gather, two stable sorts."""
    D = tlb.cubical_persistence(x, dim, superlevel=True)
    n, P, dev = len(D), D.host_offsets[-1], x.device
    cnt = (D.offsets[1:] - D.offsets[:-1]).long()
    p = (D.diagram[:, 1] - D.diagram[:, 0]).abs()
    seg = torch.repeat_interleave(torch.arange(n, device=dev), cnt, output_size=P)
    o1 = torch.sort(p.detach(), descending=True, stable=True).indices
    order = o1[torch.sort(seg[o1], stable=True).indices]  # by map, p descending, ties by position
    rank = torch.empty_like(order)
    rank[order] = torch.arange(P, device=dev) - D.offsets[:-1].long()[seg[order]]
    p64 = p.double()
    terms = torch.where(rank < betti, 1.0 - p64 * p64, p64 * p64)
    cost = torch.zeros(n, dtype=torch.float64, device=dev).index_add(0, seg, terms)
    return (cost + (betti - cnt).clamp(min=0).double()).float()


def prior(dim, betti):
    return lambda pred, truth: tlb.topological_prior(pred, dim, betti, superlevel=True)


def composed(dim, betti):
    return lambda pred, truth: composed_cost(pred, dim, betti)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--B", type=int, default=64)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prior_probe.py needs a CUDA device")
    torch.cuda.set_device(0)
    pred, truth = make_batch(a.B, a.size, a.size, seed=0, device="cuda")
    costs = {"prior_d0_b1": prior(0, 1), "prior_d1_b0": prior(1, 0),
             "composed_d0_b1": composed(0, 1), "composed_d1_b0": composed(1, 0)}
    forms = dict(costs, fused=lambda p, t: fused(p, t))
    outs, times = {}, {k: [] for k in forms}

    def step(name):
        p = pred.detach().clone().requires_grad_(True)
        c = forms[name](p, truth)
        loss = c.mean() if name in costs else c
        loss.backward()
        return c.detach(), p.grad

    for name in forms:
        for _ in range(a.warmup):
            outs[name] = step(name)
    torch.cuda.synchronize()
    for _, name in itertools.product(range(a.steps), forms):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(name)
        e1.record()
        e1.synchronize()
        times[name].append(e0.elapsed_time(e1))
    gpu, limits = card()
    res = {
        "probe": "scripts/prior_probe.py",
        "gpu": gpu, "power_limit_and_max_sm_clock": limits,
        "shape": [a.B, int(pred.shape[1]), a.size, a.size], "filtration": "superlevel",
        "steps": a.steps, "warmup": a.warmup,
        "forms": {},
    }
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    for name in forms:
        t = sorted(times[name])
        res["forms"][name] = {"ms_median": round(med[name], 3), "ms_min": round(t[0], 3), "ms_max": round(t[-1], 3),
                              "x_fused": round(med[name] / med["fused"], 2)}
        if name in costs:
            res["forms"][name]["loss"] = float(outs[name][0].mean())
    for d in ("d0_b1", "d1_b0"):
        (c1, g1), (c2, g2) = outs["prior_" + d], outs["composed_" + d]
        res["forms"]["prior_" + d].update({
            "x_composed": round(med["prior_" + d] / med["composed_" + d], 2),
            "max_abs_cost_diff_vs_composed": float((c1 - c2).abs().max()),
            "max_abs_grad_diff_vs_composed": float((g1 - g2).abs().max()),
            "max_abs_grad": float(g2.abs().max()),
        })
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
