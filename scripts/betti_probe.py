#!/usr/bin/env python
"""Forward + backward time of the Betti matching loss at the C2 shape (64 x 14 maps of 256 x 256, sublevel), for
dim 1 and dim 0, next to the two Wasserstein forms of the topological loss on the same inputs, on one GPU:

  betti_d1 / betti_d0  betti_matching(pred, truth, dim).cost.mean(); backward
  fused                topo_loss(pred, truth, 0.1, feat_d=1); backward
  composed             the same loss from cubical_persistence + wasserstein_distance; backward

Each form is warmed up, then timed step by step with CUDA events around forward + backward (betti_matching and the
composed form synchronise the host once inside the step: the events include that).  The forms run interleaved, one
step of each per round.  The card's name and power limit are read in the same run.

    python scripts/betti_probe.py [--steps 10] [--warmup 3] [--out FILE.json]
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
from scripts.tda_probe import card, composed, fused  # noqa: E402


def betti(dim):
    return lambda pred, truth: tlb.betti_matching(pred, truth, dim).cost.mean()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--B", type=int, default=64)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("betti_probe.py needs a CUDA device")
    torch.cuda.set_device(0)
    pred, truth = make_batch(a.B, a.size, a.size, seed=0, device="cuda")
    forms = {"betti_d1": betti(1), "betti_d0": betti(0), "fused": fused, "composed": composed}
    losses, times = {}, {k: [] for k in forms}

    def step(name):
        p = pred.detach().clone().requires_grad_(True)
        loss = forms[name](p, truth)
        loss.backward()
        return loss.detach()

    for name in forms:
        for _ in range(a.warmup):
            losses[name] = step(name)
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
        "probe": "scripts/betti_probe.py",
        "gpu": gpu, "power_limit_and_max_sm_clock": limits,
        "shape": [a.B, int(pred.shape[1]), a.size, a.size], "filtration": "sublevel",
        "steps": a.steps, "warmup": a.warmup,
        "forms": {},
    }
    fused_med = sorted(times["fused"])[len(times["fused"]) // 2]
    for name in forms:
        t = sorted(times[name])
        med = t[len(t) // 2]
        res["forms"][name] = {"ms_median": round(med, 3), "ms_min": round(t[0], 3), "ms_max": round(t[-1], 3),
                              "x_fused": round(med / fused_med, 2), "loss": float(losses[name])}
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
