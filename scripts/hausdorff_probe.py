#!/usr/bin/env python
"""Forward + backward time of the Hausdorff distance-transform loss on one GPU, at two workloads of layered masks from
synthetic.make_batch (logits = logit(pred), targets = the one-hot truth):

  W1  64 x 14 x 256 x 256   the C2 shape
  W2  64 x 14 x 496 x 512   the shape dice_ce_loss sees after postprocess_masks

and for each, three forms on the same inputs:

  fused     hausdorff_dt_loss(x, t).mean(); backward (forward and backward also timed apart)
  composed  the same loss in torch from distance_transform_edt: four transforms, the single-label rule and the
            elementwise ops, autograd through sigmoid; backward
  scipy     the host path monai takes (scipy.ndimage.distance_transform_edt, four transforms per map, one thread), on a
            subset of maps, reported per map with the host's core count

The GPU forms are warmed up, then timed step by step with CUDA events, interleaved, one step of each per round.  The
card's name and power limit are read in the same run, and the largest cost and gradient differences between the fused
and the composed form are reported.

    python scripts/hausdorff_probe.py [--steps 10] [--warmup 3] [--scipy-maps 8] [--out FILE.json]
"""
from __future__ import annotations

import argparse
import itertools
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import scipy.ndimage as ndi  # noqa: E402
import torch  # noqa: E402

import dilabhelmholtzoct_b200 as tlb  # noqa: E402
from dilabhelmholtzoct_b200.synthetic import make_batch  # noqa: E402
from scripts.tda_probe import card  # noqa: E402

WORKLOADS = {"W1": (64, 256, 256), "W2": (64, 496, 512)}


def composed_cost(x, t, alpha=2.0):
    p = torch.sigmoid(x)
    P, T = p.detach() > 0.5, t > 0.5

    def field(M):
        mixed = (M.any((2, 3)) & (~M).any((2, 3)))[..., None, None]
        return torch.where(mixed, tlb.distance_transform_edt(M) + tlb.distance_transform_edt(~M), 0.0)

    D = field(P) ** alpha + field(T) ** alpha
    return ((p - t) ** 2 * D).mean((2, 3))


def scipy_cost(p, t, alpha=2.0):
    """One map on the host, as monai computes it: four scipy transforms and the elementwise ops in float64."""
    def field(M):
        if M.all() or not M.any():
            return np.zeros(M.shape)
        return ndi.distance_transform_edt(M) + ndi.distance_transform_edt(~M)
    D = field(p > 0.5) ** alpha + field(t > 0.5) ** alpha
    return float(((p.astype(np.float64) - t) ** 2 * D).mean())


def run(name, B, H, W, a):
    pred, truth = make_batch(B, H, W, seed=0, device="cuda")
    x = torch.logit(pred.clamp(1e-6, 1 - 1e-6))
    del pred
    forms = {"fused": lambda p: tlb.hausdorff_dt_loss(p, truth), "composed": lambda p: composed_cost(p, truth)}
    outs, times, split = {}, {k: [] for k in forms}, {"forward": [], "backward": []}

    def step(form, events=None):
        p = x.detach().clone().requires_grad_(True)
        if events:
            events[0].record()
        c = forms[form](p)
        if events:
            events[1].record()
        c.mean().backward()
        if events:
            events[2].record()
        return c.detach(), p.grad

    for form in forms:
        for _ in range(a.warmup):
            outs[form] = step(form)
    torch.cuda.synchronize()
    for _, form in itertools.product(range(a.steps), forms):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        step(form, ev)
        ev[2].synchronize()
        times[form].append(ev[0].elapsed_time(ev[2]))
        if form == "fused":
            split["forward"].append(ev[0].elapsed_time(ev[1]))
            split["backward"].append(ev[1].elapsed_time(ev[2]))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    res = {"shape": [B, int(x.shape[1]), H, W], "forms": {}}
    for form in forms:
        t = sorted(times[form])
        res["forms"][form] = {"ms_median": round(med[form], 3), "ms_min": round(t[0], 3), "ms_max": round(t[-1], 3),
                              "loss": float(outs[form][0].mean())}
    res["forms"]["fused"]["forward_ms_median"] = round(sorted(split["forward"])[a.steps // 2], 3)
    res["forms"]["fused"]["backward_ms_median"] = round(sorted(split["backward"])[a.steps // 2], 3)
    res["forms"]["fused"]["x_composed"] = round(med["fused"] / med["composed"], 3)
    (c1, g1), (c2, g2) = outs["fused"], outs["composed"]
    res["forms"]["fused"].update({
        "max_rel_cost_diff_vs_composed": float(((c1.double() - c2.double()).abs() / c2.double().abs().clamp_min(1e-30)).max()),
        "max_abs_grad_diff_vs_composed": float((g1 - g2).abs().max()),
        "max_abs_grad": float(g2.abs().max()),
    })
    # the host path on the first maps
    p_host = torch.sigmoid(x[:1].reshape(-1, H, W)[: a.scipy_maps]).cpu().numpy()
    t_host = truth[:1].reshape(-1, H, W)[: a.scipy_maps].cpu().numpy()
    t0 = time.perf_counter()
    host = [scipy_cost(p, t) for p, t in zip(p_host, t_host)]
    dt = (time.perf_counter() - t0) * 1e3 / len(host)
    fused_first = c1.reshape(-1)[: len(host)].double().cpu().numpy()
    res["forms"]["scipy"] = {"ms_per_map": round(dt, 3), "maps_timed": len(host),
                             "ms_per_batch_extrapolated": round(dt * B * int(x.shape[1]), 1),
                             "host_cores": os.cpu_count(), "threads": 1,
                             "max_rel_cost_diff_fused_vs_scipy": float(np.max(np.abs(fused_first - host) / np.maximum(np.abs(host), 1e-30)))}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scipy-maps", type=int, default=8)
    ap.add_argument("--workloads", default="W1,W2")
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("hausdorff_probe.py needs a CUDA device")
    torch.cuda.set_device(0)
    gpu, limits = card()
    res = {"probe": "scripts/hausdorff_probe.py", "gpu": gpu, "power_limit_and_max_sm_clock": limits,
           "inputs": "synthetic.make_batch(seed=0): logits = logit(pred), target = one-hot truth; alpha = 2",
           "steps": a.steps, "warmup": a.warmup, "workloads": {}}
    for name in a.workloads.split(","):
        res["workloads"][name] = run(name, *WORKLOADS[name], a)
        torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
