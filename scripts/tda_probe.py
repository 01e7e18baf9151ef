#!/usr/bin/env python
"""Forward + backward time of the topological loss in three forms, at the C2 shape (64 x 14 maps of 256 x 256,
feat_d = 1, q = 2, lamda = 0.1, interp = 0), on one GPU:

  fused     topo_loss(pred, truth, 0.1, feat_d=1); backward
  composed  the same loss from the batched ops: cubical_persistence (pred and truth), wasserstein_distance,
            per-image sum, pow(1/q), mean, lamda; backward
  layer     the reference's orchestration (octsam/models/topological_loss.py:11-96) written against the
            torch_topological-compatible layer (dilabhelmholtzoct_b200.tda); backward

Each form is warmed up, then timed step by step with CUDA events around forward + backward (the composed forms
synchronise the host inside the step: the events include that).  The forms run interleaved, one step of each
per round.  The card's name and power limit are read in the same run.  The three losses and the largest
gradient difference to the fused form are reported too.

    python scripts/tda_probe.py [--steps 10] [--warmup 3] [--out FILE.json]
"""
from __future__ import annotations

import argparse
import itertools
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import dilabhelmholtzoct_b200 as tlb  # noqa: E402
from dilabhelmholtzoct_b200 import tda  # noqa: E402
from dilabhelmholtzoct_b200.synthetic import make_batch  # noqa: E402

LAMDA, FEAT_D, Q = 0.1, 1, 2


def fused(pred, truth):
    return tlb.topo_loss(pred, truth, LAMDA, feat_d=FEAT_D, loss_q=Q)


def composed(pred, truth):
    B, C = pred.shape[:2]
    cost = tlb.wasserstein_distance(tlb.cubical_persistence(pred, FEAT_D), tlb.cubical_persistence(truth, FEAT_D), q=Q)
    return LAMDA * cost.view(B, C).sum(1).pow(1.0 / Q).mean()


def layer(pred, truth):
    """topological_loss.py:55-96 for interp = 0, loss_r = False, on the compatibility layer."""
    cubical_complex = tda.CubicalComplex(dim=2, superlevel=False)
    pers_info_pred = cubical_complex(pred.squeeze())
    pers_info_true = cubical_complex(truth.squeeze())
    pred_batch = tda.batch_iter(pers_info_pred, dim=FEAT_D)
    true_batch = tda.batch_iter(pers_info_true, dim=FEAT_D)
    wasserstein = tda.WassersteinDistance(q=Q)
    topo_losses = [wasserstein(p, t) for p, t in zip(pred_batch, true_batch)]
    return LAMDA * torch.stack(topo_losses).mean()


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--B", type=int, default=64)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tda_probe.py needs a CUDA device")
    torch.cuda.set_device(0)
    pred, truth = make_batch(a.B, a.size, a.size, seed=0, device="cuda")
    forms = {"fused": fused, "composed": composed, "layer": layer}
    grads, losses, times = {}, {}, {k: [] for k in forms}

    def step(name):
        p = pred.detach().clone().requires_grad_(True)
        loss = forms[name](p, truth)
        loss.backward()
        return loss.detach(), p.grad

    for name in forms:  # warm-up, and the outputs the forms are compared on
        for _ in range(a.warmup):
            losses[name], grads[name] = step(name)
    torch.cuda.synchronize()
    for _, name in itertools.product(range(a.steps), forms):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(name)
        e1.record()
        e1.synchronize()
        times[name].append(e0.elapsed_time(e1))
    gpu, limits = card()
    ref_g = grads["fused"]
    res = {
        "probe": "scripts/tda_probe.py",
        "gpu": gpu, "power_limit_and_max_sm_clock": limits,
        "shape": [a.B, int(pred.shape[1]), a.size, a.size], "feat_d": FEAT_D, "q": Q, "lamda": LAMDA,
        "steps": a.steps, "warmup": a.warmup,
        "forms": {},
    }
    fused_med = sorted(times["fused"])[len(times["fused"]) // 2]
    for name in forms:
        t = sorted(times[name])
        med = t[len(t) // 2]
        res["forms"][name] = {
            "ms_median": round(med, 3), "ms_min": round(t[0], 3), "ms_max": round(t[-1], 3),
            "x_fused": round(med / fused_med, 2),
            "loss": float(losses[name]),
            "max_abs_grad_diff_vs_fused": float((grads[name] - ref_g).abs().max()),
            "same_grad_support_as_fused": bool(torch.equal(grads[name] != 0, ref_g != 0)),
        }
    res["max_abs_grad_fused"] = float(ref_g.abs().max())
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
