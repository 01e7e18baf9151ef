#!/usr/bin/env python
"""Cost of a physical pixel spacing in the distance family, on one GPU, at two workloads of layered masks from
synthetic.make_batch (the inputs of hausdorff_probe.py and surface_probe.py):

  W1  64 x 14 x 256 x 256
  W2  64 x 14 x 496 x 512

Three ops, each timed three ways on the same inputs:

  distance_transform_edt(pred > 0.5, sampling=...)
  hausdorff_dt_loss(logit(pred), truth, spacing=...)       forward + backward
  surface_distances(pred > 0.5, truth > 0.5, spacing=...)   HD95, NSD at tolerance 1 (in the spacing's units)

  unit        spacing=None: the integer path
  weighted_1  spacing=(1, 1) through the weighted (fp64) path
  aniso       spacing=(3.87, 11.29), an OCT-like pitch in um (illustrative)

The forms are warmed up, then timed step by step with CUDA events, interleaved, one step of each per round; medians of
--steps.  scipy with sampling=(3.87, 11.29) on one host thread is timed on a few maps for scale.  The card's name and
power limit are read in the same run.  The weighted path at (1, 1) must equal the unit path bit for bit; that is
checked on the timed outputs and reported.

    python scripts/spacing_probe.py [--steps 10] [--warmup 3] [--scipy-maps 4] [--out FILE.json]
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
from tests.test_surface_distance import ref_percentile, ref_surface  # noqa: E402

WORKLOADS = {"W1": (64, 256, 256), "W2": (64, 496, 512)}
ANISO = (3.87, 11.29)
SPACINGS = {"unit": None, "weighted_1": (1.0, 1.0), "aniso": ANISO}


def scipy_map(op, p, t):
    """One map on the host with sampling=ANISO, one thread."""
    if op == "edt":
        return ndi.distance_transform_edt(p > 0.5, sampling=ANISO)
    if op == "loss":
        def field(M):
            if M.all() or not M.any():
                return np.zeros(M.shape)
            return ndi.distance_transform_edt(M, sampling=ANISO) + ndi.distance_transform_edt(~M, sampling=ANISO)
        D = field(p > 0.5) ** 2 + field(t > 0.5) ** 2
        return float(((p.astype(np.float64) - t) ** 2 * D).mean())
    Sp, St = ref_surface(p > 0.5), ref_surface(t > 0.5)
    d_pt = ndi.distance_transform_edt(~St, sampling=ANISO)[Sp]
    d_tp = ndi.distance_transform_edt(~Sp, sampling=ANISO)[St]
    return max(ref_percentile(d_pt, 95.0), ref_percentile(d_tp, 95.0))


def run(B, H, W, a):
    pred, truth = make_batch(B, H, W, seed=0, device="cuda")
    x = torch.logit(pred.clamp(1e-6, 1 - 1e-6))
    P, T = pred > 0.5, truth > 0.5

    def edt(sp):
        return [tlb.distance_transform_edt(P, sampling=sp)]

    def loss(sp):
        xr = x.detach().clone().requires_grad_(True)
        c = tlb.hausdorff_dt_loss(xr, truth, spacing=sp)
        c.mean().backward()
        return [c.detach(), xr.grad]

    def surf(sp):
        return list(tlb.surface_distances(P, T, 95.0, 1.0, spacing=sp))

    ops = {"distance_transform_edt": edt, "hausdorff_dt_loss_fwd_bwd": loss, "surface_distances": surf}
    res = {"shape": [B, int(x.shape[1]), H, W], "ops": {}}
    for op, fn in ops.items():
        outs, times = {}, {k: [] for k in SPACINGS}
        for k, sp in SPACINGS.items():
            for _ in range(a.warmup):
                outs[k] = fn(sp)
        torch.cuda.synchronize()
        for _, k in itertools.product(range(a.steps), SPACINGS):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            fn(SPACINGS[k])
            ev[1].record()
            ev[1].synchronize()
            times[k].append(ev[0].elapsed_time(ev[1]))
        r = {}
        for k in SPACINGS:
            t = sorted(times[k])
            r[k] = {"ms_median": round(t[len(t) // 2], 3), "ms_min": round(t[0], 3), "ms_max": round(t[-1], 3)}
        for k in ("weighted_1", "aniso"):
            r[k]["x_unit"] = round(r[k]["ms_median"] / r["unit"]["ms_median"], 3)
        r["weighted_1_equals_unit_bit_for_bit"] = all(
            torch.equal(u.view(torch.int32), w.view(torch.int32)) for u, w in zip(outs["unit"], outs["weighted_1"]))
        outs.clear()
        torch.cuda.empty_cache()
        res["ops"][op] = r
    # the host path, for scale
    p_host = pred.reshape(-1, H, W)[: a.scipy_maps].cpu().numpy()
    t_host = truth.reshape(-1, H, W)[: a.scipy_maps].cpu().numpy()
    for op, key in (("edt", "distance_transform_edt"), ("loss", "hausdorff_dt_loss_fwd_bwd"),
                    ("surface", "surface_distances")):
        t0 = time.perf_counter()
        for p, t in zip(p_host, t_host):
            scipy_map(op, p, t)
        dt = (time.perf_counter() - t0) * 1e3 / len(p_host)
        res["ops"][key]["scipy_aniso"] = {"ms_per_map": round(dt, 3), "maps_timed": len(p_host), "threads": 1,
                                          "ms_per_batch_extrapolated": round(dt * B * int(x.shape[1]), 1),
                                          "host_cores": os.cpu_count(),
                                          "note": "loss: forward only (the four transforms and the cost)"
                                          if op == "loss" else "forward"}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scipy-maps", type=int, default=4)
    ap.add_argument("--workloads", default="W1,W2")
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("spacing_probe.py needs a CUDA device")
    torch.cuda.set_device(0)
    gpu, limits = card()
    res = {"probe": "scripts/spacing_probe.py", "gpu": gpu, "power_limit_and_max_sm_clock": limits,
           "inputs": "synthetic.make_batch(seed=0): masks pred > 0.5 and truth > 0.5; loss logits = logit(pred), "
                     "alpha = 2; surface_distances at percentile 95, tolerance 1",
           "spacings": {k: v for k, v in SPACINGS.items()}, "steps": a.steps, "warmup": a.warmup, "workloads": {}}
    for name in a.workloads.split(","):
        res["workloads"][name] = run(*WORKLOADS[name], a)
        torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
