#!/usr/bin/env python
"""The boundary loss and its signed distance map on one GPU, at two workloads of layered masks from
synthetic.make_batch (the inputs of hausdorff_probe.py and spacing_probe.py):

  W1  64 x 14 x 256 x 256
  W2  64 x 14 x 496 x 512

Timed forms, each with spacing=None (unit) and (3.87, 11.29) (an OCT-like pitch in um, illustrative):

  op           boundary_loss(logit(pred), truth).mean() forward + backward
  composed     the same loss composed in torch from two distance_transform_edt calls (d_out = edt(~T),
               d_in = edt(T), phi = where(T, 1 - d_in, d_out), 0 on single-label maps), forward + backward
  map          signed_distance_map(truth > 0.5) alone

The forms are warmed up, then timed step by step with CUDA events, interleaved, one step of each per round; medians of
--steps.  scipy (Kervadec's one_hot2dist expression and the cost) on one host thread is timed on a few maps for scale.
The card's name and power limit are read in the same run.  The largest cost difference between the op and the
composed form is reported, and whether the map op equals scipy's float64 expression rounded to float32 on the maps
timed on the host.

    python scripts/boundary_probe.py [--steps 10] [--warmup 3] [--scipy-maps 4] [--out FILE.json]
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
SPACINGS = {"unit": None, "aniso": (3.87, 11.29)}


def composed_phi(T, sp):
    """phi from two distance_transform_edt calls, in fp32 (the subtraction of 1 after rounding)."""
    d_out = tlb.distance_transform_edt(~T, sampling=sp)
    d_in = tlb.distance_transform_edt(T, sampling=sp)
    mixed = (T.any((-2, -1)) & ~T.all((-2, -1)))[..., None, None]
    return torch.where(mixed, torch.where(T, 1.0 - d_in, d_out), torch.zeros((), device=T.device))


def scipy_map(p, t, sp):
    """One map on the host, one thread: Kervadec's expression and the cost."""
    M = t > 0.5
    if M.all() or not M.any():
        phi = np.zeros(M.shape)
    else:
        kw = {} if sp is None else {"sampling": sp}
        phi = ndi.distance_transform_edt(~M, **kw) * ~M - (ndi.distance_transform_edt(M, **kw) - 1) * M
    return phi, float((p.astype(np.float64) * phi).mean())


def run(B, H, W, a):
    pred, truth = make_batch(B, H, W, seed=0, device="cuda")
    x = torch.logit(pred.clamp(1e-6, 1 - 1e-6))
    T = truth > 0.5

    def op(sp):
        xr = x.detach().clone().requires_grad_(True)
        c = tlb.boundary_loss(xr, truth, spacing=sp)
        c.mean().backward()
        return [c.detach(), xr.grad]

    def composed(sp):
        xr = x.detach().clone().requires_grad_(True)
        c = (torch.sigmoid(xr) * composed_phi(T, sp)).mean((2, 3))
        c.mean().backward()
        return [c.detach(), xr.grad]

    def phi_map(sp):
        return [tlb.signed_distance_map(T, sampling=sp)]

    forms = {"boundary_loss_fwd_bwd": op, "composed_fwd_bwd": composed, "signed_distance_map": phi_map}
    keys = list(itertools.product(forms, SPACINGS))
    outs, times = {}, {k: [] for k in keys}
    for f, s in keys:
        for _ in range(a.warmup):
            outs[(f, s)] = forms[f](SPACINGS[s])
    torch.cuda.synchronize()
    for _, (f, s) in itertools.product(range(a.steps), keys):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        forms[f](SPACINGS[s])
        ev[1].record()
        ev[1].synchronize()
        times[(f, s)].append(ev[0].elapsed_time(ev[1]))
    res = {"shape": [B, int(x.shape[1]), H, W], "forms": {}}
    for f in forms:
        res["forms"][f] = {}
        for s in SPACINGS:
            t = sorted(times[(f, s)])
            res["forms"][f][s] = {"ms_median": round(t[len(t) // 2], 3), "ms_min": round(t[0], 3), "ms_max": round(t[-1], 3)}
    for s in SPACINGS:
        c_op, g_op = outs[("boundary_loss_fwd_bwd", s)]
        c_co, g_co = outs[("composed_fwd_bwd", s)]
        res.setdefault("op_vs_composed", {})[s] = {
            "speedup": round(res["forms"]["composed_fwd_bwd"][s]["ms_median"] /
                             res["forms"]["boundary_loss_fwd_bwd"][s]["ms_median"], 3),
            "cost_max_abs_diff": float((c_op - c_co).abs().max()),
            "cost_max_abs": float(c_op.abs().max()),
            "grad_max_abs_diff_over_max_abs": float((g_op - g_co).abs().max() / g_op.abs().max().clamp_min(1e-30))}
    # the host path, for scale and as a check of the map op
    p_host = torch.sigmoid(x).reshape(-1, H, W)[: a.scipy_maps].cpu().numpy()
    t_host = truth.reshape(-1, H, W)[: a.scipy_maps].cpu().numpy()
    res["scipy"] = {}
    for s, sp in SPACINGS.items():
        phis = tlb.signed_distance_map(T.reshape(-1, H, W)[: a.scipy_maps], sampling=sp).cpu().numpy()
        t0 = time.perf_counter()
        ref = [scipy_map(p, t, sp) for p, t in zip(p_host, t_host)]
        dt = (time.perf_counter() - t0) * 1e3 / len(p_host)
        res["scipy"][s] = {"ms_per_map": round(dt, 3), "maps_timed": len(p_host), "threads": 1,
                           "ms_per_batch_extrapolated": round(dt * B * int(x.shape[1]), 1), "host_cores": os.cpu_count(),
                           "note": "forward only: the two transforms, phi and the cost",
                           "map_op_equals_scipy_bit_for_bit": all(
                               np.array_equal(g.view(np.uint32), r.astype(np.float32).view(np.uint32))
                               for g, (r, _) in zip(phis, ref))}
    outs.clear()
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
        sys.exit("boundary_probe.py needs a CUDA device")
    torch.cuda.set_device(0)
    gpu, limits = card()
    res = {"probe": "scripts/boundary_probe.py", "gpu": gpu, "power_limit_and_max_sm_clock": limits,
           "inputs": "synthetic.make_batch(seed=0): logits = logit(pred), target = truth; the map op on truth > 0.5",
           "spacings": dict(SPACINGS), "steps": a.steps, "warmup": a.warmup, "workloads": {}}
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
