#!/usr/bin/env python
"""Time of the surface-distance metrics (HD, HD95, ASSD, NSD at 1 pixel) on one GPU, at two workloads of layered
masks from synthetic.make_batch (pred > 0.5 against truth > 0.5):

  W1  64 x 14 x 256 x 256   the C2 shape
  W2  64 x 14 x 496 x 512   the shape dice_ce_loss sees after postprocess_masks

and for each, three forms on the same masks:

  op        surface_distances(pred, target, 95, 1)
  composed  the same metrics in torch: surfaces by a cross erosion, two distance_transform_edt calls on the inverted
            surfaces, and per map a sort of the surface distances and a gather for the percentile
  scipy     the host path (scipy.ndimage.binary_erosion and distance_transform_edt, np.percentile, one thread) on a
            subset of maps, reported per map with the host's core count

The GPU forms are warmed up, then timed step by step with CUDA events, interleaved, one step of each per round.  The
card's name and power limit are read in the same run, and the largest differences between the forms are reported.

    python scripts/surface_probe.py [--steps 10] [--warmup 3] [--scipy-maps 8] [--out FILE.json]
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
import torch.nn.functional as F  # noqa: E402

import dilabhelmholtzoct_b200 as tlb  # noqa: E402
from dilabhelmholtzoct_b200.synthetic import make_batch  # noqa: E402
from scripts.tda_probe import card  # noqa: E402

WORKLOADS = {"W1": (64, 256, 256), "W2": (64, 496, 512)}
Q, TOL = 95.0, 1.0


def composed(P, T, q=Q, tol=TOL):
    """[4, n] float32 from torch ops over distance_transform_edt; distances are the transform's float32 roots."""
    H, W = P.shape[-2:]

    def surface(M):
        pad = F.pad(M.reshape(-1, 1, H, W).to(torch.uint8), (1, 1, 1, 1))
        inner = pad[..., :-2, 1:-1] & pad[..., 2:, 1:-1] & pad[..., 1:-1, :-2] & pad[..., 1:-1, 2:]
        return (M.reshape(-1, 1, H, W) & (inner == 0)).reshape(-1, H * W)

    Sp, St = surface(P), surface(T)
    d_pt = torch.where(Sp, tlb.distance_transform_edt((~St).reshape(-1, H, W)).reshape(-1, H * W), torch.inf)
    d_tp = torch.where(St, tlb.distance_transform_edt((~Sp).reshape(-1, H, W)).reshape(-1, H * W), torch.inf)
    n_p, n_t = Sp.sum(1), St.sum(1)

    def pct(d, n):
        s = torch.sort(d, dim=1).values.double()
        h = (n - 1).clamp_min(0).double() * (q / 100.0)
        lo = h.floor().long().clamp(0, H * W - 1)
        hi = (lo + 1).clamp(max=H * W - 1)
        a, b = s.gather(1, lo[:, None])[:, 0], s.gather(1, hi[:, None])[:, 0]
        g = h - lo.double()
        diff = b - a
        v = torch.where(g >= 0.5, b - diff * (1 - g), a + diff * g)
        return torch.where(h >= (n - 1).double(), s.gather(1, (n - 1).clamp_min(0)[:, None])[:, 0], v)

    fin_pt, fin_tp = torch.where(Sp, d_pt, 0.0).double(), torch.where(St, d_tp, 0.0).double()
    hd = torch.maximum(torch.where(Sp, d_pt, -1.0).amax(1), torch.where(St, d_tp, -1.0).amax(1)).double()
    hp = torch.maximum(pct(d_pt, n_p), pct(d_tp, n_t))
    tot = (n_p + n_t).double()
    assd = (fin_pt.sum(1) + fin_tp.sum(1)) / tot
    nsd = (((d_pt <= tol) & Sp).sum(1) + ((d_tp <= tol) & St).sum(1)).double() / tot
    one = (n_p == 0) ^ (n_t == 0)
    none = (n_p == 0) & (n_t == 0)
    out = torch.stack([hd, hp, assd, nsd])
    out = torch.where(one, torch.tensor([torch.inf, torch.inf, torch.inf, 0.0], device=P.device, dtype=torch.float64)[:, None], out)
    return torch.where(none, torch.nan, out).float()


def scipy_metrics(p, t, q=Q, tol=TOL):
    """One map pair on the host: surfaces by binary_erosion, two scipy transforms, np.percentile, float64."""
    Sp, St = p & ~ndi.binary_erosion(p, border_value=0), t & ~ndi.binary_erosion(t, border_value=0)
    if not Sp.any() and not St.any():
        return [np.nan] * 4
    if not Sp.any() or not St.any():
        return [np.inf, np.inf, np.inf, 0.0]
    d_pt, d_tp = ndi.distance_transform_edt(~St)[Sp], ndi.distance_transform_edt(~Sp)[St]
    n = len(d_pt) + len(d_tp)
    return [max(d_pt.max(), d_tp.max()), max(np.percentile(d_pt, q), np.percentile(d_tp, q)),
            (d_pt.sum() + d_tp.sum()) / n, ((d_pt <= tol).sum() + (d_tp <= tol).sum()) / n]


def max_diff(a, b):
    """Largest |a - b| over entries finite in both, and the number of entries whose nan / inf pattern differs."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    fin = np.isfinite(a) & np.isfinite(b)
    pattern = int((~fin & ~((np.isnan(a) & np.isnan(b)) | (a == b))).sum())
    return float(np.abs(a[fin] - b[fin]).max()) if fin.any() else 0.0, pattern


def run(name, B, H, W, a):
    pred, truth = make_batch(B, H, W, seed=0, device="cuda")
    P, T = pred > 0.5, truth > 0.5
    del pred, truth
    n = P.numel() // (H * W)
    forms = {"op": lambda: torch.stack(list(tlb.surface_distances(P, T, Q, TOL))).reshape(4, n),
             "composed": lambda: composed(P, T)}
    outs, times = {}, {k: [] for k in forms}
    for form in forms:
        for _ in range(a.warmup):
            outs[form] = forms[form]()
    torch.cuda.synchronize()
    for _, form in itertools.product(range(a.steps), forms):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        forms[form]()
        ev[1].record()
        ev[1].synchronize()
        times[form].append(ev[0].elapsed_time(ev[1]))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    res = {"shape": [B, int(P.shape[1]), H, W], "forms": {}}
    for form in forms:
        t = sorted(times[form])
        res["forms"][form] = {"ms_median": round(med[form], 3), "ms_min": round(t[0], 3), "ms_max": round(t[-1], 3)}
    res["forms"]["op"]["x_composed"] = round(med["op"] / med["composed"], 3)
    op, comp = outs["op"].cpu().numpy(), outs["composed"].cpu().numpy()
    fields = ("hausdorff", "hausdorff_percentile", "assd", "nsd")
    res["forms"]["op"]["max_abs_diff_vs_composed"] = {f: max_diff(op[i], comp[i])[0] for i, f in enumerate(fields)}
    res["forms"]["op"]["nonfinite_pattern_mismatches_vs_composed"] = sum(max_diff(op[i], comp[i])[1] for i in range(4))
    res["forms"]["op"]["nan_maps"] = int(np.isnan(op[0]).sum())
    res["forms"]["op"]["median_hd95"] = float(np.nanmedian(op[1]))
    # the host path on the first maps
    Ph = P.reshape(-1, H, W)[: a.scipy_maps].cpu().numpy()
    Th = T.reshape(-1, H, W)[: a.scipy_maps].cpu().numpy()
    t0 = time.perf_counter()
    host = np.array([scipy_metrics(p, t) for p, t in zip(Ph, Th)], dtype=np.float64).T
    dt = (time.perf_counter() - t0) * 1e3 / Ph.shape[0]
    sub = op[:, : Ph.shape[0]]
    res["forms"]["scipy"] = {"ms_per_map": round(dt, 3), "maps_timed": int(Ph.shape[0]),
                             "ms_per_batch_extrapolated": round(dt * n, 1), "host_cores": os.cpu_count(), "threads": 1,
                             "max_abs_diff_op_vs_scipy": {f: max_diff(sub[i], host[i].astype(np.float32))[0]
                                                          for i, f in enumerate(fields)},
                             "nonfinite_pattern_mismatches": sum(max_diff(sub[i], host[i])[1] for i in range(4))}
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
        sys.exit("surface_probe.py needs a CUDA device")
    torch.cuda.set_device(0)
    gpu, limits = card()
    res = {"probe": "scripts/surface_probe.py", "gpu": gpu, "power_limit_and_max_sm_clock": limits,
           "inputs": f"synthetic.make_batch(seed=0): pred > 0.5 against truth > 0.5; percentile {Q}, tolerance {TOL}",
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
