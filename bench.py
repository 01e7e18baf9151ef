#!/usr/bin/env python
"""Headline benchmark: topological-loss forward + backward throughput on synthetic
256x256 x 14-class maps (BASELINE.json configs[1]: bs = 64 per GPU, interp = 0, feat_d = 1, q = 2,
lamda = 0.1), reported as masks/s (one mask = one image's 14-class stack = 14 maps).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle port on host cores
    python bench.py --steps K --warmup W --dump-outputs DIR   # also write the last timed step's outputs

Under torchrun (N > 1) every rank processes its own 64 images (weak scaling); the only collective is
the all-reduce of the scalar loss.  Rank 0 prints ONE JSON line.

--dump-outputs DIR writes what the last timed (device-resident) step handed its caller, so that two builds can be
compared output for output on identical seeded inputs: DIR/loss.npy (float32, 0-d) and DIR/grad_sample.npy
(float32, rank 0's gradient d loss / d pred flattened and taken at sample_index(pred.numel()), a fixed seeded
set of at most DUMP_MAX_ELEMS positions: 32 MB).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C = 14
LAMDA, FEAT_D, LOSS_Q = 0.1, 1, 2
ALGO_BYTES_PER_PIXEL = 12  # read pred fp32 + read truth fp32 + write grad fp32 (SURVEY.md 8d)
E2E_CHUNKS = 16  # upper bound on the groups of whole images whose H2D copy overlaps the previous group's kernels
# BASELINE.json configs: c2 = configs[1], the headline (256^2 x 14, bs 64 per GPU); c5 = configs[4], the
# full-resolution stress test (1024^2 x 14, bs 128 over 8 GPUs = 16 images per GPU)
CONFIGS = {"c2": dict(side=256, batch=64, seed=2, name="C2"), "c5": dict(side=1024, batch=16, seed=5, name="C5")}
METRIC = "topo-loss fwd+bwd masks/sec (256^2, 14 cls)"
DUMP_SEED = 0
DUMP_MAX_ELEMS = 1 << 23  # float32 gradient positions written by --dump-outputs (32 MB)


def input_seed(cfg, rank=0):
    """Seed of make_batch for a config's inputs on one rank: the same arguments give the same inputs."""
    return 1234 + 1000 * cfg["seed"] + rank


def sample_index(n: int):
    """Sorted flat positions of the fixed, seeded sample that --dump-outputs takes of an n-element output."""
    import torch
    if n <= DUMP_MAX_ELEMS:
        return torch.arange(n)
    g = torch.Generator().manual_seed(DUMP_SEED)
    return torch.unique(torch.randint(0, n, (DUMP_MAX_ELEMS,), generator=g))


def dump_outputs(out_dir, loss, grad):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    flat = grad.detach().reshape(-1)
    sample = flat[sample_index(flat.numel()).to(flat.device)]
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "grad_sample.npy"), sample.float().cpu().numpy())


def _metric(side):
    return METRIC if side == 256 else f"topo-loss fwd+bwd masks/sec ({side}^2, 14 cls)"


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _host_cores() -> int:
    """Threads the CPU arm uses: every core this process may run on.  (torchrun exports
    OMP_NUM_THREADS=1; the oracle's num_threads() clause overrides it.)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 5.0:  # nvidia-smi takes a few 100 ms to start streaming:
                time.sleep(0.01)                            # the timed region (tens of ms) must not be over by then
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark(self):
        """Start of the timed region: samples before this point are dropped (if any remain after)."""
        self.first = len(self.rows)

    def mark_end(self):
        """End of the device-timed region (the sampler keeps running through the end-to-end region)."""
        self.last = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        first, last = getattr(self, "first", 0), getattr(self, "last", None)
        window = "timed region"
        if last is not None and last > first:
            self.rows = self.rows[first:last]
        elif len(self.rows) > first:  # the device-timed region was shorter than one sampling period
            self.rows = self.rows[first:]
            window = "timed + end-to-end region"
        else:
            window = "before the timed region"
        self.window = window
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "window": self.window}


class NvmlSampler:
    """The same reading through NVML (nvidia_ml_py) from a thread of this process, every millisecond: the
    device-timed region is only tens of milliseconds long, which nvidia-smi's 20 ms loop samples once or twice.
    Samples carry a host timestamp; the ones between mark() and mark_end() are reported."""
    HW_SLOWDOWN, SW_POWER_CAP, SW_THERMAL, HW_THERMAL = 0x8, 0x4, 0x20, 0x40

    def __init__(self, index: int, uuid: str = ""):
        self.rows, self.ok, self.stop_flag = [], False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            h = None
            if uuid:
                for u in (uuid, uuid.encode()):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(u)
                        break
                    except Exception:
                        h = None
            self.h = h if h is not None else pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._read()
            self.ok = True
        except Exception:
            self.ok = False

    def _read(self):
        nv = self.nv
        sm = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        try:
            why = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            why = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        return time.perf_counter(), sm, why

    def start(self):
        def pump():
            while not self.stop_flag:
                try:
                    self.rows.append(self._read())
                except Exception:
                    pass
                time.sleep(0.001)
        self.t = threading.Thread(target=pump, daemon=True)
        self.t.start()

    def mark(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        self.stop_flag = True
        self.t.join(timeout=2)
        t0, t1 = getattr(self, "t0", 0.0), getattr(self, "t1", float("inf"))
        rows, window = [r for r in self.rows if t0 <= r[0] <= t1], "timed region"
        if not rows:
            rows, window = [r for r in self.rows if r[0] >= t0] or self.rows, "timed + end-to-end region"
        sm = sorted(r[1] for r in rows)
        bits = 0
        for r in rows:
            bits |= r[2]
        names = [("hw_slowdown", self.HW_SLOWDOWN), ("hw_thermal_slowdown", self.HW_THERMAL),
                 ("sw_thermal_slowdown", self.SW_THERMAL), ("sw_power_cap", self.SW_POWER_CAP)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm,
                "reasons": [n for n, b in names if bits & b], "samples": len(sm), "window": window,
                "source": "NVML, 1 ms period"}


def make_sampler(index: int, uuid: str = ""):
    s = NvmlSampler(index, uuid)
    return s if s.ok else ClockSampler(index)


def cpu_arm(pred, truth, nthreads, steps, warmup):
    """Oracle port (oracle/topo_oracle.c) forward + backward on host cores; returns masks/s."""
    import oracle
    p, t = pred.numpy(), truth.numpy()
    for _ in range(warmup):
        oracle.topo_loss(p, t, LAMDA, feat_d=FEAT_D, loss_q=LOSS_Q, nthreads=nthreads)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle.topo_loss(p, t, LAMDA, feat_d=FEAT_D, loss_q=LOSS_Q, nthreads=nthreads)
    dt = (time.perf_counter() - t0) / max(1, steps)
    return p.shape[0] / dt, dt


def run_reference(args, rank, world):
    """--impl reference: the reference's own implementation cannot run here (torch_topological /
    gudhi / POT absent, SURVEY.md 8c), so this arm times the oracle port -- the CPU restatement of
    the same path -- with all host threads, on the same per-GPU batch as our arm (a bounded sample of it
    with --ref-images N)."""
    if rank != 0:
        return
    import torch
    import oracle
    from dilabhelmholtzoct_b200.synthetic import make_batch
    cfg = CONFIGS[args.config]
    H = W = cfg["side"]
    B = args.batch or cfg["batch"]
    cores = _host_cores()
    sample = min(args.ref_images or B, B)
    pred, truth = make_batch(B, H, W, seed=input_seed(cfg), device="cpu")
    pred, truth = pred[:sample].contiguous(), truth[:sample].contiguous()
    value, dt = cpu_arm(pred, truth, cores, args.steps, max(1, min(args.warmup, 1)))
    what = "the whole batch" if sample == B else f"the first {sample} of {B} images"
    line = {
        "impl": "reference", "metric": _metric(H), "value": value, "unit": "masks/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{cfg['name']} topo-loss fwd+bwd, fp32[{B},{C},{H},{W}] per GPU, interp=0 feat_d=1 q=2 lamda=0.1",
                   "sample_per_step": f"{what} ({sample * C} maps) per step, same seed as the GPU arm"},
        "cpu_baseline": {"value": value, "unit": "masks/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} images x {C} classes per step, OpenMP over maps, oracle/topo_oracle.c"},
        "e2e": {"value": value, "unit": "masks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


_SAVED_STDOUT = None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json workload (c2 = headline)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: the config's)")
    ap.add_argument("--ref-images", type=int, default=0, help="images per step of the CPU arm (default: the whole batch)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="images of the cpu_baseline sample (default: ~10 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's loss and a seeded sample of its "
                                                          "gradient as DIR/<name>.npy (CUDA path only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's outputs (--impl ours)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import dilabhelmholtzoct_b200 as tlb
    from dilabhelmholtzoct_b200 import _lib
    from dilabhelmholtzoct_b200.parallel import reduce_scalar_async, topo_loss_sharded
    from dilabhelmholtzoct_b200.synthetic import make_batch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the topological loss has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version / debug lines on stdout (fd 1) when it initialises: park fd 1 on stderr for
        # the whole run and give it back just before the one JSON line is printed
        sys.stdout.flush()
        global _SAVED_STDOUT
        _SAVED_STDOUT = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    cfg = CONFIGS[args.config]
    H = W = cfg["side"]
    B = args.batch or cfg["batch"]
    gb = B * world

    pred, truth = make_batch(B, H, W, seed=input_seed(cfg, rank), device=dev)
    pred_h = pred.cpu().pin_memory()
    # one-hot ground truth is {0, 1}: it crosses PCIe as bits (numpy.packbits) and is widened on the device
    # (the reference builds these masks on the CPU, training_utils.py:413, :432)
    truth_h = tlb.pack_mask_bits(truth.cpu())
    p = pred.clone().requires_grad_(True)

    def step_resident():
        p.grad = None
        if world > 1:
            # this rank's share of the global mean; the scalar all-reduce runs behind a side stream while the
            # backward (which does not depend on it) proceeds
            part = topo_loss_sharded(p, truth, LAMDA, feat_d=FEAT_D, loss_q=LOSS_Q, global_batch=gb, reduce="local")
            total = reduce_scalar_async(part)
            part.backward()
            return total.result()
        loss = tlb.topo_loss(p, truth, LAMDA, feat_d=FEAT_D, loss_q=LOSS_Q)
        loss.backward()
        return loss

    def step_e2e():
        # host-resident (pinned) inputs through the public host API: H2D copies are pipelined against
        # the kernels in E2E_CHUNKS groups of whole images; loss read back to the host every step
        loss, grad = tlb.topo_loss_from_host(pred_h, truth_h, LAMDA, feat_d=FEAT_D, loss_q=LOSS_Q, chunks=E2E_CHUNKS,
                                             truth_packed=True)
        if world > 1:
            loss = loss * (1.0 / world)  # every rank holds lamda * mean over ITS images
            dist.all_reduce(loss, op=dist.ReduceOp.SUM)
        return float(loss.cpu())  # device -> host read of the step's result (the gradient stays on the device)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps, out  # out: what the last step returned

    try:
        uuid = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        uuid = ""
    sampler = make_sampler(local_rank, uuid)
    if rank == 0:
        try:
            sampler.start()
        except Exception:
            sampler = ClockSampler(local_rank)
            sampler.start()
    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    if rank == 0:
        sampler.mark()
    L.tl_timing_enable(1)
    ms_step, last_loss = timed(step_resident, args.steps)
    sums = (ctypes.c_float * 6)()
    calls = (ctypes.c_int * 2)()
    L.tl_timing_read(sums, calls)
    L.tl_timing_enable(0)
    if rank == 0:
        sampler.mark_end()

    for _ in range(3):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    clocks = None
    if rank == 0:
        try:
            clocks = sampler.stop()
        except Exception as e:  # the clock record must never cost the bench line
            clocks = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"sampler failed: {type(e).__name__}"]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:  # the end-to-end steps use their own buffers: p.grad is still the last timed step's
        dump_outputs(args.dump_outputs, last_loss, p.grad)

    value = gb / (ms_step * 1e-3)
    e2e_value = gb / (ms_e2e * 1e-3)
    peak, peak_src = _peaks()
    stages = ["persistence", "unused_sort", "matching", "loss", "unused", "grad_fill_scatter"]
    nf, nb = max(1, calls[0]), max(1, calls[1])
    stage_ms = {s: (sums[i] / (nf if i < 4 else nb)) for i, s in enumerate(stages)}
    dom = max(stage_ms, key=stage_ms.get)
    algo_bytes = ALGO_BYTES_PER_PIXEL * H * W * B * C  # per launch: one launch covers this GPU's B*C maps
    achieved = algo_bytes / (stage_ms[dom] * 1e-3) / 1e9 if stage_ms[dom] > 0 else 0.0
    traffic, traffic_src = None, None
    try:  # static: dram__bytes of the dominant kernel from the committed ncu launch list of this command
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        traffic = tj.get(args.config, {}).get(dom)
        traffic_src = tj.get("source")
    except Exception:
        pass
    line = {
        "metric": _metric(H), "value": value, "unit": "masks/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{cfg['name']} topo-loss fwd+bwd, fp32[{B},{C},{H},{W}] per GPU, interp=0 feat_d=1 q=2 lamda=0.1",
                   "maps_per_s": value * C, "l2": "inputs (2 x %.0f MB per GPU) larger than the 126 MB L2" % (pred.numel() * 4 / 1e6),
                   "parallelism": f"dp{world} (batch axis sharded, scalar-loss all-reduce only)"},
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": algo_bytes, "stage_ms": stage_ms,
                     "whole_step_frac": (algo_bytes / (ms_step * 1e-3) / 1e9) / peak,
                     "stage_note": "the persistence launch also runs the matching and writes the gradient in its tail "
                                   "(tl_forward_backward); grad_fill_scatter is the launch for the images it left over"},
        "e2e": {"value": e2e_value, "unit": "masks/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(pred_h.numel() * pred_h.element_size() + truth_h.numel() * truth_h.element_size()),
                "d2h_bytes_per_step": 4, "grad": "device-resident (only the 4-byte loss is read back)",
                "api": f"topo_loss_from_host(pinned fp32 pred, pinned bit-packed {{0,1}} truth, chunks={E2E_CHUNKS}): H2D pipelined against the kernels"},
        # per step: persistence (+ matching + gradient in its tail), general matching (empty list), loss, gradient of the
        # images the tail left over (none here), gradient scaling (returns at once for an upstream gradient of 1)
        "gpu_launches": 5 * args.steps,
        "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        import oracle
        cores = _host_cores()
        n = min(args.cpu_sample or B, B)
        truth_f = truth[:n].cpu()
        passes = 1
        v, dt = cpu_arm(pred_h[:n], truth_f, cores, 1, 0)
        if dt < 2.5:  # bounded sample of ~10 s of CPU work: repeat the pass
            passes = max(1, min(8, int(10.0 / max(dt, 1e-3))))
            v, dt = cpu_arm(pred_h[:n], truth_f, cores, passes, 0)
        line["cpu_baseline"] = {"value": v, "unit": "masks/s", "cores": cores, "kind": "port",
                                "sample": f"first {n} images ({n * C} maps) of the same batch, {passes} pass(es) of {dt:.2f} s, "
                                          f"oracle/topo_oracle.c with OpenMP over maps"}
    if _SAVED_STDOUT is not None:
        sys.stdout.flush()
        os.dup2(_SAVED_STDOUT, 1)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
