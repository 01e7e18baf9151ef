"""bench.py's CPU arm (`--impl reference`) runs without a GPU: one JSON line on stdout with the keys the
driver reads, same metric / unit / config as the GPU arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--ref-images", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "masks/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("topo-loss fwd+bwd masks/sec")
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1", "--ref-images", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_nvml_clock_sampler_with_a_fake_nvml(monkeypatch):
    """The in-process NVML sampler: samples between mark() and mark_end() only, median clock, reason bits -> names;
    without NVML (this container) make_sampler falls back to the nvidia-smi loop."""
    import sys
    import time
    import types
    import bench
    assert type(bench.make_sampler(0)).__name__ == "ClockSampler"  # no libnvidia-ml here
    fake = types.ModuleType("pynvml")
    state = {"why": 0}
    fake.NVML_CLOCK_SM = 1
    fake.nvmlInit = lambda: None
    fake.nvmlDeviceGetHandleByUUID = lambda u: (_ for _ in ()).throw(RuntimeError("no such uuid"))
    fake.nvmlDeviceGetHandleByIndex = lambda i: ("handle", i)
    fake.nvmlDeviceGetMaxClockInfo = lambda h, k: 1965
    fake.nvmlDeviceGetClockInfo = lambda h, k: 1950
    fake.nvmlDeviceGetCurrentClocksEventReasons = lambda h: state["why"]
    monkeypatch.setitem(sys.modules, "pynvml", fake)
    s = bench.make_sampler(0, "GPU-123")
    assert type(s).__name__ == "NvmlSampler" and s.h == ("handle", 0)
    s.start()
    time.sleep(0.02)
    state["why"] = 0x4 | 0x1  # sw_power_cap + gpu_idle (ignored)
    s.mark()
    time.sleep(0.03)
    s.mark_end()
    state["why"] = 0x8        # after the window: must not be reported
    time.sleep(0.01)
    out = s.stop()
    assert out["sm_mhz"] == 1950 and out["sm_max_mhz"] == 1965 and out["samples"] >= 5
    assert out["reasons"] == ["sw_power_cap"] and out["window"] == "timed region"


def test_bad_steps_and_dump_without_the_cuda_path_are_rejected(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=300, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "" and "error" in out.stderr, extra
    assert os.listdir(tmp_path) == []


def test_dump_sample_is_fixed_sorted_and_bounded():
    import bench
    small = bench.sample_index(1000)
    assert small.tolist() == list(range(1000))
    n = 64 * 14 * 256 * 256
    a, b = bench.sample_index(n), bench.sample_index(n)
    assert a.equal(b) and 0.9 * bench.DUMP_MAX_ELEMS < a.numel() <= bench.DUMP_MAX_ELEMS
    assert bool((a[1:] > a[:-1]).all()) and int(a[0]) >= 0 and int(a[-1]) < n
    assert a.numel() * 4 + 4096 <= 64 << 20  # float32 sample + loss + .npy headers stay under 64 MB


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs writes the loss and the sampled gradient of the resident path; on the same seeded inputs the
    oracle computes the same values.  Ten images: the gradient has more positions than the sample holds."""
    import bench
    import oracle
    from dilabhelmholtzoct_b200.synthetic import make_batch
    B = 10
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", str(B),
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2 and d["gpu_launches"] == 10
    assert sorted(os.listdir(tmp_path)) == ["grad_sample.npy", "loss.npy"]
    loss, grad = np.load(tmp_path / "loss.npy"), np.load(tmp_path / "grad_sample.npy")
    cfg = bench.CONFIGS["c2"]
    pred, truth = make_batch(B, cfg["side"], cfg["side"], seed=bench.input_seed(cfg), device="cuda")
    want, wgrad, _ = oracle.topo_loss(pred.cpu().numpy(), truth.cpu().numpy(), bench.LAMDA, feat_d=bench.FEAT_D,
                                      loss_q=bench.LOSS_Q, nthreads=os.cpu_count() or 1)
    idx = bench.sample_index(wgrad.size).numpy()
    assert wgrad.size > bench.DUMP_MAX_ELEMS and grad.shape == idx.shape
    assert loss.dtype == np.float32 and loss.shape == () and abs(float(loss) - want) <= 1e-5 * abs(want)
    assert grad.dtype == np.float32
    assert np.abs(grad - wgrad.reshape(-1)[idx]).max() <= 1e-5 * np.abs(wgrad).max()
    assert np.count_nonzero(grad) > 0
