"""bench.py's CPU-runnable leg (--impl reference: the oracle port on the host cores) prints one JSON line with the
contract's keys; the GPU leg refuses to run without a device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--envs", "64", "--frames", "80"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-500:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "env_steps_per_sec" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True,
                         text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)


def _bench_module():
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench
    return bench


def test_dump_outputs_sample_stays_under_the_limit(tmp_path):
    """Above the size limit --dump-outputs writes the same seeded sample of envs from every array, and lists it."""
    import numpy as np
    import torch
    import aigar_b200.layout as lay
    bench = _bench_module()

    class Batch(object):  # the AgarBatch surface dump_outputs reads, on the CPU
        n_envs = 1000
        obs = torch.arange(1000 * 123, dtype=torch.float32).reshape(1000, 1, 123)

        def get(self, which):
            if which == lay.GET_STATS:
                return torch.arange(4000, dtype=torch.float64).reshape(1000, 1, 4)
            if which in (lay.GET_OVERFLOW, lay.GET_EVENT_HASH):
                return torch.arange(1000, dtype=torch.int64 if which == lay.GET_EVENT_HASH else torch.int32) - 3
            return torch.arange(1000, dtype=torch.int32).reshape(1000, 1)

    for limit, kept in ((1 << 30, 1000), (200000, None)):
        d = tmp_path / str(limit)
        bench.dump_outputs(Batch(), str(d), limit=limit)
        out = {f[:-4]: np.load(str(d / f)) for f in os.listdir(str(d))}
        assert sum(os.path.getsize(str(d / f)) for f in os.listdir(str(d))) <= limit
        assert set(bench.DUMP_GETTERS) | {"obs", "event_hash"} <= set(out)
        assert all(v.dtype in (np.float32, np.float64) for v in out.values())
        assert sum(v.nbytes for v in out.values()) <= limit
        if kept is None:
            idx = out["env_index"].astype(np.int64)
            assert 0 < len(idx) < 1000 and np.all(np.diff(idx) > 0)
        else:
            assert "env_index" not in out
            idx = np.arange(kept)
        assert np.array_equal(out["obs"][:, 0, 0], idx * 123) and np.array_equal(out["reward"][:, 0], idx)
        h = (idx - 3).astype(np.uint64)
        assert np.array_equal(out["event_hash"], np.stack([h >> np.uint64(32), h & np.uint64(0xFFFFFFFF)], -1).astype(np.float64))
        assert np.array_equal(out["overflow"], (idx - 3).astype(np.int32).view(np.uint32).astype(np.float64))


@pytest.mark.gpu
def test_dump_outputs_repeat_and_follow_steps(tmp_path):
    """--dump-outputs: the same arguments give the same arrays; --steps sets the number of timed launches, and one more step
    changes what the last one computed."""
    import numpy as np

    def run(steps, d):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--envs", "256",
                              "--frames", "80", "--no-extra", "--no-cpu", "--no-e2e", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["gpu_launches"] == steps
        return {f[:-4]: np.load(str(d / f)) for f in os.listdir(str(d))}

    a, b, c = run(2, tmp_path / "a"), run(2, tmp_path / "b"), run(3, tmp_path / "c")
    assert "obs" in a and a["obs"].shape[0] == 256 and sorted(a) == sorted(b) == sorted(c)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["event_hash"], c["event_hash"])


def test_clock_sampler_degrades_without_a_gpu():
    """ClockSampler reads NVML in-process (fallback: nvidia-smi); without a driver both are absent and the contract's `clocks`
    object carries nulls instead of raising."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler(0)
    s.start()
    res = s.stop()
    assert set(("sm_mhz", "sm_max_mhz", "reasons")) <= set(res) and res["reasons"] == []
