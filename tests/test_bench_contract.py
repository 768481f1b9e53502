"""The reference arm of bench.py (``--impl reference``: the unmodified reference on the host cores) runs without a GPU:
its JSON line must carry the keys the driver reads, with the metric / unit / config of the CUDA arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line(built):
    from oracle import oracle_binding as ob
    if not ob.have_ref():
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "32", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert len(out.stdout.strip().splitlines()) == 1            # the contract: ONE line on stdout
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype",
                "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "QP/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert "nx=21 nu=3 N=40" in line["config"]["workload"]


def test_other_configuration_and_thread_team(built):
    """``--config`` selects another BASELINE.json shape for the same line; the thread team of the host arms is the affinity mask
    capped by the cgroup CPU quota (a 128-CPU mask with a 16-CPU quota must not get 128 threads)."""
    from acados_b200.binding import host_threads
    nt = host_threads()
    assert 1 <= nt <= len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            assert nt <= -(-int(quota) // int(period))
    except OSError:
        pass
    # without the reference library the host arm times the oracle port: the same line, the same thread team
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c3", "--batch", "64", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip())
    assert "pendulum" in line["metric"] and line["config"]["name"] == "c3" and "nx=4 nu=1 N=20" in line["config"]["workload"]
    assert line["cpu_baseline"]["cores"] == nt
