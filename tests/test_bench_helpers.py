"""CPU-only: arithmetic helpers of bench.py (no GPU, no engine)."""
import importlib.util
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_algorithmic_bytes_match_design_table():
    b = _bench()
    n = 65536
    assert b.algorithmic_bytes("knn_covariance", n, n, 32) == n * 64
    assert b.algorithmic_bytes("gicp_correspondences", n, n, 32) == 16 * 2 * n + 16 * n
    assert b.algorithmic_bytes("gicp_linearize", n, n, 32) == 248 * n + 232
    assert b.algorithmic_bytes("no_such_class", n, n, 32) is None


def test_whole_step_algorithmic_throughput():
    b = _bench()
    n = 65536
    calls = {"knn_covariance": 200, "gicp_correspondences": 974, "gicp_linearize": 974, "misc": 7, "nn_fitness": 0}
    gbs, per_step, unknown = b.whole_step_algorithmic_gbs(calls, n, n, 32, 92.6, 200)
    want = 200 * n * 64 + 974 * (48 * n) + 974 * (248 * n + 232)
    assert per_step == want / 200 and unknown == ["misc"]
    assert abs(gbs - want / 92.6e-3 / 1e9) < 1e-9
    assert b.whole_step_algorithmic_gbs(calls, n, n, 32, 0.0, 200) is None


def test_dump_outputs_writes_float32_or_float64(tmp_path):
    import numpy as np
    b = _bench()
    T = np.arange(16, dtype=np.float32).reshape(4, 4)
    b.dump_outputs(str(tmp_path / "d"), {"odom": T, "iterations": 7, "converged": True})
    assert sorted(os.listdir(tmp_path / "d")) == ["converged.npy", "iterations.npy", "odom.npy"]
    odom, it, conv = (np.load(tmp_path / "d" / f"{k}.npy") for k in ("odom", "iterations", "converged"))
    assert odom.dtype == np.float32 and np.array_equal(odom, T)
    assert it.dtype == np.float64 and it == 7.0 and conv.dtype == np.float64 and conv == 1.0


def test_reference_arm_line_has_the_contract_keys(oracle, synth):
    """`bench.py --impl reference` (the CPU oracle replaying the same workload) prints ONE JSON line with the driver's keys"""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--workload", "gicp_odometry_vlp16_64k"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "registrations/sec" and d["higher_is_better"] is True and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]


def test_loop_workload_identical_shards_for_weak_scaling():
    """bench.py --gpus N: every rank's contiguous shard of the loop-closure batch is the same keyframe groups and guesses (per-GPU work
    exactly fixed), and the N = 1 workload is untouched by the option"""
    import numpy as np
    from hdl_graph_slam_b200 import batch
    g1, q1, f1 = batch.loop_workload(4)
    g1b, q1b, f1b = batch.loop_workload(4, period=4)
    assert g1 == g1b and np.array_equal(q1, q1b) and f1 == f1b
    g, q, f = batch.loop_workload(12, period=4)
    assert f == [8 * i for i in range(13)]
    for r in range(3):
        g0, gend = batch.shard_range(12, 3, r)
        assert (g0, gend) == (4 * r, 4 * r + 4)
        assert g[g0:gend] == g1 and np.array_equal(q[f[g0]:f[gend]], q1)


def test_auxiliary_workloads_have_no_reference_arm_but_say_so():
    """the voxel-grid / KITTI-chain workloads carry their CPU figure as cpu_baseline; --impl reference answers with one JSON line"""
    import json
    import subprocess
    import sys
    for wl in ("voxelgrid", "kitti_pipeline"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", wl], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stderr
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["impl"] == "reference" and "unavailable" in line


def test_clock_sampler_window_and_hold(tmp_path, monkeypatch):
    """ClockSampler keeps the samples whose timestamps lie inside [begin(), stop()] and holds untimed steps until the window is long
    enough for nvidia-smi; without nvidia-smi it says so and never holds"""
    import datetime
    import time
    b = _bench()
    s = b.ClockSampler(0)
    s.p = None  # nvidia-smi unavailable
    assert not s.hold_needed()
    calls = []
    s.hold(lambda k: calls.append(k), lambda: None)
    assert calls == [] and s.stop()["samples"] == 0 and "nvidia-smi unavailable" in s.stop()["reasons"]
    # a fake nvidia-smi log: one sample before the window, two inside (one of them throttled), one malformed line
    s = b.ClockSampler(0)
    s.path = str(tmp_path / "clocks.csv")

    class P:  # stands in for the nvidia-smi process
        def terminate(self): pass
        def wait(self, timeout=None): return 0
        def kill(self): pass
    s.p, s.f = P(), open(s.path, "w")
    s.MIN_WINDOW_S = 0.05
    s.begin()
    fmt = "%Y/%m/%d %H:%M:%S.%f"
    def line(t, mhz, power_cap):
        return ", ".join([datetime.datetime.fromtimestamp(t).strftime(fmt)[:-3], str(mhz), "1965", "400.0", "0x0", "Not Active", "Not Active", "Not Active", power_cap]) + "\n"
    s.f.write(line(s.t0 - 5.0, 345, "Not Active"))
    s.f.write(line(s.t0 + 0.01, 1965, "Not Active"))
    s.f.write(line(s.t0 + 0.02, 1950, "Active"))
    s.f.write("garbage\n")
    s.f.flush()
    steps = []
    s.hold(lambda k: (steps.append(k), time.sleep(0.01)), lambda: None)
    assert len(steps) >= 3 and s.extra_steps == len(steps)
    out = s.stop()
    assert out["samples"] == 2 and out["sm_mhz"] == 1957.5 and out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"]
    assert "untimed steps" in out["window"]
