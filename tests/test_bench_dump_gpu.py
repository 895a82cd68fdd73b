"""GPU: `bench.py --dump-outputs DIR` writes what the last timed step of the odometry chain returned, bit for bit what the same chain
gives when it is replayed call by call through the library, and `--steps` / `--warmup` set the frames it runs."""
import json
import os
import subprocess
import sys
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_equal_the_replayed_chain(synth, tmp_path):
    import hdl_graph_slam_b200 as pkg
    K, W = 4, 2
    out_dir = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(K), "--warmup", str(W), "--no-anchor", "--no-profile",
                        "--cpu-sample", "0", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=tmp_path)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == K and line["warmup"] == W
    d = {f[:-4]: np.load(out_dir / f) for f in os.listdir(out_dir)}
    assert sorted(d) == sorted(["odom", "trans", "converged", "iterations", "keyframe_updated", "frame_rejected"])
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    # the bench's chain: the first keyframe, W warm-up frames, then K timed frames of the same seeded sequence
    reg = pkg.select_registration_method({"registration_method": "FAST_GICP"})
    odo = pkg.ScanMatchingOdometry(reg, keyframe_delta_trans=1.0, keyframe_delta_angle=1.0, keyframe_delta_time=10000.0)
    for i in range(W + 1 + K):
        st = odo.matching(0.1 * i, synth.scan("vlp16", frame=i, stride=8))
    odo.close()
    reg.close()
    assert np.array_equal(d["odom"], st["odom"]) and np.array_equal(d["trans"], st["trans"])
    for k in ("converged", "iterations", "keyframe_updated", "frame_rejected"):
        assert float(d[k]) == float(st[k]), k
