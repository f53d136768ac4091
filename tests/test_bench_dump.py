"""bench.py --dump-outputs: the pose and HoleMap after the last timed step of the cfg2 line, written as float32 .npy files,
equal the CPU oracle's after the same scans (so two builds can be compared through their dumps)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, cwd=ROOT,
                          timeout=timeout)


@pytest.mark.parametrize("extra", [["--impl", "reference"], ["--workload", "cfg3"], ["--streaming"]])
def test_dump_outputs_is_refused_where_it_has_no_timed_replay(extra, tmp_path):
    r = _run(extra + ["--steps", "2", "--warmup", "3", "--dump-outputs", str(tmp_path / "out")], timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_equal_the_oracle_after_the_timed_steps(tmp_path):
    K, W, seed = 4, 3, 1234
    out = tmp_path / "out"
    r = _run(["--steps", str(K), "--warmup", str(W), "--seed", str(seed), "--no-cpu-baseline", "--no-sharded",
              "--dump-outputs", str(out)])
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == K and line["warmup"] == W
    assert sorted(os.listdir(out)) == ["hole_map.npy", "pose.npy"]
    pose, hole = np.load(out / "pose.npy"), np.load(out / "hole_map.npy")
    wl = bench.WORKLOADS["cfg2"]
    assert pose.dtype == hole.dtype == np.float32 and pose.shape == (3,) and hole.shape == (wl["size"], wl["size"])

    # the inputs bench.py generates for the whole run; scans [0, PRIME_SCANS + W + K) have been applied when the timed steps end
    n_total = bench.PRIME_SCANS + W + K + min(K, 200) + W + K
    rp, offs, n_cand = bench.build_workload(wl, n_total, seed)
    T = bench.pow2_threads(n_cand, os.cpu_count() or 1)
    o = orc.Processor(wl["phys"], wl["size"], rp.odometry[0], bench.SIGMA_XY, bench.SIGMA_THETA, n_cand // T, T)
    w = orc.Worker(T)
    for k in range(bench.PRIME_SCANS + W + K):
        o.update(rp.points[k], rp.odometry[k], offs[k], worker=w)
    w.close()
    assert np.array_equal(pose, o.pose)
    assert np.array_equal(hole.reshape(-1), np.array(o.map.pixels, dtype=np.float32))
