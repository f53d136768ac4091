"""Step time of the cfg5 session batch (1024 sessions x 360 points x 1000 candidates, 1600^2 HoleMap, production mode, one
shared device-resident scan log) with an ObstacleMap per session, by obstacle_map_size (0 = none).

All batches live in one process and are timed in turn, alternating over the rounds: per batch and round, W replay steps of
warm-up, then K steps (one cs_batch_replay each) timed by the host clock and ended by cs_batch_sync.  Prints one JSON line per
measurement and a summary line with the GPU's name and power limit; --out also writes them to a file."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import slam.net_b200 as sn  # noqa: E402
from slam.net_b200 import synth  # noqa: E402
from bench import WORKLOADS, cfg5_session_params  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as e:  # the numbers are still printed, flagged as unlabelled
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="0,64,400,1600")
    ap.add_argument("--sessions", type=int, default=WORKLOADS["cfg5"]["sessions"])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0x5EED0000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if sn.lib().cs_device_count() <= 0:
        raise SystemExit("no CUDA device: this probe measures the GPU and has nothing to report without one")
    sizes = [int(s) for s in args.sizes.split(",")]
    wl = WORKLOADS["cfg5"]
    P, K, W, n = wl["points"], args.steps, args.warmup, args.sessions
    n_log = args.rounds * (W + K)
    rp = synth.make_replay(n_log, P, wl["phys"], seed=args.seed)
    log = sn.ScanLog(n_log, P, n_offsets=0)
    for k in range(n_log):
        log.set(k, rp.points[k], rp.odometry[k])
    log.upload()
    prm = [cfg5_session_params(s, args.seed) for s in range(n)]
    batches = {}
    for size in sizes:
        b = sn.Batch(n, wl["phys"], wl["size"], rp.odometry[0], np.array([q[0] for q in prm], dtype=np.float32),
                     np.array([q[1] for q in prm], dtype=np.float32), wl["iters"], wl["threads"], max_points=P,
                     seeds=[q[4] for q in prm], obstacle_map_size=size)
        for j, q in enumerate(prm):
            b.set_params(j, q[2], q[3])
        if size:
            for j in range(n):
                b.set_obstacle_params(j, -5, (1, 3, 10, 127)[j % 4])
        batches[size] = b
    name, power = gpu_info()
    lines = []
    times = {s: [] for s in sizes}
    for r in range(args.rounds):
        first = r * (W + K)
        for size in sizes:
            b = batches[size]
            b.replay(log, first, W, want_results=False)
            b.sync()
            t0 = time.perf_counter()
            for i in range(K):
                b.replay(log, first + W + i, 1, want_results=False)
            b.sync()
            ms = (time.perf_counter() - t0) * 1e3 / K
            times[size].append(ms)
            line = {"round": r, "obstacle_map_size": size, "sessions": n, "steps": K, "ms_per_step": round(ms, 4)}
            if size:
                line["obstacle_cells_touched_per_session_step"] = round(float(b.obstacle_visits().mean()) / ((r + 1) * (W + K)), 1)
            lines.append(line)
            print(json.dumps(line), flush=True)
    base = float(np.mean(times[sizes[0]])) if sizes[0] == 0 else None
    summary = {"gpu": name, "power_limit": power, "workload": "cfg5 geometry, production mode, shared device-resident log",
               "sessions": n, "points": P, "candidates": wl["iters"] * wl["threads"] + 1, "hole_map": wl["size"],
               "timing": "host clock around %d cs_batch_replay steps after %d warm-up steps, ended by cs_batch_sync" % (K, W),
               "ms_per_step": {str(s): [round(t, 4) for t in times[s]] for s in sizes}}
    if base:
        summary["added_percent"] = {str(s): round(100.0 * (float(np.mean(times[s])) / base - 1.0), 2) for s in sizes if s}
    # bytes of no-hit bitmap per step the sweep reads for all sessions (one 4-byte word per 8x4 cells), for scale
    summary["sweep_bitmap_mb_per_step"] = {str(s): round(n * ((s + 7) // 8) * ((s + 3) // 4) * 4 / 1e6, 1) for s in sizes if s}
    print(json.dumps(summary), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for line in lines + [summary]:
                f.write(json.dumps(line) + "\n")
    for b in batches.values():
        b.close()
    log.close()


if __name__ == "__main__":
    main()
