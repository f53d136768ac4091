"""Throughput of cs_relocalize (whole-room pose lattices) against today's route (cs_search with absolute candidates).

For each workload: build the HoleMap with a synthetic drive through the room (production-mode Updates), then
  * one warm-up call, then --calls timed calls of cs_relocalize (window 2, k 8) over the whole-room lattice; each call
    ends in a stream synchronise, so the host clock around it is the call's time (upload of the scan, the lattice,
    select and merge kernels, the copy of the hits);
  * the first 2^20 poses of the same lattice through cs_search, T*I absolute candidates per call (the handle's T*I);
  * cs_gather_peak over a table of the map's size (random 2-byte loads, L2-resident), the ceiling for scattered lookups.
The map stays in L2 between calls (no flush), as it does between the Updates of a drive.  Prints the card's name and power
limit and one JSON line per workload; --out writes them all to one JSON file (default profiles/relocalize_bench.json)."""
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

# (hole map size, physical size, points per scan, candidates T x I of today's route, lattice step x, y (m), theta (deg))
WORKLOADS = {
    "cfg1": dict(size=1600, phys=40.0, points=360, threads=4, iters=1000, step=(0.10, 0.10, 2.0)),
    "cfg2": dict(size=2048, phys=40.0, points=1024, threads=4, iters=1024, step=(0.05, 0.05, 1.0)),
}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as e:  # the numbers are still printed, flagged as unlabelled
        return "unknown (%s)" % e, "unknown"


def room_lattice(wl):
    """The room of synth.Room (1/8 .. 7/8 of the map) at the workload's steps, headings over [-pi, pi)."""
    lo, hi = 0.125 * wl["phys"], 0.875 * wl["phys"]
    sx, sy, sdeg = wl["step"]
    n_theta = int(round(360.0 / sdeg))
    count = [int(round((hi - lo) / sx)) + 1, int(round((hi - lo) / sy)) + 1, n_theta]
    return [lo, lo, -np.pi], [sx, sy, float(np.float32(2 * np.pi / n_theta))], count


def measure(name, wl, calls, drive_scans, legacy_poses):
    rp = synth.make_replay(drive_scans + 1, wl["points"], wl["phys"])
    p = sn.Processor(wl["phys"], wl["size"], rp.odometry[0], 0.1, 0.17, wl["iters"], wl["threads"], max_points=wl["points"], seed=5)
    for k in range(drive_scans):
        r = p.update(rp.points[k], rp.odometry[k])
    p.sync()
    pts = rp.points[drive_scans]
    origin, step, count = room_lattice(wl)
    poses = count[0] * count[1] * count[2]

    p.relocalize(pts, origin, step, count, window=2, k=8)  # warm-up (allocates the volume)
    times = []
    for _ in range(calls):
        t0 = time.perf_counter()
        hits, _ = p.relocalize(pts, origin, step, count, window=2, k=8)
        times.append(time.perf_counter() - t0)
    sec = float(np.median(times))

    # today's route: the first `legacy_poses` lattice poses as absolute candidates, T*I per cs_search call
    c0, c1 = count[0], count[1]
    idx = np.arange(legacy_poses)
    xs = np.float32(origin[0]) + (idx % c0).astype(np.float32) * np.float32(step[0])
    ys = np.float32(origin[1]) + (idx // c0 % c1).astype(np.float32) * np.float32(step[1])
    ts = np.float32(origin[2]) + (idx // (c0 * c1)).astype(np.float32) * np.float32(step[2])
    cand = np.stack([xs, ys, ts], axis=1)
    n = p.n_cand
    p.search(pts, cand[0], cand[:n], want_distances=False)  # warm-up
    t0 = time.perf_counter()
    for b in range(0, legacy_poses, n):
        blk = cand[b:b + n]
        if blk.shape[0] < n:
            break
        p.search(pts, blk[0], blk, want_distances=False)
    legacy_sec = time.perf_counter() - t0
    legacy_done = legacy_poses // n * n
    peak = sn.gather_peak(wl["size"] * wl["size"])
    p.close()
    lookups = poses * wl["points"]
    return {
        "workload": name, "map": "%d^2 cells over %.0f m" % (wl["size"], wl["phys"]), "points": wl["points"],
        "lattice": {"origin": [float(v) for v in origin], "step": [float(v) for v in step], "count": count, "poses": poses,
                    "window": 2, "k": 8},
        "seconds_per_call_median": sec, "seconds_per_call": times,
        "poses_per_s": poses / sec, "lookups_per_s": lookups / sec,
        "drive_pose_last_scan": [float(v) for v in r.pose],
        "best_hit": {"pose": [float(v) for v in hits[0].pose], "distance": hits[0].distance} if hits else None,
        "cs_search_route": {"poses": legacy_done, "candidates_per_call": n, "seconds": legacy_sec,
                            "poses_per_s": legacy_done / legacy_sec},
        "speedup_per_pose": (poses / sec) / (legacy_done / legacy_sec),
        "cs_gather_peak_lookups_per_s": peak,
        "map_residency": "L2-resident across calls (no flush), as between the Updates of a drive",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg1,cfg2")
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--drive", type=int, default=60, help="scans of the synthetic drive that builds the map")
    ap.add_argument("--legacy-poses", type=int, default=1 << 20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "relocalize_bench.json"))
    args = ap.parse_args()
    name, power = gpu_info()
    print("gpu: %s, power limit %s" % (name, power), flush=True)
    rows = []
    for w in args.workloads.split(","):
        row = measure(w, WORKLOADS[w], args.calls, args.drive, args.legacy_poses)
        row.update(gpu=name, power_limit=power)
        print(json.dumps(row), flush=True)
        rows.append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"gpu": name, "power_limit": power, "results": rows}, f, indent=1)


if __name__ == "__main__":
    main()
