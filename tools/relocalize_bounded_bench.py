"""cs_relocalize_bounded (branch and bound) against cs_relocalize (every pose) on whole-room lattices.

For each workload of tools/relocalize_bench.py (cfg1, cfg2): the HoleMap after the same synthetic drive, then the
whole-room lattice (window 2, k 8) through both calls, alternating, --calls times each after one warm-up of each.  Every
call ends in a stream synchronise, so the host clock around it is the call's time.  The hits of the two calls must be
identical.  Then one 2 cm x 0.5 degree cfg2 room lattice (about 1.6e9 poses, beyond cs_relocalize's 2^28) through the
bounded call alone.  Prints the card's name and power limit and one JSON line per measurement; --out writes them all to
one JSON file (default profiles/relocalize_bounded_bench.json)."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

import slam.net_b200 as sn  # noqa: E402
from slam.net_b200 import synth  # noqa: E402
from relocalize_bench import WORKLOADS, gpu_info, room_lattice  # noqa: E402


def _key(hits):
    return [(h.distance, h.index, h.pose.tobytes()) for h in hits]


def _timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


def measure(name, wl, calls, drive_scans, fine):
    rp = synth.make_replay(drive_scans + 1, wl["points"], wl["phys"])
    p = sn.Processor(wl["phys"], wl["size"], rp.odometry[0], 0.1, 0.17, wl["iters"], wl["threads"], max_points=wl["points"], seed=5)
    for k in range(drive_scans):
        p.update(rp.points[k], rp.odometry[k])
    p.sync()
    pts = rp.points[drive_scans]
    rows = []
    origin, step, count = room_lattice(wl)
    poses = count[0] * count[1] * count[2]
    ex, _ = p.relocalize(pts, origin, step, count, window=2, k=8)  # warm-ups (allocate the scratch)
    bd, stats = p.relocalize_bounded(pts, origin, step, count, window=2, k=8)
    assert _key(bd) == _key(ex), name
    t_ex, t_bd = [], []
    for _ in range(calls):
        (ex, _), t = _timed(lambda: p.relocalize(pts, origin, step, count, window=2, k=8))
        t_ex.append(t)
        (bd, stats), t = _timed(lambda: p.relocalize_bounded(pts, origin, step, count, window=2, k=8))
        t_bd.append(t)
        assert _key(bd) == _key(ex), name
    rows.append({
        "workload": name, "map": "%d^2 cells over %.0f m" % (wl["size"], wl["phys"]), "points": wl["points"],
        "lattice": {"origin": [float(v) for v in origin], "step": [float(v) for v in step], "count": count, "poses": poses,
                    "window": 2, "k": 8},
        "exhaustive_seconds_median": float(np.median(t_ex)), "exhaustive_seconds": t_ex,
        "bounded_seconds_median": float(np.median(t_bd)), "bounded_seconds": t_bd,
        "speedup": float(np.median(t_ex) / np.median(t_bd)),
        "evaluated_fraction": stats["evaluated"] / stats["poses"], "stats": stats,
        "hits_identical": True,
        "best_hit": {"pose": [float(v) for v in bd[0].pose], "distance": bd[0].distance} if bd else None,
        "drive_pose_last_scan": [float(v) for v in rp.odometry[drive_scans]],
    })
    if fine:
        # 2 cm x 0.5 degree over the same room
        lo, hi = 0.125 * wl["phys"], 0.875 * wl["phys"]
        n_theta = 720
        count = [int(round((hi - lo) / 0.02)) + 1, int(round((hi - lo) / 0.02)) + 1, n_theta]
        step = [0.02, 0.02, float(np.float32(2 * np.pi / n_theta))]
        origin = [lo, lo, -np.pi]
        t_f = []
        try:
            p.relocalize_bounded(pts, origin, step, count, window=2, k=8)  # warm-up
            for _ in range(calls):
                (bd, stats), t = _timed(lambda: p.relocalize_bounded(pts, origin, step, count, window=2, k=8))
                t_f.append(t)
        except sn.CoreSlamError as e:  # e.g. CS_ERR_CAPACITY: more survivors than the call's budget
            rows.append({"workload": name + "-fine", "lattice": {"count": count, "step": step}, "error": str(e)})
            p.close()
            return rows
        rows.append({
            "workload": name + "-fine", "map": "%d^2 cells over %.0f m" % (wl["size"], wl["phys"]), "points": wl["points"],
            "lattice": {"origin": [float(v) for v in origin], "step": step, "count": count,
                        "poses": count[0] * count[1] * count[2], "window": 2, "k": 8},
            "bounded_seconds_median": float(np.median(t_f)), "bounded_seconds": t_f,
            "evaluated_fraction": stats["evaluated"] / stats["poses"], "stats": stats,
            "best_hit": {"pose": [float(v) for v in bd[0].pose], "distance": bd[0].distance} if bd else None,
            "drive_pose_last_scan": [float(v) for v in rp.odometry[drive_scans]],
        })
    p.close()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg1,cfg2")
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--drive", type=int, default=60, help="scans of the synthetic drive that builds the map")
    ap.add_argument("--no-fine", action="store_true", help="skip the 2 cm x 0.5 degree cfg2 lattice")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "relocalize_bounded_bench.json"))
    args = ap.parse_args()
    name, power = gpu_info()
    print("gpu: %s, power limit %s" % (name, power), flush=True)
    rows = []
    for w in args.workloads.split(","):
        for row in measure(w, WORKLOADS[w], args.calls, args.drive, fine=(w == "cfg2" and not args.no_fine)):
            row.update(gpu=name, power_limit=power)
            print(json.dumps(row), flush=True)
            rows.append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"gpu": name, "power_limit": power, "results": rows}, f, indent=1)


if __name__ == "__main__":
    main()
