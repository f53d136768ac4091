"""cs_relocalize_sequence and cs_relocalize_sequence_bounded: what scoring a pose with K scans costs, and what it buys.

For each workload of tools/relocalize_bench.py (cfg1, cfg2): the HoleMap after the same synthetic drive, then the
whole-room lattice (window 2, k 8) scored with the last K in {1, 4, 8} scans of the drive and their odometry, through both
sequence calls, alternating, --calls times each after one warm-up; at K = 1 the single-scan calls (cs_relocalize,
cs_relocalize_bounded) alternate with them on the same handle.  Every call ends in a stream synchronise, so the host
clock around it is the call's time; a row reports the median.  The hits of the exhaustive and bounded calls must be
identical.  The exhaustive rows report lookups/s as (points of the K scans) * poses / time.  Then the 2 cm x 0.5 degree
cfg2 room lattice through the bounded sequence call, and the aliasing corridor of tests/test_gpu_relocalize_sequence.py:
the position error of the best single-scan hit and of the best sequence hit.  Prints the card's name and power limit and
one JSON line per measurement; --out writes them all to one JSON file (default profiles/relocalize_sequence_bench.json)."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import slam.net_b200 as sn  # noqa: E402
from slam.net_b200 import synth  # noqa: E402
from relocalize_bench import WORKLOADS, gpu_info, room_lattice  # noqa: E402


def _key(hits):
    return [(h.distance, h.index, h.pose.tobytes()) for h in hits]


def _median_time(fn, calls, out):
    ts = []
    for _ in range(calls):
        t0 = time.perf_counter()
        out.append(fn())
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts


def measure(name, wl, calls, drive_scans, fine):
    rp = synth.make_replay(drive_scans + 1, wl["points"], wl["phys"])
    p = sn.Processor(wl["phys"], wl["size"], rp.odometry[0], 0.1, 0.17, wl["iters"], wl["threads"], max_points=wl["points"], seed=5)
    for k in range(drive_scans):
        p.update(rp.points[k], rp.odometry[k])
    p.sync()
    origin, step, count = room_lattice(wl)
    poses = count[0] * count[1] * count[2]
    rows = []
    lattices = [("room", origin, step, count)]
    if fine:
        lo, hi = 0.125 * wl["phys"], 0.875 * wl["phys"]
        n = int(round((hi - lo) / 0.02)) + 1
        lattices.append(("fine", [lo, lo, -np.pi], [0.02, 0.02, float(np.float32(2 * np.pi / 720))], [n, n, 720]))
    for K in (1, 4, 8):
        idx = list(range(drive_scans - K + 1, drive_scans + 1))
        scans, odo = [rp.points[i] for i in idx], rp.odometry[idx]
        n_points = int(sum(len(s) for s in scans))
        for lname, lo_, st_, co_ in lattices:
            row = {"workload": name, "lattice_name": lname, "K": K, "points": n_points,
                   "map": "%d^2 cells over %.0f m" % (wl["size"], wl["phys"]),
                   "lattice": {"origin": [float(v) for v in lo_], "step": [float(v) for v in st_], "count": co_,
                               "poses": co_[0] * co_[1] * co_[2], "window": 2, "k": 8}}
            fns = {"sequence_bounded": lambda: p.relocalize_sequence_bounded(scans, odo, lo_, st_, co_, window=2, k=8)}
            if lname == "room":
                fns["sequence"] = lambda: p.relocalize_sequence(scans, odo, lo_, st_, co_, window=2, k=8)
                if K == 1:
                    fns["single"] = lambda: p.relocalize(scans[0], lo_, st_, co_, window=2, k=8)
                    fns["single_bounded"] = lambda: p.relocalize_bounded(scans[0], lo_, st_, co_, window=2, k=8)
            try:
                out = {f: [fn()] for f, fn in fns.items()}  # warm-ups (allocate the scratch)
            except sn.CoreSlamError as e:  # e.g. CS_ERR_CAPACITY: more survivors than the call's budget
                row["error"] = str(e)
                rows.append(row)
                continue
            times = {f: [] for f in fns}
            for _ in range(calls):  # alternate the calls
                for f, fn in fns.items():
                    times[f].append(_median_time(fn, 1, out[f])[1][0])
            keys = {f: _key(v[-1][0]) for f, v in out.items()}
            assert len(set(map(str, keys.values()))) == 1, (name, lname, K)
            for f in fns:
                row[f + "_seconds_median"] = float(np.median(times[f]))
                row[f + "_seconds"] = times[f]
            stats = out["sequence_bounded"][-1][1]
            row["evaluated_fraction"] = stats["evaluated"] / stats["poses"]
            row["stats"] = stats
            if "sequence" in fns:
                row["sequence_lookups_per_second"] = n_points * poses / row["sequence_seconds_median"]
            best = out["sequence_bounded"][-1][0]
            row["best_hit"] = {"pose": [float(v) for v in best[0].pose], "distance": best[0].distance} if best else None
            row["truth_last_scan"] = [float(v) for v in rp.truth[drive_scans]]
            row["hits_identical"] = True
            rows.append(row)
    p.close()
    return rows


def aliasing():
    from test_gpu_relocalize_sequence import NicheCorridor, corridor_case
    room, map_truth, map_scans, truth, scans, odo, lattice = corridor_case()
    p = sn.Processor(20.0, 400, [0, 0, 0], 0.1, 0.17, 8, 1, max_points=512)
    for t, pts in zip(map_truth, map_scans):
        p.integrate(pts, t.astype(np.float32))
    single, _ = p.relocalize(scans[-1], *lattice, window=10, k=8)
    seq, _ = p.relocalize_sequence(scans, odo, *lattice, window=10, k=8)
    p.close()
    err = lambda h: float(np.hypot(h.pose[0] - truth[-1][0], h.pose[1] - truth[-1][1]))
    return {"workload": "aliasing-corridor", "K": len(scans), "niche_period_m": NicheCorridor.PERIOD,
            "lidar_range_m": NicheCorridor.RANGE, "lattice": {"origin": [float(v) for v in lattice[0]],
                                                             "step": [float(v) for v in lattice[1]], "count": lattice[2]},
            "truth": [float(v) for v in truth[-1]],
            "single_scan_best": {"pose": [float(v) for v in single[0].pose], "distance": single[0].distance,
                                 "position_error_m": err(single[0])},
            "sequence_best": {"pose": [float(v) for v in seq[0].pose], "distance": seq[0].distance,
                              "position_error_m": err(seq[0])}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg1,cfg2")
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--drive", type=int, default=60, help="scans of the synthetic drive that builds the map")
    ap.add_argument("--no-fine", action="store_true", help="skip the 2 cm x 0.5 degree cfg2 lattice")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "relocalize_sequence_bench.json"))
    args = ap.parse_args()
    name, power = gpu_info()
    print("gpu: %s, power limit %s" % (name, power), flush=True)
    rows = []
    for w in args.workloads.split(","):
        for row in measure(w, WORKLOADS[w], args.calls, args.drive, fine=(w == "cfg2" and not args.no_fine)):
            row.update(gpu=name, power_limit=power)
            print(json.dumps(row), flush=True)
            rows.append(row)
    row = aliasing()
    row.update(gpu=name, power_limit=power)
    print(json.dumps(row), flush=True)
    rows.append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"gpu": name, "power_limit": power, "results": rows}, f, indent=1)


if __name__ == "__main__":
    main()
