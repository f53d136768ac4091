#!/usr/bin/env python
"""bench.py — CoreSLAM scan-to-map hot path on B200: scan-point map lookups/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg1|cfg3|cfg4|cfg5]
                    [--dump-outputs DIR]

A *step* is one CoreSLAMProcessor.Update of the replay: Monte-Carlo pose search over C+1 candidate
poses x P scan points (the lookups) followed by the HoleMap integration of the same scan.  The N=1
workload is BASELINE.json configs[1]: synthetic replay, 4096 candidates x 1024-point scans, HoleMap
2048x2048 over 40 m, verification mode (candidate tables uploaded, results bit-exact vs the oracle).

  value     lookups/s with the scan log already resident in HBM; per-step CUDA-event time on the
            launching stream, L2 flushed (256 MB write) before every timed step, max over ranks.
  e2e       the same metric through the C-ABI call cs_update() with HOST buffers: pinned staging,
            H2D of points + candidate table and the pose read back inside the timed region (wall clock).
  roofline  the search kernel (dominant): algorithmic bytes per launch / its mean CUDA-event duration,
            against MEASURED_PEAKS.json hbm_gbs, plus the measured random-gather ceiling.
  cpu_baseline / --impl reference: the CPU oracle port of the reference (oracle/, multithreaded like
            BaseSLAM/ParallelWorker) on the box's host cores.  The reference itself is C#/.NET and cannot
            run here, so kind = "port".

N > 1 (torchrun, one rank per GPU): independent replays (sessions) sharded one per GPU, no data-path
collective, weak scaling; value = lookups of all ranks / max-over-ranks time.

--dump-outputs DIR (cfg1 / cfg2 line): after the K timed steps, rank 0 writes what a caller of the timed Update holds
after the last of them, as float32: DIR/pose.npy (x, y, theta) and DIR/hole_map.npy (the HoleMap, size x size; the u16
cells are exact in float32).  The inputs are generated from --seed, so two builds run with the same arguments can be
compared array for array.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (points, threads, iters, map size, physical size)
    "cfg1": dict(points=360, threads=4, iters=1000, size=1600, phys=40.0,
                 desc="CoreSLAM 360-point scans, 4x1000 search iterations, HoleMap 1600x1600 @2.5 cm"),
    "cfg2": dict(points=1024, threads=4, iters=1024, size=2048, phys=40.0,
                 desc="CoreSLAM synthetic replay, 4096 candidates x 1024-point scans, HoleMap 2048x2048, verification mode"),
    "cfg3": dict(points=8192, threads=1, iters=1, size=4096, phys=40.96,
                 desc="HoleMap integration stress: 8192-ray scans at 1 cm into a 4096x4096 map (UpdateHoleMap only, no search), "
                      "map checksum bit-exact vs the oracle"),
    "cfg4": dict(points=1024, threads=64, iters=1024, size=8192, phys=81.92,
                 desc="Large-map HBM regime: HoleMap 8192x8192 @1 cm (128 MB), 65536 candidates x 1024-point scans, candidates split "
                      "across the GPUs with one 8-byte arg-min exchange (NCCL MIN all-reduce) per scan"),
    "cfg5": dict(points=360, threads=1, iters=1000, size=1600, phys=40.0, sessions=1024,
                 desc="Batched independent sessions: 1024 CoreSLAM replays (parameter sweep over sigma_xy, sigma_theta, HoleWidth, "
                      "Quality, seed; cfg1 geometry) sharded over the GPUs, no collective"),
}
PRIME_SCANS = 5  # PositionSearchBeginning: the first 5 scans only build the map (CoreSLAMProcessor.cs:92, :726)
SIGMA_XY, SIGMA_THETA = 0.1, 0.17453292  # 0.1 m, 10 degrees (Simulation/MainWindow.xaml.cs:69)


ALL_CORES = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None  # before any per-rank pinning


class all_cores:
    """Context: lift this rank's core pinning (parallel.pin_rank_to_cores) while the multi-threaded CPU oracle checks a result."""

    def __enter__(self):
        self.saved = os.sched_getaffinity(0) if ALL_CORES is not None else None
        if ALL_CORES is not None:
            os.sched_setaffinity(0, ALL_CORES)

    def __exit__(self, *exc):
        if self.saved is not None:
            os.sched_setaffinity(0, self.saved)
        return False


def cpu_min_seconds(default=10.0):
    """Shortest CPU sample of the reference arm / cpu_baseline (CS_BENCH_CPU_MIN_S shortens it for the CPU test-suite)."""
    try:
        return float(os.environ.get("CS_BENCH_CPU_MIN_S", default))
    except ValueError:
        return default


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int, period: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    self.nv, "nvmlDeviceGetCurrentClocksEventReasons") else self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def build_workload(wl, n_scans, seed):
    from slam.net_b200 import synth
    rp = synth.make_replay(n_scans, wl["points"], wl["phys"], seed=seed)
    n_cand = wl["threads"] * wl["iters"]
    offs = [synth.candidate_offsets(seed, k, n_cand, SIGMA_XY, SIGMA_THETA) for k in range(n_scans)]
    return rp, offs, n_cand


def pow2_threads(n_cand, cores):
    t = 1
    while t * 2 <= cores and n_cand % (t * 2) == 0:
        t *= 2
    return t


def run_cpu(wl, rp, offs, n_cand, first, count, budget_s=25.0, min_s=10.0, threads=None):
    """The oracle port (reference algorithm, ParallelWorker-style threads) over scans [first, first+count).
    The first pass is the parity sample (same scans as the GPU arm); when it ends before `min_s` seconds the
    same scans are replayed back and forth (count-1 .. 0 .. count-1, so odometry stays continuous) until the
    sample holds at least `min_s` seconds of CPU work.  Returns (lookups/s, scans timed, threads, seconds,
    pose after the first pass, whether the first pass was complete)."""
    from oracle import oracle as orc
    cores = os.cpu_count() or 1
    T = pow2_threads(n_cand, cores if threads is None else min(threads, cores))
    o = orc.Processor(wl["phys"], wl["size"], rp.odometry[0], SIGMA_XY, SIGMA_THETA, n_cand // T, T)
    w = orc.Worker(T)
    for k in range(first):  # bring the map to the same state as the GPU arm (untimed)
        o.update(rp.points[k], rp.odometry[k], offs[k], worker=w)
    lookups, done = 0, 0
    pose, complete = None, False
    order = list(range(first, first + count))
    t0 = time.perf_counter()
    while True:
        for k in order:
            o.update(rp.points[k], rp.odometry[k], offs[k], worker=w)
            lookups += (n_cand + 1) * rp.points[k].shape[0]
            done += 1
            if time.perf_counter() - t0 > budget_s:
                break
        else:
            if pose is None:
                pose, complete = o.pose.copy(), True
            if time.perf_counter() - t0 < min_s and count > 1:
                order = order[::-1]
                continue
        break
    dt = time.perf_counter() - t0
    if pose is None:
        pose = o.pose.copy()
    w.close()
    return lookups / dt, done, T, dt, pose, complete


def kernel_src_sha():
    """Hash of the kernel sources (slam.net_b200/csrc), as tools/ncu_summary.py stamps its captures with."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "slam.net_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(f.encode())
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def latest_capture(kernel):
    """The newest committed ncu capture of `kernel` (profiles/*_traffic.json, written by tools/ncu_summary.py) -> (entry,
    file name, stale).  A capture taken from other kernel sources than the ones in the tree is reported as stale and its
    numbers are NOT used (traffic = null): ncu counters describe the code they were measured on."""
    import glob
    sha = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")), reverse=True):
        try:
            d = json.load(open(path))
            k = d[kernel]
        except Exception:
            continue
        if sha is None:
            sha = kernel_src_sha()
        return k, os.path.basename(path), d.get("kernel_src_sha") != sha
    return None, None, True


def latest_traffic(kernel):
    """DRAM bytes per launch of `kernel` from its newest capture, or (None, why)."""
    k, src, stale = latest_capture(kernel)
    if k is None:
        return None, None
    if stale:
        return None, "%s is stale (kernel sources changed since the capture)" % src
    return float((k.get("dram_bytes_read") or 0.0) + (k.get("dram_bytes_write") or 0.0)), src


def limiter_of(kernel, launch_ms, sm_count=148, clock_hz=1.965e9):
    """What bounds `kernel` according to its newest capture: its stall mix, issue-slot use, and the fraction of the launch an
    issue-bound kernel of the same instruction count would need (warp instructions / (SMs x 4 schedulers x clock))."""
    k, src, stale = latest_capture(kernel)
    if k is None:
        return None
    out = {"source": src, "stale": bool(stale)}
    if stale:
        return out
    wi = k.get("warp_instructions")
    out.update({"stall_mix": k.get("stall_mix"), "issue_slots_busy_pct": k.get("issue_slots_busy_pct"), "ipc_active": k.get("ipc_active"),
                "achieved_occupancy_pct": k.get("achieved_occupancy_pct"), "warp_instructions_per_launch": wi,
                "capture_duration_us": k.get("duration_us")})
    if wi and launch_ms:
        floor_ms = wi / (sm_count * 4 * clock_hz) * 1e3
        out["issue_floor_ms"] = floor_ms
        out["frac_of_issue_ceiling"] = floor_ms / launch_ms
    return out


def cfg5_session_params(s, seed):
    """Parameter grid of session s (SURVEY 8d): sigma_xy, sigma_theta, Quality, HoleWidth, seed."""
    return (0.05 + 0.025 * (s % 5), 0.0873 + 0.0436 * ((s // 5) % 4), 30 + 20 * ((s // 20) % 6), 0.4 + 0.2 * ((s // 120) % 4), seed + s)


def measure_cfg5(args, rank, world, local, K, W, n_sessions=None, sub_batches=0, e2e=True, parity_sessions=3):
    """configs[4]: n_sessions independent CoreSLAM replays (cfg1 geometry, production mode) sharded session i -> rank i mod world,
    strong scaling, no collective.  Returns (on every rank) the reduced numbers; `parity` = pose and map checksum of a sample
    of sessions after the timed steps equal the CPU oracle's (fed the host twin of each session's Philox stream)."""
    import torch
    import torch.distributed as dist
    import slam.net_b200 as sn
    from slam.net_b200 import _native as N
    from slam.net_b200 import parallel as par
    from slam.net_b200 import synth

    wl = WORKLOADS["cfg5"]
    P = wl["points"]
    n_cand = wl["threads"] * wl["iters"]
    n_sessions = n_sessions or wl["sessions"]
    Ke = min(K, 20) if e2e else 0
    n_total = PRIME_SCANS + W + K + (2 * Ke + 2 if e2e else 0)
    rp = synth.make_replay(n_total, P, wl["phys"], seed=args.seed)  # same scans on every rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    mine = par.session_shard(n_sessions, world, rank)
    n_sub = max(1, min(sub_batches if sub_batches > 0 else 1, max(len(mine), 1)))
    subs = [mine[i::n_sub] for i in range(n_sub)]
    stream = torch.cuda.Stream()
    streams = [stream] + [torch.cuda.Stream() for _ in range(n_sub - 1)]
    sampler = ClockSampler(local)
    out = {}
    with torch.cuda.stream(stream):
        batches = []
        for part, st in zip(subs, streams):
            prm = [cfg5_session_params(s, args.seed) for s in part]
            b = sn.Batch(len(part), wl["phys"], wl["size"], rp.odometry[0], np.array([q[0] for q in prm], dtype=np.float32),
                         np.array([q[1] for q in prm], dtype=np.float32), wl["iters"], wl["threads"], device=local,
                         max_points=P, seeds=[q[4] for q in prm], stream=st.cuda_stream)
            for j, q in enumerate(prm):
                b.set_params(j, q[2], q[3])
            batches.append(b)
        log = sn.ScanLog(n_total, P, n_offsets=0, device=local)
        for k in range(n_total):
            log.set(k, rp.points[k], rp.odometry[k])
        log.upload()
        torch.cuda.synchronize()  # the log is read from every stream
        for b in batches:
            b.replay(log, 0, PRIME_SCANS + W, want_results=False)
        launches0 = sum(b.launch_count() for b in batches)
        barrier()
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        done = [torch.cuda.Event() for _ in streams[1:]]
        e0.record(stream)
        for st in streams[1:]:
            st.wait_event(e0)
        if n_sub == 1:
            batches[0].replay(log, PRIME_SCANS + W, K, want_results=False)
        else:  # steps are queued round-robin so that no stream runs ahead of another by more than one step
            for i in range(K):
                for b in batches:
                    b.replay(log, PRIME_SCANS + W + i, 1, want_results=False)
        for st, ev in zip(streams[1:], done):
            ev.record(st)
            stream.wait_event(ev)
        e1.record(stream)
        barrier()
        clocks = sampler.stop()
        dev_ms = e0.elapsed_time(e1)
        launches = sum(b.launch_count() for b in batches) - launches0
        poses = np.concatenate([b.poses() for b in batches], axis=0) if mine else np.zeros((0, 3), dtype=np.float32)
        sums = np.concatenate([b.map_checksums() for b in batches], axis=0) if mine else np.zeros(0, dtype=np.uint64)
        order = [s for part in subs for s in part]

        # ---- parity: a sample of sessions against the CPU oracle (the oracle only checks; it is not timed here)
        parity_ok, checked = True, []
        if parity_sessions > 0:
            from oracle import oracle as orc
            sample = sorted(set([0, n_sessions // 2, n_sessions - 1][:parity_sessions]))
            for s in sample:
                if s not in order:
                    continue
                sxy, sth, q, hw, seed = cfg5_session_params(s, args.seed)
                o = orc.Processor(wl["phys"], wl["size"], rp.odometry[0], np.float32(sxy), np.float32(sth), wl["iters"], wl["threads"])
                o.quality, o.hole_width = q, np.float32(hw)
                wk = orc.Worker(1)
                for k in range(PRIME_SCANS + W + K):
                    off = sn.philox_offsets(seed, k, n_cand, np.float32(sxy), np.float32(sth)) if k >= PRIME_SCANS else None
                    o.update(rp.points[k], rp.odometry[k], off, worker=wk)
                wk.close()
                j = order.index(s)
                ok = bool(np.array_equal(poses[j], o.pose) and int(sums[j]) == int(sn.host_map_checksum(np.array(o.map.pixels), wl["size"])))
                parity_ok = parity_ok and ok
                checked.append(s)

        e2e_wall, e2e_blocking_wall = 0.0, 0.0
        if e2e and mine:
            # the same step through the C ABI with HOST buffers: every session's scan goes host -> device inside the timed
            # region and every session's result record comes back
            L = sn.lib()
            fp, ip = C.POINTER(C.c_float), C.POINTER(C.c_int32)
            packed = []
            for b, part in zip(batches, subs):
                per_step = []
                for i in range(2 * Ke + 2):
                    k = PRIME_SCANS + W + K + i
                    pts = np.zeros((len(part), P, 2), dtype=np.float32)
                    pts[:, :rp.points[k].shape[0]] = rp.points[k]
                    npts = np.full(len(part), rp.points[k].shape[0], dtype=np.int32)
                    odo = np.ascontiguousarray(np.tile(rp.odometry[k], (len(part), 1)), dtype=np.float32)
                    per_step.append((pts, npts, odo))
                packed.append((per_step, (N.Result * len(part))()))
            barrier()
            t0e = time.perf_counter()
            for i in range(Ke):
                for b, (per_step, res) in zip(batches, packed):
                    pts, npts, odo = per_step[i]
                    st = L.cs_batch_update(b._h, pts.ctypes.data_as(fp), npts.ctypes.data_as(ip), odo.ctypes.data_as(fp), None, res)
                    if st != 0:
                        raise RuntimeError("cs_batch_update failed: %d" % st)
            torch.cuda.synchronize()
            e2e_blocking_wall = time.perf_counter() - t0e  # this rank's own end (max over ranks below): the closing barrier is not part of the steps
            barrier()

            def submit(i):
                for b, (per_step, res) in zip(batches, packed):
                    pts, npts, odo = per_step[i]
                    st = L.cs_batch_submit(b._h, pts.ctypes.data_as(fp), npts.ctypes.data_as(ip), odo.ctypes.data_as(fp), None)
                    if st != 0:
                        N.check(st, batch=b._h)

            def collect():
                for b, (per_step, res) in zip(batches, packed):
                    st = L.cs_batch_collect(b._h, res)
                    if st != 0:
                        N.check(st, batch=b._h)

            submit(Ke)      # untimed: the two pipeline slots (pinned + device staging) are allocated on first use
            submit(Ke + 1)
            collect()
            collect()
            barrier()
            t0e = time.perf_counter()
            submit(Ke + 2)
            for i in range(Ke + 3, 2 * Ke + 2):
                submit(i)
                collect()
            collect()
            torch.cuda.synchronize()
            e2e_wall = time.perf_counter() - t0e  # this rank's own end (max over ranks below): the closing barrier is not part of the steps
            barrier()
        elif e2e:
            barrier(); barrier(); barrier(); barrier()
        log.close()
        for b in batches:
            b.close()
    t_all = torch.tensor([dev_ms, e2e_wall * 1e3, e2e_blocking_wall * 1e3, 0.0 if parity_ok else 1.0, float(len(checked)), float(launches)],
                         dtype=torch.float64, device="cuda")
    t_sum = t_all.clone()
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_sum, op=dist.ReduceOp.SUM)
    dev_ms_max, e2e_ms_max, e2e_blk_max, bad, _, _ = (float(x) for x in t_all.tolist())
    n_checked, launches_all = int(t_sum[4].item()), int(t_sum[5].item())
    lookups_per_step = (n_cand + 1) * P * n_sessions
    out = {"sessions": n_sessions, "sessions_this_rank": len(mine), "batches_per_rank": n_sub, "steps": K, "warmup": W,
           "ms_per_step": dev_ms_max / K, "sessions_per_s": n_sessions * K / (dev_ms_max * 1e-3),
           "lookups_per_s": lookups_per_step * K / (dev_ms_max * 1e-3), "scaling": "strong",
           "parity": {"sessions_checked": n_checked, "pose_and_map_checksum_equal_oracle": bool(bad == 0.0 and n_checked > 0),
                      "how": "sessions 0, n/2, n-1 replayed by the CPU oracle fed the host twin of their Philox streams"},
           "gpu_launches": launches_all, "clocks": clocks,
           "pose_spread_m": float(np.ptp(poses[:, 0]) + np.ptp(poses[:, 1])) if len(poses) else 0.0,
           "mode": "production (on-device Philox candidates), shared device-resident scan log",
           "l2": "per-rank working set %d maps x %.1f MB >> L2" % (len(mine), wl["size"] ** 2 * 2 / 1e6)}
    if e2e:
        out["e2e"] = {"value": lookups_per_step * Ke / (e2e_ms_max * 1e-3), "unit": "lookups/s", "ms_per_step": e2e_ms_max / Ke,
                      "sessions_per_s": n_sessions * Ke / (e2e_ms_max * 1e-3),
                      "h2d_bytes_per_step": n_sessions * (8 * P + 12 + 4), "d2h_bytes_per_step": n_sessions * 32,
                      "api": "cs_batch_submit + cs_batch_collect (C ABI, host buffers: every session's scan uploaded each step, every "
                             "result record read back; step k+1 is submitted before step k is collected), %d steps" % Ke,
                      "blocking": {"api": "cs_batch_update (blocking call), %d steps" % Ke, "ms_per_step": e2e_blk_max / Ke}}
    return out


def measure_cfg4(args, rank, world, local, K, W, oracle_check=True):
    """configs[3]: one session, 8192x8192 map (128 MB), 65536 candidates split over the ranks (flat indices
    [g*C/G, (g+1)*C/G)), replicated map, one 8-byte MIN exchange per scan; production mode.  `parity`: every rank ends with the
    same pose and map checksum, equal to an unsplit handle's on rank 0 and (oracle_check) to the CPU oracle's."""
    import torch
    import torch.distributed as dist
    import slam.net_b200 as sn
    from slam.net_b200 import parallel as par
    from slam.net_b200 import synth

    wl = WORKLOADS["cfg4"]
    P = wl["points"]
    n_cand = wl["threads"] * wl["iters"]
    n_total = PRIME_SCANS + W + K
    rp = synth.make_replay(n_total, P, wl["phys"], seed=args.seed)  # same scans on every rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stream = torch.cuda.Stream()
    sampler = ClockSampler(local)
    with torch.cuda.stream(stream):
        proc = sn.Processor(wl["phys"], wl["size"], rp.odometry[0], SIGMA_XY, SIGMA_THETA, wl["iters"], wl["threads"],
                            device=local, max_points=P, seed=args.seed, stream=stream.cuda_stream)
        if args.split == "nccl":  # search kernel -> torch.distributed all_reduce(MIN) -> set-up kernel (round 1's exchange)
            ss = par.SplitSearch(proc, rank, world, local, torch_stream=stream)
        else:                     # the exchange inside the search kernel over peer-mapped memory (cs_group_attach)
            par.attach_group(proc, rank, world)
            ss = proc
        for k in range(PRIME_SCANS + W):
            ss.update(rp.points[k], rp.odometry[k], None)
        proc.sync()
        launches0 = proc.launch_count()
        lat = np.zeros(K)
        barrier()
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t0 = time.perf_counter()
        for i in range(K):
            k = PRIME_SCANS + W + i
            ta = time.perf_counter()
            r = ss.update(rp.points[k], rp.odometry[k], None)
            lat[i] = time.perf_counter() - ta
        e1.record(stream)
        proc.sync()
        wall = time.perf_counter() - t0  # this rank's own end (max over ranks below): the closing barrier is not part of the steps
        barrier()
        clocks = sampler.stop()
        dev_ms = e0.elapsed_time(e1)
        launches = proc.launch_count() - launches0
        pose = np.array(r.pose, dtype=np.float32)
        checksum = int(proc.map_checksum())
        proc.close()
        # rank 0: the same replay on one unsplit handle (what N = 1 computes), and the CPU oracle
        ref_ok, oracle_ok = None, None
        if rank == 0:
            if world > 1:
                q = sn.Processor(wl["phys"], wl["size"], rp.odometry[0], SIGMA_XY, SIGMA_THETA, wl["iters"], wl["threads"],
                                 device=local, max_points=P, seed=args.seed, stream=stream.cuda_stream)
                for k in range(n_total):
                    rq = q.update(rp.points[k], rp.odometry[k], None)
                ref_ok = bool(np.array_equal(rq.pose, pose) and int(q.map_checksum()) == checksum)
                q.close()
            if oracle_check:
                from oracle import oracle as orc
                T = pow2_threads(n_cand, os.cpu_count() or 1)  # same flat candidate order, fewer and longer threads
                o = orc.Processor(wl["phys"], wl["size"], rp.odometry[0], SIGMA_XY, SIGMA_THETA, n_cand // T, T)
                with all_cores():
                    wk = orc.Worker(T)
                    for k in range(n_total):
                        off = sn.philox_offsets(args.seed, k, n_cand, SIGMA_XY, SIGMA_THETA) if k >= PRIME_SCANS else None
                        o.update(rp.points[k], rp.odometry[k], off, worker=wk)
                    wk.close()
                oracle_ok = bool(np.array_equal(o.pose, pose) and int(sn.host_map_checksum(np.array(o.map.pixels), wl["size"])) == checksum)
    # all ranks: same pose, same map
    sig = torch.tensor([float(pose[0]), float(pose[1]), float(pose[2]), float(checksum & 0xFFFFFF), float((checksum >> 24) & 0xFFFFFF),
                        float(checksum >> 48)], dtype=torch.float64, device="cuda")
    lo, hi = sig.clone(), sig.clone()
    t_all = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    ranks_equal = bool(torch.equal(lo, hi))
    dev_ms_max, wall_ms_max = (float(x) for x in t_all.tolist())
    lookups_per_step = (n_cand + 1) * P  # whole job: all ranks together evaluate every candidate once
    return {"candidates": n_cand + 1, "points": P, "map": "%dx%d u16 (%.0f MB, replicated)" % (wl["size"], wl["size"], wl["size"] ** 2 * 2 / 1e6),
            "steps": K, "warmup": W, "us_per_update": dev_ms_max / K * 1e3, "ms_per_step": dev_ms_max / K,
            "lookups_per_s": lookups_per_step * K / (dev_ms_max * 1e-3), "scaling": "strong",
            "e2e": {"value": lookups_per_step * K / (wall_ms_max * 1e-3), "unit": "lookups/s", "ms_per_step": wall_ms_max / K,
                    "h2d_bytes_per_step": 64 + 8 * P, "d2h_bytes_per_step": 32,
                    "api": ("cs_update_begin -> all_reduce(MIN) -> cs_update_finish" if args.split == "nccl" else
                            "cs_update on a handle attached to the group (cs_group_attach)") + " with host points (the timed loop itself)"},
            "scan_to_pose_latency_ms": {"p50": float(np.percentile(lat, 50) * 1e3), "p99": float(np.percentile(lat, 99) * 1e3)},
            "exchange": ("torch.distributed all_reduce(MIN) on the 8-byte in-session key, %d ranks" % world) if args.split == "nccl" else
                        ("inside the search kernel: every rank's publishing thread stores {key, tag} (16 B) into every rank's table "
                         "over peer-mapped memory (CUDA IPC, NVLink) and waits for the world's keys in its own; %d ranks, no "
                         "collective launch, no host step" % world),
            "nvlink_bytes_per_step": 16 * max(world - 1, 0) * world,
            "parity": {"pose_and_map_checksum_equal_on_all_ranks": ranks_equal, "equal_to_unsplit_handle_rank0": ref_ok,
                       "equal_to_cpu_oracle": oracle_ok},
            "final_pose": [float(x) for x in pose], "map_checksum": checksum, "gpu_launches": int(launches), "clocks": clocks,
            "mode": "production (on-device Philox candidates; nothing but the scan is uploaded)"}


def run_sharded(args, wl, metric, config, rank, world, local, K, W):
    """--workload cfg4 / cfg5 as the line's headline (the default cfg2 line carries both as its `sharded` block)."""
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        from slam.net_b200 import parallel as _par
        if os.environ.get("CS_BENCH_NO_PIN") != "1":
            _par.pin_rank_to_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)))  # each rank on its own cores (e2e at N > 1)
    P = wl["points"]
    if args.workload == "cfg4":
        m = measure_cfg4(args, rank, world, local, K, W)
    else:
        m = measure_cfg5(args, rank, world, local, K, W, n_sessions=args.sessions if args.sessions > 0 else None,
                         sub_batches=args.sub_batches)
    if rank == 0:
        value = m["lookups_per_s"]
        e2e = m.pop("e2e")
        line = {"metric": metric, "value": value, "unit": "lookups/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32 transform -> u16 gather -> i64 sum", "data": "synthetic",
                "config": dict(config, mode=m.pop("mode")),
                "timing": "CUDA events on the launching stream around the K steps; max over ranks",
                "candidate_poses_per_s": value / P, "clocks": m.pop("clocks"), "e2e": e2e, "gpu_launches": m.pop("gpu_launches")}
        line.update(m)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_cpu_cfg3(wl, rp, first, count, min_s=10.0):
    """The oracle's UpdateHoleMap (serial, like the reference: CoreSLAMProcessor.cs:515-533) over scans [0, first+count) at their
    odometry poses; scans [first, first+count) are timed, then integrated again back and forth until the sample holds `min_s`
    seconds.  Returns (visits, seconds, calls timed, checksum of the map after the first pass)."""
    from oracle import oracle as orc
    import slam.net_b200 as sn
    S = wl["size"]
    m = orc.HoleMap(S, wl["phys"])
    m.fill(32750)

    def one(k):
        pose = rp.odometry[k].copy()
        pose[2] = orc.normalize_angle(float(pose[2]))  # :746
        ta = time.perf_counter()
        v = orc.update_hole_map(m, rp.points[k], pose, 0.6, 50)
        return v, time.perf_counter() - ta

    visits, secs, done = 0, 0.0, 0
    for k in range(first + count):
        v, dt = one(k)
        if k >= first:
            visits, secs, done = visits + v, secs + dt, done + 1
    checksum = int(sn.host_map_checksum(np.array(m.pixels), S))
    k, step = first + count - 1, -1
    while secs < min_s and done < 100000 and count > 1:
        v, dt = one(k)
        visits, secs, done = visits + v, secs + dt, done + 1
        if not first <= k + step < first + count:
            step = -step
        k += step
    return visits, secs, done, checksum


def run_cfg3(args, wl, config, rank, world, local, K, W):
    """configs[2]: the integration half alone.  A step = UpdateHoleMap (CoreSLAMProcessor.cs:496-534) of one 8192-ray scan
    into the 4096x4096 map at the scan's odometry pose — `Update` with the search gated off (PositionSearchBeginning out of
    reach, :726-742), so the replay runs cs_setup_kernel + cs_rings_kernel only.  Metric: HoleMap cell visits/s (one visit =
    one iteration of the draw loop :404-442 = one 2-byte read + one 2-byte write)."""
    import torch
    import torch.distributed as dist
    import slam.net_b200 as sn
    from slam.net_b200 import _native as N
    from slam.net_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        from slam.net_b200 import parallel as _par
        if os.environ.get("CS_BENCH_NO_PIN") != "1":
            _par.pin_rank_to_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)))  # each rank on its own cores (e2e at N > 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    P, S = wl["points"], wl["size"]
    Kb = min(K, 100)
    n_total = W + K + Kb + W + K
    rp = synth.make_replay(n_total, P, wl["phys"], seed=args.seed + 7919 * rank)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        proc = sn.Processor(wl["phys"], S, rp.odometry[0], SIGMA_XY, SIGMA_THETA, 1, 1, device=local, max_points=P,
                            seed=args.seed, stream=stream.cuda_stream)
        proc.set_position_search_beginning(2 ** 31 - 1)  # map-only scans: newPose = odoPose (:740-743)
        log = sn.ScanLog(n_total, P, n_offsets=0, device=local)
        for k in range(n_total):
            log.set(k, rp.points[k], rp.odometry[k])
        log.upload()
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        cur = 0
        proc.replay(log, cur, W, want_results=False)
        cur += W

        ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        sampler = ClockSampler(local)
        launches0 = proc.launch_count()
        barrier()
        sampler.start()
        wall0 = time.perf_counter()
        for i in range(K):
            flush.fill_(i & 0xFF)
            ev0[i].record(stream)
            proc.replay(log, cur + i, 1, want_results=False)
            ev1[i].record(stream)
        torch.cuda.synchronize()
        wall_region = time.perf_counter() - wall0  # this rank's own end (max over ranks below): the closing barrier is not part of the steps
        barrier()
        clocks = sampler.stop()
        launches = proc.launch_count() - launches0
        total_ms = float(sum(ev0[i].elapsed_time(ev1[i]) for i in range(K)))
        cur += K
        checksum_after_timed = int(proc.map_checksum())

        # per-kernel pass: events around the rings kernel, visits counted by the device
        proc.set_flags(N.FLAG_TIMING)
        i_ms, visits = [], []
        for i in range(Kb):
            flush.fill_(i & 0xFF)
            r = proc.replay(log, cur + i, 1, want_results=True)
            i_ms.append(proc.timing().integrate_ms)
            visits.append(r[0].visits)
        proc.set_flags(0)
        cur += Kb

        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        proc.replay(log, cur, W, want_results=False)
        e1.record(stream)
        barrier()
        warm_ms = e0.elapsed_time(e1) / W
        cur += W

        # e2e: cs_integrate through the C ABI, host points in, visit count out, wall clock
        L = sn.lib()
        fp = C.POINTER(C.c_float)
        pts_p = [rp.points[cur + i].ctypes.data_as(fp) for i in range(K)]
        pose_c = [np.ascontiguousarray(rp.odometry[cur + i]) for i in range(K)]
        v64 = C.c_int64(0)
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            st = L.cs_integrate(proc._h, pts_p[i], rp.points[cur + i].shape[0], pose_c[i].ctypes.data_as(fp), None, C.byref(v64))
            if st != 0:
                N.check(st, proc._h)
        proc.sync()
        e2e_s = time.perf_counter() - t0  # this rank's own end (max over ranks below): the closing barrier is not part of the steps
        barrier()

    mean_visits = float(np.mean(visits))
    t_all = torch.tensor([total_ms, e2e_s * 1e3, warm_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    total_ms_max, e2e_ms_max, warm_ms_max = (float(x) for x in t_all.tolist())
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
        launch_ms = float(np.mean(i_ms))
        traffic, traffic_src = latest_traffic("cs_wedge_kernel_cfg3")
        alg_bytes = 4.0 * mean_visits + 8.0 * P
        achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
        value = world * mean_visits * K / (total_ms_max * 1e-3)
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu_visits, t_cpu, done, cpu_checksum = run_cpu_cfg3(wl, rp, W, K)
            parity = bool(cpu_checksum == checksum_after_timed)
            cpu = {"value": cpu_visits / t_cpu, "unit": "visits/s", "cores": 1, "kind": "port",
                   "sample": "%d UpdateHoleMap calls (the %d timed scans of the same replay first, then the same scans again until >= 10 s), "
                             "%.1f s, 1 thread (the reference integrates serially, CoreSLAMProcessor.cs:515-533)" % (done, K, t_cpu),
                   "map_checksum_bit_exact_vs_gpu": parity}
        line = {"metric": "HoleMap cell visits/sec", "value": value, "unit": "visits/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": total_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 ray set-up -> i32 closed-form walk -> u16 blend", "data": "synthetic",
                "config": dict(config, candidates_per_scan=0, prime_scans=0, mode="integration only (search gated off)"),
                "l2": "flushed (256 MB write) before every timed step",
                "timing": "per-step CUDA events on the launching stream, summed; max over ranks",
                "visits_per_step": mean_visits, "rays_per_s": value / mean_visits * P, "clocks": clocks,
                "e2e": {"value": world * mean_visits * K / (e2e_ms_max * 1e-3), "unit": "visits/s", "h2d_bytes_per_step": 64 + 8 * P,
                        "d2h_bytes_per_step": 8, "ms_per_step": e2e_ms_max / K,
                        "api": "cs_integrate (C ABI, host points, visit count read back)"},
                "gpu_launches": int(launches),
                "replay_l2_warm": {"ms_per_step": warm_ms_max, "value": world * mean_visits / (warm_ms_max * 1e-3),
                                   "note": "same replay without L2 flushes, %d scans back to back (the 32 MB map stays in L2)" % W},
                "roofline": {"bound": "hbm", "kernel": "cs_wedge_kernel", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                             "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": launch_ms,
                             "limiter": limiter_of("cs_wedge_kernel_cfg3", launch_ms, clock_hz=(clocks.get("sm_mhz") or 1965) * 1e6),
                             "note": "4 B (2 B read + 2 B write) per visited cell + the scan's points; per-cell ray order is kept inside "
                                     "(ring range x wedge) tasks, one warp each; at this size the kernel is bound by instruction issue and "
                                     "dependency latency (see limiter), not by memory"},
                "cpu_baseline": cpu, "wall_s_timed_region": wall_region, "map_checksum": checksum_after_timed}
        print(json.dumps(line))
    proc.close()
    log.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streaming", action="store_true",
                    help="extra cfg2 measurement: a replay longer than L2 holds, queued back to back, no flush (single GPU)")
    ap.add_argument("--seed", type=int, default=0x5EED0000)
    ap.add_argument("--sessions", type=int, default=0, help="cfg5: number of sessions in the job (default: the config's 1024)")
    ap.add_argument("--sub-batches", type=int, default=0,
                    help="cfg5: independent batches (streams) a rank's sessions are run as (default 1)")
    ap.add_argument("--split", default="group", choices=["group", "nccl"],
                    help="cfg4: how the 8-byte arg-min is exchanged: inside the search kernel over peer-mapped memory (group), or by "
                         "a torch.distributed all_reduce between two kernels (nccl)")
    ap.add_argument("--no-sharded", action="store_true",
                    help="default (cfg2) line: skip the `sharded` block (cfg5 session batches and the cfg4 candidate split over the ranks)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="cfg1 / cfg2 line: write the pose and HoleMap after the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("cfg1", "cfg2") or args.streaming):
        ap.error("--dump-outputs covers the timed replay of the cfg1 / cfg2 line (--impl ours, no --streaming)")

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    K, W = args.steps, max(args.warmup, 3)
    wl = WORKLOADS[args.workload]
    P = wl["points"]
    metric = "scan-point map lookups/sec"
    config = {"workload": args.workload + ": " + wl["desc"], "points_per_scan": P,
              "candidates_per_scan": wl["threads"] * wl["iters"] + 1, "map": "%dx%d u16" % (wl["size"], wl["size"]),
              "prime_scans": PRIME_SCANS, "mode": "verification (uploaded candidate tables)",
              "sharding": {"cfg4": "candidate slices [g*C/G, (g+1)*C/G) per GPU, replicated map, one 8-byte MIN exchange per scan",
                           "cfg5": "sessions i mod G per GPU, no collective"}.get(
                               args.workload, "one independent replay per GPU, no collective" if world > 1 else "single session")}

    # ------------------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        if args.workload == "cfg3":
            from slam.net_b200 import synth
            rp = synth.make_replay(W + K, P, wl["phys"], seed=args.seed)
            visits, secs, done, _ = run_cpu_cfg3(wl, rp, W, K, min_s=cpu_min_seconds())
            v = visits / secs
            line = {"impl": "reference", "metric": "HoleMap cell visits/sec", "value": v, "unit": "visits/s", "n_gpus": args.gpus, "steps": K,
                    "updates_timed": done, "warmup": W, "ms_per_step": secs / max(done, 1) * 1e3, "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "f32 ray set-up -> i32 walk -> u16 blend", "data": "synthetic",
                    "config": dict(config, candidates_per_scan=0, prime_scans=0, mode="integration only (search gated off)"),
                    "cpu_baseline": {"value": v, "unit": "visits/s", "cores": 1, "kind": "port",
                                     "sample": "%d UpdateHoleMap calls over the %d requested scans (again back and forth until >= 10 s), %.1f s"
                                               % (done, K, secs),
                                     "note": "reference is C#/.NET (no runtime here): CPU oracle port; the reference integrates on one thread"},
                    "e2e": {"value": v, "unit": "visits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
            print(json.dumps(line))
            return 0
        n_total = PRIME_SCANS + W + K
        rp, offs, n_cand = build_workload(wl, n_total, args.seed)
        first = PRIME_SCANS + W
        v, done, T, dt, _, _ = run_cpu(wl, rp, offs, n_cand, first, K, budget_s=120.0, min_s=cpu_min_seconds())
        sample = "%d Updates over the %d requested scans of the %s replay (replayed back and forth until >= 10 s; after %d untimed " \
                 "priming/warm-up scans), %.1f s" % (done, K, args.workload, first, dt)
        line = {"impl": "reference", "metric": metric, "value": v, "unit": "lookups/s", "n_gpus": args.gpus, "steps": K, "updates_timed": done,
                "warmup": W, "ms_per_step": dt / max(done, 1) * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 transform -> u16 gather -> i64 sum", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": v, "unit": "lookups/s", "cores": T, "kind": "port", "sample": sample,
                                 "note": "reference is C#/.NET (no runtime here): CPU oracle port, ParallelWorker-style threads"},
                "e2e": {"value": v, "unit": "lookups/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    if args.workload == "cfg3":
        return run_cfg3(args, wl, config, rank, world, local, K, W)
    if args.workload in ("cfg4", "cfg5"):
        return run_sharded(args, wl, metric, config, rank, world, local, K, W)

    # ------------------------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    import slam.net_b200 as sn
    from slam.net_b200 import _native as N

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        from slam.net_b200 import parallel as _par
        if os.environ.get("CS_BENCH_NO_PIN") != "1":
            _par.pin_rank_to_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)))  # each rank on its own cores (e2e at N > 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.streaming:
        # Extra measurement (not the default line): the replay as production runs it — scans queued back to back on the
        # stream, no flush; the INPUTS are larger than L2 and each is read once from HBM, the map stays L2-resident by design.
        per_scan = 64 + 8 * P + 12 * wl["threads"] * wl["iters"]
        Ks = max(K, int(140e6 // per_scan) + 1)
        n_total = PRIME_SCANS + W + Ks
        rp, offs, n_cand = build_workload(wl, n_total, args.seed)
        stream = torch.cuda.Stream()
        with torch.cuda.stream(stream):
            proc = sn.Processor(wl["phys"], wl["size"], rp.odometry[0], SIGMA_XY, SIGMA_THETA, wl["iters"], wl["threads"],
                                device=local, max_points=P, seed=args.seed, stream=stream.cuda_stream)
            log = sn.ScanLog(n_total, P, n_offsets=n_cand, device=local)
            for k in range(n_total):
                log.set(k, rp.points[k], rp.odometry[k], offs[k])
            log.upload()
            proc.replay(log, 0, PRIME_SCANS + W, want_results=False)
            sampler = ClockSampler(local)
            launches0 = proc.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            sampler.start()
            e0.record(stream)
            proc.replay(log, PRIME_SCANS + W, Ks, want_results=False)
            e1.record(stream)
            barrier()
            clocks = sampler.stop()
            ms = e0.elapsed_time(e1)
            launches = proc.launch_count() - launches0
            value = (n_cand + 1) * P * Ks / (ms * 1e-3)
            line = {"metric": metric, "value": value, "unit": "lookups/s", "n_gpus": 1, "steps": Ks, "warmup": W, "ms_per_step": ms / Ks,
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 transform -> u16 gather -> i64 sum",
                    "data": "synthetic",
                    "config": dict(config, l2="no flush: inputs larger than L2 (%d scans x %d B = %.0f MB of points and candidate tables, each "
                                              "read once from HBM); the %.0f MB map stays L2-resident between scans by design"
                                              % (Ks, per_scan, Ks * per_scan / 1e6, wl["size"] ** 2 * 2 / 1e6),
                                   timing="one pair of CUDA events around %d Updates queued back to back (cs_replay)" % Ks),
                    "candidate_poses_per_s": value / P, "clocks": clocks, "e2e": None, "gpu_launches": int(launches),
                    "launch_shape": proc.search_plan(P), "final_pose": [float(x) for x in proc.get_pose()]}
            print(json.dumps(line))
            proc.close()
            log.close()
        return 0

    Kb = min(K, 200)  # per-kernel timing pass (roofline)
    Ke = K            # e2e pass
    n_total = PRIME_SCANS + W + K + Kb + W + Ke
    rp, offs, n_cand = build_workload(wl, n_total, args.seed + 7919 * rank)
    lookups_per_step = (n_cand + 1) * P

    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        proc = sn.Processor(wl["phys"], wl["size"], rp.odometry[0], SIGMA_XY, SIGMA_THETA, wl["iters"], wl["threads"],
                            device=local, max_points=P, seed=args.seed, stream=stream.cuda_stream)
        log = sn.ScanLog(n_total, P, n_offsets=n_cand, device=local)
        for k in range(n_total):
            log.set(k, rp.points[k], rp.odometry[k], offs[k])
        log.upload()
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

        cur = 0
        proc.replay(log, cur, PRIME_SCANS + W, want_results=False)  # priming + W warm-up steps, untimed
        cur += PRIME_SCANS + W

        # ---- timed region: K steps, L2 flushed before each, per-step CUDA events on the launching stream
        ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        sampler = ClockSampler(local)
        launches0 = proc.launch_count()
        barrier()
        sampler.start()
        wall0 = time.perf_counter()
        for i in range(K):
            flush.fill_(i & 0xFF)
            ev0[i].record(stream)
            proc.replay(log, cur + i, 1, want_results=False)
            ev1[i].record(stream)
        torch.cuda.synchronize()
        wall_region = time.perf_counter() - wall0  # this rank's own end (max over ranks below): the closing barrier is not part of the steps
        barrier()
        clocks = sampler.stop()
        launches = proc.launch_count() - launches0
        step_ms = np.array([ev0[i].elapsed_time(ev1[i]) for i in range(K)])
        total_ms = float(step_ms.sum())
        cur += K
        pose_after_timed = proc.get_pose()
        plan = proc.search_plan(P)
        if args.dump_outputs and rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "pose.npy"), pose_after_timed.astype(np.float32))
            np.save(os.path.join(args.dump_outputs, "hole_map.npy"),
                    proc.map_download().reshape(wl["size"], wl["size"]).astype(np.float32))

        # ---- per-kernel pass (roofline numerator): same replay continues, events around every kernel
        proc.set_flags(N.FLAG_TIMING)
        s_ms, i_ms = [], []
        visits = []
        for i in range(Kb):
            flush.fill_(i & 0xFF)
            r = proc.replay(log, cur + i, 1, want_results=True)
            t = proc.timing()
            s_ms.append(t.search_ms)
            i_ms.append(t.integrate_ms)
            visits.append(r[0].visits)
        proc.set_flags(0)
        cur += Kb

        # ---- steady-state replay without flushes (map stays L2-resident between scans, by design)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        proc.replay(log, cur, W, want_results=False)
        e1.record(stream)
        barrier()
        warm_ms_per_step = e0.elapsed_time(e1) / W
        cur += W

        # ---- e2e: cs_update through the C ABI with host buffers, wall clock
        L = sn.lib()
        fp = C.POINTER(C.c_float)
        res = N.Result()
        h2d = 64 + 8 * P + 12 * n_cand
        lat = np.zeros(Ke)
        pts_p = [rp.points[cur + i].ctypes.data_as(fp) for i in range(Ke)]
        odo_c = [np.ascontiguousarray(rp.odometry[cur + i]) for i in range(Ke)]
        odo_p = [a.ctypes.data_as(fp) for a in odo_c]
        off_p = [offs[cur + i].ctypes.data_as(fp) for i in range(Ke)]
        barrier()
        t0 = time.perf_counter()
        for i in range(Ke):
            ta = time.perf_counter()
            st = L.cs_update(proc._h, pts_p[i], P, odo_p[i], off_p[i], C.byref(res))
            lat[i] = time.perf_counter() - ta
            if st != 0:
                N.check(st, proc._h)
        proc.sync()
        e2e_s = time.perf_counter() - t0  # this rank's own end (max over ranks below): the closing barrier is not part of the steps
        barrier()
        final_pose = proc.get_pose()

        # ---- the same call in production mode: no candidate table, the deviates are generated on the device (Philox);
        # only the scan is uploaded.  Reported next to e2e (which is the verification mode the parity claim is made in).
        Kp = min(Ke, 200)
        latp = np.zeros(Kp)
        barrier()
        t0 = time.perf_counter()
        for i in range(Kp):
            ta = time.perf_counter()
            st = L.cs_update(proc._h, pts_p[i], P, odo_p[i], None, C.byref(res))
            latp[i] = time.perf_counter() - ta
            if st != 0:
                N.check(st, proc._h)
        proc.sync()
        prod_s = time.perf_counter() - t0  # this rank's own end (max over ranks below): the closing barrier is not part of the steps
        barrier()

    # ---- reduce over ranks: max time, summed work
    t_all = torch.tensor([total_ms, e2e_s * 1e3, warm_ms_per_step], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    total_ms_max, e2e_ms_max, warm_ms_max = (float(x) for x in t_all.tolist())
    per_rank = None  # every rank's own step time (device-timed, and end to end): where the max over ranks comes from
    step_trace = [round(float(x) * 1e3, 1) for x in step_ms] if os.environ.get("CS_BENCH_STEP_TRACE") == "1" else None
    if world > 1:
        mine_t = torch.tensor([total_ms / K, e2e_s * 1e3 / max(Ke, 1)], dtype=torch.float64, device="cuda")
        all_t = [torch.empty_like(mine_t) for _ in range(world)]
        dist.all_gather(all_t, mine_t)
        per_rank = {"ms_per_step": [float(x[0]) for x in all_t], "e2e_ms_per_step": [float(x[1]) for x in all_t]}

    value = world * lookups_per_step * K / (total_ms_max * 1e-3)
    e2e_value = world * lookups_per_step * Ke / (e2e_ms_max * 1e-3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
        search_ms = float(np.mean(s_ms))
        alg_bytes = 2.0 * lookups_per_step + 8.0 * P + 12.0 * n_cand + 8.0
        achieved = alg_bytes / (search_ms * 1e-3) / 1e9
        try:
            gather_peak = sn.gather_peak(wl["size"] * wl["size"], 256, 5, device=local)
        except Exception as e:  # noqa
            gather_peak = None
        search_rate = lookups_per_step / (search_ms * 1e-3)
        kname = "cs_search2_kernel" if plan["slab"] else "cs_search_kernel"
        draw_kernel = "cs_rings_kernel" if os.environ.get("CS_TUNE_INTEGRATE") == "1" else "cs_wedge_kernel"
        traffic, traffic_src = latest_traffic(kname) if args.workload == "cfg2" else (None, None)  # the captures are cfg2's
        integrate_ms = float(np.mean(i_ms))
        step_s = total_ms_max / K * 1e-3
        sm_clock = (clocks.get("sm_mhz") or 1965) * 1e6
        roofline = {"bound": "hbm", "kernel": plan["kernel"] + " (+ the Update glue and pose hand-off in its last warp/block)",
                    "launch_shape": plan, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": search_ms,
                    "note": "the contract's HBM fraction of the dominant stage (search: sort + search kernels, events around the stage): "
                            "2-byte gathers out of an L2-resident map, so this number is small by construction and is NOT what limits "
                            "the stage — `limiter` says what does, per kernel, from the newest ncu capture of the same sources",
                    "limiter": {"search": dict(limiter_of(kname, search_ms, clock_hz=sm_clock) or {},
                                               what="issue + latency: ~24 issue slots per lookup with L1-resident tiles; the stage "
                                                    "also holds the candidate sort, the cold first touch of the map and the pose hand-off"),
                                "integrate": dict(limiter_of(draw_kernel, integrate_ms, clock_hz=sm_clock) or {},
                                                  what="latency chain pose -> rays -> wedge tasks (no block-wide barrier in the draw "
                                                       "loop); issue-bound only for big scans (cfg3)")},
                    "gather": {"achieved_lookups_per_s": search_rate, "peak_lookups_per_s": gather_peak,
                               "frac": (search_rate / gather_peak) if gather_peak else None,
                               "whole_update_frac": (lookups_per_step / step_s / gather_peak) if gather_peak else None,
                               "peak_source": "cs_gather_peak: random u16 loads over a table the size of the map (one line per lane), "
                                              "measured in this run; `frac` is the search stage alone, `whole_update_frac` the "
                                              "lookups of a step over the whole step time"},
                    "integrate": {"kernel": draw_kernel, "launch_ms": integrate_ms,
                                  "visits_per_launch": float(np.mean(visits)),
                                  "achieved_GBps": 4.0 * float(np.mean(visits)) / (integrate_ms * 1e-3) / 1e9,
                                  "frac_of_hbm": 4.0 * float(np.mean(visits)) / (integrate_ms * 1e-3) / 1e9 / hbm_peak,
                                  "note": "4 B (read + write) per visited cell; ordered per cell"}}

        cpu = None
        if not args.no_cpu_baseline and world == 1:
            first = PRIME_SCANS + W
            v, done, T, dt, cpu_pose, complete = run_cpu(wl, rp, offs, n_cand, first, K, budget_s=25.0, min_s=10.0)
            parity = bool(complete and np.array_equal(cpu_pose, pose_after_timed))
            cpu = {"value": v, "unit": "lookups/s", "cores": T, "kind": "port",
                   "sample": "%d Updates over the %d timed scans of the same replay (replayed back and forth until >= 10 s) after %d "
                             "untimed scans, %.1f s, %d threads (search) + 1 thread (integration)" % (done, K, first, dt, T),
                   "pose_bit_exact_vs_gpu": parity if complete else None}
            # the simulator's own setting: 4 search threads (Simulation/MainWindow.xaml.cs:69), a shorter sample of the same scans
            v4, done4, T4, dt4, _, _ = run_cpu(wl, rp, offs, n_cand, first, min(K, 100), budget_s=8.0, min_s=4.0, threads=4)
            cpu["simulator_setting"] = {"value": v4, "unit": "lookups/s", "cores": T4,
                                        "sample": "%d Updates of the same replay, %.1f s, %d search threads as in the reference's simulator" % (done4, dt4, T4)}

        line = {"metric": metric, "value": value, "unit": "lookups/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": total_ms_max / K, "per_rank": per_rank, "step_trace_us_rank0": step_trace, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 transform -> u16 gather -> i64 sum", "data": "synthetic",
                "config": config,
                "l2": "flushed (256 MB write) before every timed step; e2e inputs arrive from host memory each step",
                "timing": "per-step CUDA events on the launching stream, summed; max over ranks",
                "candidate_poses_per_s": value / P,
                "per_gpu": {"value": value / world, "e2e": e2e_value / world,
                            "note": "whole-job numbers are N independent replays; the reference arm is ONE CPU process whatever N is, "
                                    "so a ratio against it is meaningful per GPU"},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "lookups/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 32,
                        "ms_per_step": e2e_ms_max / Ke, "api": "cs_update (C ABI, host buffers, pinned staging, mapped result)",
                        "scan_to_pose_latency_ms": {"p50": float(np.percentile(lat, 50) * 1e3),
                                                    "p99": float(np.percentile(lat, 99) * 1e3)}},
                "gpu_launches": int(launches),
                "e2e_production_mode": {"value": lookups_per_step * Kp / prod_s, "unit": "lookups/s", "ms_per_step": prod_s / Kp * 1e3,
                                        "h2d_bytes_per_step": 64 + 8 * P, "d2h_bytes_per_step": 32, "steps": Kp,
                                        "api": "cs_update(cand_offsets = NULL): on-device Philox candidates, rank 0",
                                        "scan_to_pose_latency_ms": {"p50": float(np.percentile(latp, 50) * 1e3),
                                                                    "p99": float(np.percentile(latp, 99) * 1e3)}},
                "replay_l2_warm": {"ms_per_step": warm_ms_max, "value": world * lookups_per_step / (warm_ms_max * 1e-3),
                                   "note": "same replay without L2 flushes, %d scans back to back" % W},
                "sort_ahead": ("off (CS_TUNE_PRESORT=-1): every step sorts its candidate table in front of its search" if os.environ.get("CS_TUNE_PRESORT") == "-1" else
                               "`value` replays a device-resident log, so the library queues the candidate sort of scan k+1 behind the draw "
                               "kernel of scan k: every timed step still holds exactly one sort (the next scan's, under its own draw kernel), "
                               "none in front of its search; `e2e` uploads a table with every scan and sorts in front of the search; "
                               "`e2e_production_mode` generates candidates on the device and sorts ahead like `value`"),
                "roofline": roofline,
                "cpu_baseline": cpu,
                "wall_s_timed_region": wall_region,
                "final_pose": [float(x) for x in final_pose]}

    proc.close()
    log.close()
    # ---- the configs that shard (BASELINE configs[3], [4]), measured in the same run over the same ranks so that the
    # driver's --gpus N lines carry them: cfg5 = 1024 session replays sharded i mod N (strong scaling, no collective),
    # cfg4 = 65536 candidates split over the ranks with one 8-byte MIN exchange per scan
    sharded = None
    if not args.no_sharded:
        Ks = min(K, 20)
        sharded = {"cfg5": measure_cfg5(args, rank, world, local, Ks, 3, sub_batches=args.sub_batches),
                   "cfg4": measure_cfg4(args, rank, world, local, Ks, 3)}
    if rank == 0:
        line["sharded"] = sharded
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
