"""Diagnostics: per-scan device times of the search and draw kernels over a long cfg2 replay."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import slam.net_b200 as sn
from slam.net_b200 import synth, _native as N
P, size = 1024, 2048
n = int(sys.argv[1]) if len(sys.argv) > 1 else 700
rp = synth.make_replay(n, P, 40.0)
p = sn.Processor(40.0, size, rp.odometry[0], 0.1, 0.17, 1024, 4, max_points=P, flags=N.FLAG_TIMING)
log = sn.ScanLog(n, P, n_offsets=4096)
for k in range(n):
    log.set(k, rp.points[k], rp.odometry[k], synth.candidate_offsets(1, k, 4096, 0.1, 0.17))
log.upload()
s, g, v = [], [], []
for k in range(n):
    r = p.replay(log, k, 1, want_results=True)
    t = p.timing()
    s.append(t.search_ms * 1e3); g.append(t.integrate_ms * 1e3); v.append(r[0].visits)
s, g, v = np.array(s), np.array(g), np.array(v)
for a in range(0, n, 50):
    b = min(n, a + 50)
    print("scans %4d-%4d: search mean %.1f max %.1f | draw mean %.1f max %.1f | visits %.0f | min wall dist %.2f m" % (
        a, b, s[a:b].mean(), s[a:b].max(), g[a:b].mean(), g[a:b].max(), v[a:b].mean(),
        min(np.hypot(rp.points[k][:, 0], rp.points[k][:, 1]).min() for k in range(a, b))))
