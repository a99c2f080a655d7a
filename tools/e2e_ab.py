"""A/B of the number of host calls in flight inside one process: alternates legs of BatchSolver.run_many
(20 steps of static4096 from pinned host memory) over the depths below and prints the solves/s of every leg
plus the medians.  Round 2, one B200: 5 calls in flight 552 k (mean of 7), 6 calls 537 k, 7 calls 530 k,
8 calls 527 k; letting the parameter blocks of concurrent calls take turns on the PCIe link (tried, removed)
changed nothing (536 k against 541 k).
usage: python tools/e2e_ab.py [repeats]"""
import os, sys, time, statistics
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import trajtrack_mpcndqn_rlboost_b200 as t
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
w = t.scenes.WORKLOADS["static4096"]
cfg = t.Configurator().to_ttmpc(**w["solver"])
ps = []
for j in range(4):
    p = t.scenes.make_scenes(w["n"], cfg, seed=1000 + 100 * j, n_static=w["n_static"], n_dynamic=w["n_dynamic"],
                             blocking_fraction=w["blocking_fraction"])
    pp = t.pinned_empty(p.shape); pp[...] = p; ps.append(pp)
s = t.BatchSolver(cfg)
s.run_many(ps + ps, depth=6)
def leg(depth, steps=20):
    t0 = time.perf_counter(); s.run_many([ps[i % 4] for i in range(steps)], depth=depth); dt = time.perf_counter() - t0
    return 4096 * steps / dt / 1e3
cases = {"depth 5": 5, "depth 6": 6, "depth 7": 7, "depth 8": 8}
res = {k: [] for k in cases}
for r in range(reps):
    for k, d in cases.items():
        res[k].append(leg(d))
for k, v in res.items():
    print(f"{k:32s} median {statistics.median(v):6.0f} k solves/s   runs {[round(x) for x in v]}", flush=True)
