"""Diagnostic: host-path throughput (BatchSolver.run_many, pinned inputs) of this process at several
depths; run several copies at once (one per GPU) to see how ranks disturb each other.
usage: CUDA_VISIBLE_DEVICES=k python tools/e2e_probe.py [start_epoch_seconds]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import trajtrack_mpcndqn_rlboost_b200 as t
start = float(sys.argv[1]) if len(sys.argv) > 1 else 0.0
short = os.environ.get("PROBE_SHORT") == "1"
if "LOCAL_RANK" in os.environ:            # under torchrun: one GPU per rank
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
if os.environ.get("PROBE_NCCL") == "1":  # does an initialised NCCL communicator disturb the host path?
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    dist.barrier(); torch.cuda.synchronize()
w = t.scenes.WORKLOADS["static4096"]
cfg = t.Configurator().to_ttmpc(**w["solver"])
ps = []
for j in range(4):
    p = t.scenes.make_scenes(w["n"], cfg, seed=1000 + 100 * j, n_static=w["n_static"], n_dynamic=w["n_dynamic"], blocking_fraction=w["blocking_fraction"])
    pp = t.pinned_empty(p.shape); pp[...] = p; ps.append(pp)
s = t.BatchSolver(cfg)
s.run_many(ps + ps, depth=6)
tag = os.environ.get("LOCAL_RANK", os.environ.get("CUDA_VISIBLE_DEVICES", "?")) + ("/nccl" if os.environ.get("PROBE_NCCL") == "1" else "") + "/omp" + os.environ.get("OMP_NUM_THREADS", "-")
print(tag, "cpus", len(os.sched_getaffinity(0)), flush=True)
k = 0
def leg(name, depth, steps=18):
    global k
    # all copies start each leg at the same wall-clock time
    k += 1
    if start:
        while time.time() < start + 6.0 * k: time.sleep(0.001)
    t0 = time.perf_counter(); s.run_many([ps[i % 4] for i in range(steps)], depth=depth); dt = time.perf_counter() - t0
    print(f"{tag} {name}: {1e3 * dt / steps:.2f} ms per step = {4096 * steps / dt / 1e3:.0f} k solves/s", flush=True)
leg("depth 6", 6)
if short: sys.exit(0)
leg("depth 3", 3)
leg("depth 2", 2)
leg("depth 1", 1, steps=8)
leg("depth 6 again", 6)
