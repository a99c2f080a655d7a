#!/usr/bin/env python
"""Closed-loop fleet drive on one GPU, with and without the fleet-step options.

  python tools/bench_fleet.py [n=4096] [max_steps=200] [--action-steps k]

Each leg builds the same seeded fleet and calls FleetPlanner.step() -- pack + solve + advance,
multipliers carried from step to step -- until every robot has stopped or max_steps steps have
run.  Legs: options off (0), warm start (W), skip stopped robots (S) and both (WS), run
interleaved as 0 W S WS WS S W 0 so that drift of the card affects every option alike.  Every leg
runs with the same action_steps k.  Per leg: drive time (sum of the per-step event times), step
p50 / p90, PANOC iterations (device counters, ttmpc_read_stats), reached / failed / running
robots at the end, robots that touched an obstacle (the default monitor of
FleetPlanner.enable_monitor, run after each step's end event, outside the timed window), and two
rates over the drive time: robot-seconds per wall-second (k * ts of robot time for every robot
that moved in a step, the time the reference's loop accounts for) and
metres driven per wall-second (the robots' summed displacement; with k > 1 a step moves a robot by
one RK4 step with its k-th control, see include/ttmpc.h).  The card's name and power limit are read
in the same run.  Also the CPU oracle (reference order, all host cores) doing one plain step on a
bounded sample.  Prints one JSON line.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.fleet import work_mode
from tests import oracle_lib as O

LEGS = ["0", "W", "S", "WS", "WS", "S", "W", "0"]


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    return dict(gpu=torch.cuda.get_device_name(), power_limit=pl or None)


def make(n, mc, fl, k):
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", action_steps=k)
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    fp.set_moving_obstacles(fl["moving_pos"], fl["moving_disp"])
    fp.enable_monitor()
    return fp


def drive(fp, leg, max_steps):
    stats = (C.c_ulonglong * 4)()
    _lib.check(fp.lib.ttmpc_read_stats(stats, 1), "ttmpc_read_stats")
    ev = []
    moved = torch.zeros((), dtype=torch.int64, device=fp.state.device)     # robots that moved, summed over steps
    metres = torch.zeros((), dtype=torch.float64, device=fp.state.device)
    for k in range(max_steps):
        xy = fp.state[:, :2].clone()                                        # outside the timed window
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fp.step(warm_start="W" in leg, skip_stopped="S" in leg, monitor=False)
        e1.record()
        fp.run_monitor()
        ev.append((e0, e1))
        moved += (fp.status == 0).sum()    # RUNNING after a step = took this step's controls
        metres += (fp.state[:, :2] - xy).norm(dim=1).sum()
        if k % 5 == 4 and int((fp.status == 0).sum()) == 0:
            break
    torch.cuda.synchronize()
    _lib.check(fp.lib.ttmpc_read_stats(stats, 0), "ttmpc_read_stats")
    ms = [a.elapsed_time(b) for a, b in ev]
    status = fp.status.cpu().numpy()
    q = lambda p: float(np.quantile(ms, p))
    drive_s = float(np.sum(ms)) * 1e-3
    return dict(leg=leg, steps=len(ms), drive_ms=float(np.sum(ms)), step_ms_p50=q(0.5), step_ms_p90=q(0.9),
                robot_s_per_s=int(moved) * fp.action_steps * fp.config.ts / drive_s,
                metres_per_s=float(metres) / drive_s,
                panoc_iters=int(stats[3]), reached=int((status == 1).sum()), failed=int((status == 2).sum()),
                running=int((status == 0).sum()), contact=int((fp.contact_steps > 0).sum()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int, nargs="?", default=4096)
    ap.add_argument("max_steps", type=int, nargs="?", default=200)
    ap.add_argument("--action-steps", type=int, default=1, help="FleetPlanner(action_steps=k)")
    a = ap.parse_args()
    n, max_steps, ks = a.n, a.max_steps, a.action_steps
    mc = t.Configurator()
    fl = t.scenes.make_fleet(n, seed=1000)
    warm = make(n, mc, fl, ks)  # module loads and first-launch costs stay out of the legs
    for _ in range(3):
        warm.step(warm_start=True, skip_stopped=True)
    torch.cuda.synchronize()
    legs = [drive(make(n, mc, fl, ks), leg, max_steps) for leg in LEGS]
    mean = {}
    for leg in dict.fromkeys(LEGS):
        rs = [r for r in legs if r["leg"] == leg]
        mean[leg] = {k: float(np.mean([r[k] for r in rs]))
                     for k in ("drive_ms", "step_ms_p50", "step_ms_p90", "robot_s_per_s", "metres_per_s", "panoc_iters")}
        mean[leg].update({k: rs[-1][k] for k in ("steps", "reached", "failed", "running", "contact")})
    out = dict(workload=f"fleet{n}", robots=n, max_steps=max_steps, action_steps=ks, **card(), legs=legs, mean=mean)
    # CPU: one plain step with the oracle (reference operation order), bounded sample
    ns = min(n, 256)
    tuning, base = work_mode(mc, "work")
    fh = O.FleetHost(warm.cfg, fl["init"][:ns], fl["goal"][:ns], warm.ref_traj.cpu().numpy()[:ns], warm.ref_len.cpu().numpy()[:ns],
                     warm.stc.cpu().numpy()[:ns], tuning, base, mc.low_speed, dyn_cur=fl["moving_pos"][:ns], dyn_disp=fl["moving_disp"][:ns])
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    for _ in range(2):
        p = O.fleet_pack(fh, use_libm=True)
        ref = O.solve_batch(warm.cfg, p, threads=cores, warp=False)
        O.fleet_advance(fh, ref["u"], ref["exit_status"], use_libm=True)
    dt = (time.perf_counter() - t0) / 2
    out["cpu_baseline"] = dict(robot_steps_per_s=ns / dt, cores=cores, kind="port", sample=f"{ns} robots x 2 steps")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
