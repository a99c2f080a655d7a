#!/usr/bin/env python
"""Shared obstacle map on one GPU: the map selection kernel and a warehouse drive.

  python tools/bench_world.py [--select-only | --drive-only] [--steps 300]

(a) Selection: scenes.make_warehouse(n, tasks=1, seed=1000, shelves=M) for n in {4096, 16384} and
    M in {1e3, 1e4, 1e5} (the same shelf density at every M).  From the robots' start states,
    fleet_world_select_kernel time from CUDA events over 200 warm launches (mean per launch), next to
    the time of the whole step (selection + pack + solve + advance, warm start and skip-stopped) of the
    same fleet, mean over 10 steps after 3 warm-up steps.  Also the largest and mean world_reach.
(b) Drive: make_warehouse(4096, tasks=4, seed=1000) for --steps steps, legs S and WS interleaved as
    S WS WS S (tools/bench_missions.py): step(skip_stopped=True[, warm_start=True]) with the monitor
    on the map.  Per leg: tasks completed, per-step time p50 / p90 (events), robots with a contact,
    the largest world_reach over the drive and the robot-steps with world_reach > Nstcobs.
Prints one JSON line per measurement, each with the card's name and power limit read in the same run;
writes no file.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.fleet import REACHED, RUNNING

LEGS = ["S", "WS", "WS", "S"]


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    return dict(gpu=torch.cuda.get_device_name(), power_limit=pl or None)


def planner(mc, w):
    fp = t.FleetPlanner(mc, w["init"], w["goal"], w["paths"], mode="work")
    fp.set_world(w["world_polys"])
    if any(w["task_goals"]):
        fp.set_tasks(w["task_goals"], w["task_paths"])
    return fp


def select(mc, n, M, launches=200):
    w = t.scenes.make_warehouse(n, 1, seed=1000, shelves=M)
    fp = planner(mc, w)
    for _ in range(10):
        fp.run_world_select()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        fp.run_world_select()
    e1.record()
    torch.cuda.synchronize()
    sel_ms = e0.elapsed_time(e1) / launches
    reach = fp.world_reach.cpu().numpy()
    for _ in range(3):
        fp.step(warm_start=True, skip_stopped=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(10):
        fp.step(warm_start=True, skip_stopped=True)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / 10
    return dict(bench="world_select", robots=n, shelves=fp.world.M, select_ms=sel_ms, step_ms=step_ms,
                select_share_of_step=sel_ms / step_ms, world_reach_max=int(reach.max()),
                world_reach_mean=float(reach.mean()), nstcobs=mc.Nstcobs, **card())


def drive(mc, w, leg, steps):
    fp = planner(mc, w)
    fp.enable_monitor()
    K = fp.config.Nstcobs
    dev = fp.state.device
    reach_max = torch.zeros((), dtype=torch.int32, device=dev)
    overflow = torch.zeros((), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    ev = []
    for k in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fp.step(warm_start="W" in leg, skip_stopped=True)
        e1.record()
        ev.append((e0, e1))
        reach_max = torch.maximum(reach_max, fp.world_reach.max())
        overflow += (fp.world_reach > K).sum()
        if k % 5 == 4 and int((fp.status == RUNNING).sum()) == 0:
            break
    torch.cuda.synchronize()
    ms = [a.elapsed_time(b) for a, b in ev]
    status = fp.status.cpu().numpy()
    return dict(leg=leg, steps=len(ms),
                tasks_completed=int(fp.task_next.sum().item() + (fp.status == REACHED).sum().item()),
                step_ms_p50=float(np.quantile(ms, 0.5)), step_ms_p90=float(np.quantile(ms, 0.9)),
                robots_with_contact=int((fp.contact_steps > 0).sum().item()),
                reached=int((status == REACHED).sum()), running=int((status == RUNNING).sum()),
                world_reach_max=int(reach_max.item()), robot_steps_reach_over_nstcobs=int(overflow.item()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--select-only", action="store_true")
    ap.add_argument("--drive-only", action="store_true")
    ap.add_argument("--steps", type=int, default=300)
    a = ap.parse_args()
    mc = t.Configurator()
    if not a.drive_only:
        for n in (4096, 16384):
            for M in (1_000, 10_000, 100_000):
                print(json.dumps(select(mc, n, M)), flush=True)
    if not a.select_only:
        w = t.scenes.make_warehouse(4096, 4, seed=1000)
        warm = planner(mc, w)  # module loads and first-launch costs stay out of the legs
        for _ in range(3):
            warm.step(warm_start=True, skip_stopped=True)
        torch.cuda.synchronize()
        del warm
        legs = [drive(mc, w, leg, a.steps) for leg in LEGS]
        mean = {}
        for leg in dict.fromkeys(LEGS):
            rs = [r for r in legs if r["leg"] == leg]
            mean[leg] = {k: float(np.mean([r[k] for r in rs])) for k in rs[0] if k != "leg"}
        print(json.dumps(dict(bench="world_drive", workload="warehouse4096x4", robots=4096, tasks=4,
                              shelves=len(w["world_polys"]), max_steps=a.steps, nstcobs=mc.Nstcobs, legs=legs,
                              mean=mean, **card())), flush=True)


if __name__ == "__main__":
    main()
