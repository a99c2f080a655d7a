#!/usr/bin/env python
"""The fleet monitor (ttmpc_fleet_monitor_device) on one GPU: its kernel time, and what it reports
about a closed-loop drive.

  python tools/bench_monitor.py [--sizes 4096 16384] [--launches 200] [--drive-robots 4096] [--drive-steps 200]

Kernel time: make_fleet(n, seed=1000) geometry (four rectangles and two moving obstacles per robot),
three warm, skip-stopped steps, then --launches monitor launches on the chords of the third step.
Each launch is timed by its own pair of CUDA events, and prev_xy is restored before each one outside
the pair.  A sleep kernel ahead of the loop keeps the GPU behind the host, so the events time the
kernel and not the launch; if the sleep ends before the host has queued every launch, the loop is
repeated with a longer one.  Reported per size: p50 and mean of the launch times.

Drive: make_fleet(4096, seed=1000), --drive-steps steps with warm start and skip-stopped, and the
default monitor (the robot centre against the polygons the MPC sees, DYN_OBS_SIZE discs for the
moving obstacles).  Reported: reached / failed / running robots, robots with a contact,
quantiles of min_clearance, and mean and largest tracking deviation.  The same drive again with
moving_radius = 0 ("static_only") separates the contacts with rectangles from those with the
moving obstacles' discs.

The card's name and power limit are read in the same run.  Prints one JSON line.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.fleet import COLLIDED, FAILED, REACHED, RUNNING


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    return dict(gpu=torch.cuda.get_device_name(), power_limit=pl or None)


def make(n, mc, fl):
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work")
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    fp.set_moving_obstacles(fl["moving_pos"], fl["moving_disp"])
    fp.enable_monitor()
    return fp


def kernel_time(n, mc, launches):
    fp = make(n, mc, t.scenes.make_fleet(n, seed=1000))
    for _ in range(2):
        fp.step(warm_start=True, skip_stopped=True)
    fp.step(warm_start=True, skip_stopped=True, monitor=False)
    prev = fp.prev_xy.clone()                       # the chords of the third step
    for _ in range(10):                             # warm-up
        fp.prev_xy.copy_(prev)
        fp.run_monitor()
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream
    cfg, f, m = C.byref(fp.cfg), C.byref(fp._fleet_struct()), C.byref(fp.monitor)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(launches)]
    cycles = 2_000_000 * launches                   # about 1 ms of sleep per launch at 1.9 GHz
    for _ in range(4):
        torch.cuda._sleep(cycles)                   # the host queues every launch before the GPU gets there
        asleep = torch.cuda.Event()
        asleep.record()
        rc = 0
        for e0, e1 in ev:
            fp.prev_xy.copy_(prev)
            e0.record()
            rc = rc or fp.lib.ttmpc_fleet_monitor_device(cfg, f, m, st)
            e1.record()
        caught_up = asleep.query()                  # the sleep ended while launches were still queued
        torch.cuda.synchronize()
        if rc:
            raise RuntimeError(f"ttmpc_fleet_monitor_device returned {rc}")
        if not caught_up:
            break
        cycles *= 4
    else:
        raise RuntimeError("the GPU kept up with the launches: no kernel time measured")
    us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
    contact = int((fp.clearance <= 0).sum())
    return dict(robots=n, launches=launches, kernel_us_p50=float(np.median(us)), kernel_us_mean=float(us.mean()),
                robots_in_contact_on_the_timed_chords=contact)


def drive(n, mc, steps, moving_radius=None):
    fp = make(n, mc, t.scenes.make_fleet(n, seed=1000))
    if moving_radius is not None:
        fp.enable_monitor(moving_radius=moving_radius)
    for _ in range(steps):
        fp.step(warm_start=True, skip_stopped=True)
    torch.cuda.synchronize()
    st = fp.status.cpu().numpy()
    mn = fp.min_clearance.cpu().numpy()
    moved = fp.moved_steps.cpu().numpy()
    qs = (0.0, 0.01, 0.05, 0.1, 0.5)
    return dict(robots=n, steps=steps, options="WS", robot_radius=0.0, moving_radius=fp.monitor.moving_radius,
                reached=int((st == REACHED).sum()), failed=int((st == FAILED).sum()),
                running=int((st == RUNNING).sum()), collided=int((st == COLLIDED).sum()),
                robots_with_contact=int((fp.contact_steps > 0).sum()),
                contact_steps_total=int(fp.contact_steps.sum()),
                min_clearance_quantiles={str(q): float(np.quantile(mn, q)) for q in qs},
                deviation_mean=float(fp.deviation_sum.sum()) / max(1, int(moved.sum())),
                deviation_max=float(fp.deviation_max.max()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--drive-robots", type=int, default=4096)
    ap.add_argument("--drive-steps", type=int, default=200)
    a = ap.parse_args()
    if a.launches < 1:
        ap.error("--launches must be >= 1")
    mc = t.Configurator()
    out = dict(tool="bench_monitor", **card())
    out["kernel"] = [kernel_time(n, mc, a.launches) for n in a.sizes]
    out["drive"] = drive(a.drive_robots, mc, a.drive_steps) if a.drive_steps > 0 else None
    out["drive_static_only"] = drive(a.drive_robots, mc, a.drive_steps, moving_radius=0.0) if a.drive_steps > 0 else None
    print(json.dumps(out))


if __name__ == "__main__":
    main()
