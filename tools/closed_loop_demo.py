#!/usr/bin/env python
"""Functional check of the whole stack: n robots drive their reference paths to the goal with the
device-resident fleet loop; reports how many arrive, the closest approach to the static obstacles
and the tracking error.
  python tools/closed_loop_demo.py [n=1024] [max_steps=200] [--warm-start] [--skip-stopped] [--action-steps k]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import trajtrack_mpcndqn_rlboost_b200 as t


def point_poly_clearance(px, py, polys):
    """Signed clearance of points [n] to per-robot axis-aligned rectangles [n][k][4][2] (negative inside)."""
    lo = polys.min(axis=2); hi = polys.max(axis=2)                     # [n][k][2]
    dx = np.maximum(np.maximum(lo[..., 0] - px[:, None], px[:, None] - hi[..., 0]), 0.0)
    dy = np.maximum(np.maximum(lo[..., 1] - py[:, None], py[:, None] - hi[..., 1]), 0.0)
    outside = np.hypot(dx, dy)
    inside = np.minimum(np.minimum(px[:, None] - lo[..., 0], hi[..., 0] - px[:, None]),
                        np.minimum(py[:, None] - lo[..., 1], hi[..., 1] - py[:, None]))
    return np.where(outside > 0, outside, -np.maximum(inside, 0.0)).min(axis=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int, nargs="?", default=1024)
    ap.add_argument("max_steps", type=int, nargs="?", default=200)
    ap.add_argument("--warm-start", action="store_true", help="FleetPlanner.step(warm_start=True)")
    ap.add_argument("--skip-stopped", action="store_true", help="FleetPlanner.step(skip_stopped=True)")
    ap.add_argument("--action-steps", type=int, default=1, help="FleetPlanner(action_steps=k)")
    a = ap.parse_args()
    n, max_steps = a.n, a.max_steps
    mc = t.Configurator()
    fl = t.scenes.make_fleet(n, seed=7)
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", action_steps=a.action_steps)
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    fp.set_moving_obstacles(fl["moving_pos"], fl["moving_disp"])
    polys = np.array(fl["static_polys"], dtype=np.float64)               # [n][k][4][2]
    clearance = np.full(n, np.inf)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    steps = 0
    for k in range(max_steps):
        fp.step(warm_start=a.warm_start, skip_stopped=a.skip_stopped)
        steps += 1
        if k % 5 == 4:
            st = fp.state.cpu().numpy()
            clearance = np.minimum(clearance, point_poly_clearance(st[:, 0], st[:, 1], polys))
            if int((fp.status == 0).sum()) == 0:
                break
    e1.record(); torch.cuda.synchronize()
    status = fp.status.cpu().numpy(); st = fp.state.cpu().numpy()
    dist_goal = np.hypot(st[:, 0] - fl["goal"][:, 0], st[:, 1] - fl["goal"][:, 1])
    out = dict(robots=n, warm_start=a.warm_start, skip_stopped=a.skip_stopped, action_steps=a.action_steps, steps=steps, wall_ms=e0.elapsed_time(e1), reached=int((status == 1).sum()),
               failed=int((status == 2).sum()), still_running=int((status == 0).sum()),
               dist_to_goal_p50=float(np.median(dist_goal)), dist_to_goal_max=float(dist_goal.max()),
               min_clearance_to_static_obstacles=float(clearance.min()),
               robots_that_entered_an_obstacle=int((clearance < 0).sum()))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
