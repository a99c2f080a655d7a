#!/usr/bin/env python
"""DQN-boosted closed loop on one GPU (BASELINE configs[3]): per control step and environment

  internal observation -> lidar sectors/rays + Q-net + argmax -> rl_ref hint rollout
  -> pack (hint as reference positions) -> NMPC solve -> advance

all device-resident (ttdqn_internal_obs_device, ttdqn_observe_act_device, ttdqn_rl_ref_device,
ttmpc_fleet_step_device); whether the hint is used is decided per step and environment by the
HintSwitcher logic inside the pack kernel.
  python tools/bench_hybrid.py [n=16384] [steps=10] [--warm-start] [--skip-stopped] [--action-steps k]
                               [--lidar-moving] [--monitor]

--lidar-moving: the lidar also sees the moving obstacles, as the circle_to_rect squares the
HintSwitcher uses, at the positions the step's pack treats as current (ttdqn_observe_act_moving_device;
FleetPlanner.enable_dqn(moving_shape="rect") does the same).  Off by default, so that numbers stay
comparable with earlier runs.
--monitor: the default monitor of FleetPlanner.enable_monitor, run after each step's end event,
outside the timed window (as tools/bench_fleet.py does); reports reached robots, robots with a
contact and the deepest entry into a moving obstacle's disc (-min clearance; a static polygon's
clearance is never below 0).  The 3 warm-up steps count for the monitor too.
The card's name and power limit are read in the same run.
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
from trajtrack_mpcndqn_rlboost_b200.fleet import DYN_OBS_SIZE, REACHED

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    return dict(gpu=torch.cuda.get_device_name(), power_limit=pl or None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int, nargs="?", default=16384)
    ap.add_argument("steps", type=int, nargs="?", default=10)
    ap.add_argument("--warm-start", action="store_true", help="FleetPlanner.step(warm_start=True)")
    ap.add_argument("--skip-stopped", action="store_true", help="FleetPlanner.step(skip_stopped=True)")
    ap.add_argument("--action-steps", type=int, default=1, help="FleetPlanner(action_steps=k)")
    ap.add_argument("--lidar-moving", action="store_true", help="the lidar sees the moving obstacles' squares")
    ap.add_argument("--monitor", action="store_true", help="run the fleet monitor outside the timed window")
    a = ap.parse_args()
    n, steps = a.n, a.steps
    mc = t.Configurator()
    fl = t.scenes.make_fleet(n, seed=1000)
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", action_steps=a.action_steps)
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    fp.set_moving_obstacles(fl["moving_pos"], fl["moving_disp"])
    # lidar geometry: each env's rectangles (padded by the robot radius) + a boundary ring
    g = np.load(os.path.join(ROOT, "tests", "golden", "qnet_ray.npz"))
    wq = t.dqn.QNetWeights(*[g[k] for k in ("w0", "b0", "w1", "b1", "w2", "b2")])
    lay = t.dqn.default_layout(max_poly=6, max_vert=192)
    rings, solid = [], []
    for i in range(n):
        r = [t.geometry.pad_polygon_round(np.array(poly), 0.5) for poly in fl["static_polys"][i]]
        x0, y0 = fl["init"][i, 0], fl["init"][i, 1]
        r.append(np.array([(x0 - 30, y0 - 30), (x0 + 30, y0 - 30), (x0 + 30, y0 + 30), (x0 - 30, y0 + 30)]))
        rings.append(r); solid.append([True] * (len(r) - 1) + [False])
    xy, off, sol, cnt = t.dqn.pack_geometry(lay, rings, solid)
    xy, off, sol, cnt = (torch.from_numpy(a).cuda() for a in (xy, off, sol, cnt))
    pxy, pcnt = t.dqn.pack_paths(fl["paths"])
    pxy, pcnt = torch.from_numpy(pxy).cuda(), torch.from_numpy(pcnt).cuda()
    comp = t.dqn.DqnCompanion(lay, wq); qs = wq.device_struct()
    old = torch.zeros(n, 16, dtype=torch.float32, device="cuda")
    out = dict(ext=torch.zeros(n, 32, device="cuda"), q=torch.zeros(n, 9, device="cuda"),
               action=torch.zeros(n, dtype=torch.int32, device="cuda"))
    internal = torch.empty(n, 14, dtype=torch.float32, device="cuda")
    progress = torch.empty(n, dtype=torch.float64, device="cuda")
    rl = torch.empty(n, fp.N, 2, dtype=torch.float64, device="cuda")
    use = torch.zeros(n, dtype=torch.int32, device="cuda")
    agent5 = torch.empty(n, 5, dtype=torch.float64, device="cuda")
    fp.set_hint(rl, use)
    fp.enable_hint_switch(fl["static_polys"], per_robot=True)      # HintSwitcher(10, 2, 10), main.py:129
    moving = None
    if a.lidar_moving:                                              # the switcher's squares, one template for all
        k = fp.n_dyn_live
        moving = (fp.dyn_cur, torch.from_numpy(np.repeat(t.dqn.rect_shape(DYN_OBS_SIZE)[None, None], k, 1)).cuda(),
                  torch.full((1, k), 4, dtype=torch.int32, device="cuda"))
    if a.monitor:
        fp.enable_monitor()
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def one_step(times=None):
        e = [ev() for _ in range(3)]
        e[0].record()
        agent5[:, :3] = fp.state; agent5[:, 3:] = fp.last_u          # env.set_agent_state (main.py:175-176)
        t.dqn.internal_obs_device(agent5, pxy, pcnt, out=internal, progress=progress)
        comp.observe_act_device(fp.state, xy, off, sol, cnt, internal, old, out, qs, moving=moving)
        t.dqn.rl_ref_device(agent5, out["action"], steps=fp.N, ts=mc.ts, ref_speed=1.0, out=rl)
        e[1].record()
        fp.step(keep_multipliers=os.environ.get('KEEP_Y', '1') == '1', warm_start=a.warm_start,
                skip_stopped=a.skip_stopped, monitor=False)
        e[2].record()
        if a.monitor:
            fp.run_monitor()
        if times is not None:
            torch.cuda.synchronize()
            times.append((e[0].elapsed_time(e[2]), e[0].elapsed_time(e[1])))
    for _ in range(3):
        one_step()
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        one_step(times)
    tt = np.array(times)
    res = dict(workload=f"hybrid{n}", envs=n, **card(), warm_start=a.warm_start, skip_stopped=a.skip_stopped,
               action_steps=a.action_steps, lidar_moving=a.lidar_moving, steps=steps, step_ms_p50=float(np.median(tt[:, 0])),
               step_ms_p90=float(np.quantile(tt[:, 0], 0.9)), dqn_part_ms_p50=float(np.median(tt[:, 1])),
               env_steps_per_s=n / (float(np.median(tt[:, 0])) * 1e-3),
               actions_hist=np.bincount(out["action"].cpu().numpy(), minlength=9).tolist(),
               running=int((fp.status == 0).sum()), mean_inner_iters=float(fp.inner.float().mean()),
               hint_on=int(fp.use_hint.sum()))
    if a.monitor:
        res.update(reached=int((fp.status == REACHED).sum()), robots_with_contact=int((fp.contact_steps > 0).sum()),
                   deepest_moving_disc_entry=max(0.0, -float(fp.min_clearance.min())))
    print(json.dumps(res))
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "bench_hybrid.json"), "a") as f:
        f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
