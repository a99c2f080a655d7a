#!/usr/bin/env python
"""Fleet missions on one GPU: robots take their next task on arrival, on the device or from the host.

  python tools/bench_missions.py [n=4096] [max_steps=300] [--tasks 4] [--profile-pack]

Workload: scenes.make_missions(n, tasks, seed=1000): every robot has a chain of `tasks` tasks (the
first given to the FleetPlanner constructor, the others queued).  Legs, on the same scenario, run
interleaved as S WS H H WS S:
  S, WS  FleetPlanner.set_tasks + step(skip_stopped=True[, warm_start=True]): a robot that arrives
         takes its next task inside the step (ttmpc_fleet_step_tasks_device), no host round trip.
  H      host re-tasking, step(skip_stopped=True) without queues: after every step the host syncs,
         finds the robots that arrived, samples their next task with
         TrajectoryGenerator.get_global_ref_traj and writes rows, goal, idx_ref, last_u and status
         back through tensors.  Such a robot drives its new task from the next step on.
Every leg runs until no robot is RUNNING or max_steps steps have run.  Per leg: tasks completed
(tasks taken + robots REACHED at the end), steps, drive time (wall clock, including the host leg's
host work), tasks/s and robot-steps/s over it, per-step GPU time p50 / p90 (events), and for H the
host time (spent in the re-task code, including the sync that waits for the step).  The card's name and power limit are read in the same run.  Prints one JSON line and
writes no file.

--profile-pack instead reports the fleet_pack_kernel time (torch.profiler) of one step in which every
robot takes a task and of the next, in which none does.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.fleet import BAD_TASK, REACHED, RUNNING
from trajtrack_mpcndqn_rlboost_b200.planner import TrajectoryGenerator

LEGS = ["S", "WS", "H", "H", "WS", "S"]


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    return dict(gpu=torch.cuda.get_device_name(), power_limit=pl or None)


def make(mc, m, queued=True):
    fp = t.FleetPlanner(mc, m["init"], m["goal"], m["paths"], mode="work")
    fp.update_static_constraints(m["static_polys"], per_robot=True)
    fp.set_moving_obstacles(m["moving_pos"], m["moving_disp"])
    fp.set_tasks(m["task_goals"], m["task_paths"])   # also sizes ref_stride for every task
    if not queued:
        fp.tasks = None
    return fp


class HostRetask:
    """The host side of re-tasking: InterfaceMpc.initialization for every robot that arrived."""

    def __init__(self, fp, m):
        self.fp, self.m = fp, m
        self.next = np.zeros(fp.n, np.int64)
        self.count = np.array([len(g) for g in m["task_goals"]])

    def __call__(self):
        fp = self.fp
        status = fp.status.cpu().numpy()                                      # the device-to-host sync
        idx = np.flatnonzero((status == REACHED) & (self.next < self.count))
        if len(idx) == 0:
            return 0
        state = fp.state[idx].cpu().numpy()
        rows = np.zeros((len(idx), fp.ref_stride, 3))
        rlen, goal, st = np.zeros(len(idx), np.int32), np.zeros((len(idx), 3)), np.full(len(idx), RUNNING, np.int32)
        for j, e in enumerate(idx):
            k = self.next[e]
            self.next[e] += 1
            goal[j] = self.m["task_goals"][e][k]
            try:
                r = TrajectoryGenerator.get_global_ref_traj(fp.config.ts, self.m["task_paths"][e][k], state[j], fp.base_speed)
            except IndexError:
                r = np.zeros((0, 3))
            if not 0 < len(r) <= fp.ref_stride:
                st[j] = BAD_TASK
                continue
            rows[j, :len(r)] = r
            rlen[j] = len(r)
        dev = fp.state.device
        ok = torch.from_numpy(st == RUNNING).to(dev)
        ti = torch.from_numpy(idx).to(dev)
        tj = ti[ok]
        fp.ref_traj[tj] = torch.from_numpy(rows).to(dev)[ok]
        fp.ref_len[tj] = torch.from_numpy(rlen).to(dev)[ok]
        fp.goal[tj] = torch.from_numpy(goal).to(dev)[ok]
        fp.idx_ref[tj] = 0
        fp.last_u[tj] = 0.0
        fp.status[ti] = torch.from_numpy(st).to(dev)
        return len(idx)

    def completed(self):
        return int(self.next.sum() + (self.fp.status == REACHED).sum().item())


def drive(mc, m, leg, max_steps):
    host = leg == "H"
    fp = make(mc, m, queued=not host)
    rt = HostRetask(fp, m) if host else None
    torch.cuda.synchronize()
    ev, host_s, robot_steps = [], 0.0, torch.zeros((), dtype=torch.int64, device=fp.state.device)
    t0 = time.perf_counter()
    for k in range(max_steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fp.step(warm_start="W" in leg, skip_stopped=True)
        e1.record()
        ev.append((e0, e1))
        robot_steps += (fp.status == RUNNING).sum()
        if host:
            h0 = time.perf_counter()
            rt()
            host_s += time.perf_counter() - h0
        if (host or k % 5 == 4) and int((fp.status == RUNNING).sum()) == 0:
            break
    torch.cuda.synchronize()
    drive_s = time.perf_counter() - t0
    ms = [a.elapsed_time(b) for a, b in ev]
    done = rt.completed() if host else int(fp.task_next.sum().item() + (fp.status == REACHED).sum().item())
    status = fp.status.cpu().numpy()
    out = dict(leg=leg, tasks_completed=done, steps=len(ms), drive_s=drive_s, tasks_per_s=done / drive_s,
               robot_steps_per_s=int(robot_steps) / drive_s, step_ms_p50=float(np.quantile(ms, 0.5)),
               step_ms_p90=float(np.quantile(ms, 0.9)), reached=int((status == REACHED).sum()),
               running=int((status == RUNNING).sum()), bad_task=int((status == BAD_TASK).sum()),
               failed=int((status == 2).sum()))
    if host:
        out["host_s"] = host_s
    return out


def profile_pack(mc, m):
    from torch.profiler import ProfilerActivity, profile
    n = len(m["init"])
    m = dict(m, init=m["init"].copy())
    m["init"][:, :2] = m["goal"][:, :2] + 0.01                 # every robot arrives in the first step
    warm = make(mc, m)
    warm.step(skip_stopped=True); warm.step(skip_stopped=True)
    fp = make(mc, m)
    torch.cuda.synchronize()
    res = {}
    for name in ("all_switch", "no_switch"):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fp.step(skip_stopped=True)
            torch.cuda.synchronize()
        ev = [e for e in prof.key_averages() if "fleet_pack_kernel" in e.key]
        res[name] = dict(pack_us=float(sum(e.device_time_total for e in ev)), launches=int(sum(e.count for e in ev)))
    res["switched_in_first_step"] = int((fp.task_next == 1).sum().item())
    res["robots"] = n
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int, nargs="?", default=4096)
    ap.add_argument("max_steps", type=int, nargs="?", default=300)
    ap.add_argument("--tasks", type=int, default=4)
    ap.add_argument("--profile-pack", action="store_true")
    a = ap.parse_args()
    mc = t.Configurator()
    m = t.scenes.make_missions(a.n, a.tasks, seed=1000)
    out = dict(workload=f"missions{a.n}x{a.tasks}", robots=a.n, tasks=a.tasks, max_steps=a.max_steps, **card())
    if a.profile_pack:
        out["profile_pack"] = profile_pack(mc, m)
        print(json.dumps(out))
        return
    warm = make(mc, m)  # module loads and first-launch costs stay out of the legs
    for _ in range(3):
        warm.step(warm_start=True, skip_stopped=True)
    torch.cuda.synchronize()
    del warm
    legs = [drive(mc, m, leg, a.max_steps) for leg in LEGS]
    mean = {}
    for leg in dict.fromkeys(LEGS):
        rs = [r for r in legs if r["leg"] == leg]
        mean[leg] = {k: float(np.mean([r[k] for r in rs])) for k in rs[0] if k != "leg"}
    out.update(legs=legs, mean=mean)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
