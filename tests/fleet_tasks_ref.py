"""CPU restatement of the fleet step with task queues (``ttmpc_fleet_step_tasks_device``) on top of
the fleet oracle of tests/oracle_lib.py and the task oracle oracle/ttfleet_tasks_oracle.c (bound
here) -- TEST INFRASTRUCTURE.

The mission step is composed from the oracle's unchanged pack and advance and its sampler
``ttfleet_oracle_global_ref_traj``:

* pack every robot (closest point, goal test, HintSwitcher, parameter vector);
* every robot that is REACHED with a task left takes it, as ``InterfaceMpc.initialization`` does:
  goal, reference trajectory sampled from its current state, ``idx_ref = 0``, ``last_u = 0``,
  RUNNING.  Then it is packed again on its own, which repeats the search from 0 and the goal test
  on the new task; a robot whose new goal is already reached takes the next task.  A task that
  cannot be driven stops the robot as BAD_TASK and leaves goal, rows, idx_ref and last_u as they
  were.  The HintSwitcher state of a robot that took a task is the one of its last RUNNING pack
  (once, on the new task); if the robot is not RUNNING afterwards it keeps its state from before the
  step and is packed from it without the search;
* with a warm start, robots that took a task start from zeros.

``OracleFleetTasks.step`` is what ``FleetPlanner.step`` computes with tasks queued, with the solve
in the kernel's WARP order, so the two agree bit for bit.
"""
from __future__ import annotations

import copy
import ctypes as C
import os
import subprocess

import numpy as np

from tests import oracle_lib as O
from tests.fleet_action_steps_ref import FleetHostK, OracleFleetK, fleet_advance_k, fleet_pack_k, warm_start_k
from tests.fleet_options_ref import RUNNING

REACHED, BAD_TASK = 1, 3

TASKS_ORACLE_PATH = os.path.join(O.ROOT, "oracle", "libttfleet_tasks_oracle.so")
_lib = None


def load():
    """oracle/libttfleet_tasks_oracle.so (built by ``make``; compiled here when it is missing)."""
    global _lib
    if _lib is None:
        if not os.path.exists(TASKS_ORACLE_PATH):
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", TASKS_ORACLE_PATH,
                                   os.path.join(O.ROOT, "oracle", "ttfleet_tasks_oracle.c"), "-lm"])
        lib = C.CDLL(TASKS_ORACLE_PATH)
        D = C.c_double
        lib.ttmpc_oracle_atan2.argtypes = [D, D]
        lib.ttmpc_oracle_atan2.restype = D
        lib.ttfleet_oracle_global_ref_traj.argtypes = [C.c_void_p, C.c_int, D, D, D, D, C.c_int, C.c_void_p, C.c_int]
        lib.ttfleet_oracle_global_ref_traj.restype = C.c_int
        _lib = lib
    return _lib


def atan2(y, x):
    """tt_atan2 of the kernels (csrc/ttmpc_device.cuh)."""
    return load().ttmpc_oracle_atan2(float(y), float(x))


def global_ref_traj(path, x, y, ts, speed, cap, use_libm=True):
    """get_global_ref_traj of a queued task from (x, y): rows [r][3], or None for a task that cannot
    be driven (ttfleet_oracle_global_ref_traj returns -1)."""
    xy = np.ascontiguousarray(np.asarray(path, np.float64).reshape(-1, 2))
    out = np.zeros((max(int(cap), 1), 3))
    r = load().ttfleet_oracle_global_ref_traj(xy.ctypes.data, len(xy), float(x), float(y), float(ts), float(speed),
                                              int(cap), out.ctypes.data, 1 if use_libm else 0)
    return None if r < 0 else out[:r].copy()


class TaskQueues:
    """Host copy of struct ttmpc_fleet_tasks: goals [n][T][3], paths [n][T][M][2], counts, cursor."""

    def __init__(self, goals, paths, max_nodes=None):
        n = len(goals)
        T = max(1, max(len(g) for g in goals))
        M = max_nodes or max([1] + [len(q) for pl in paths for q in pl])
        self.count = np.array([len(g) for g in goals], np.int32)
        self.next = np.zeros(n, np.int32)
        self.goal = np.zeros((n, T, 3))
        self.path_xy = np.zeros((n, T, M, 2))
        self.path_n = np.zeros((n, T), np.int32)
        for e in range(n):
            for k, (g, q) in enumerate(zip(goals[e], paths[e])):
                a = np.asarray(q, np.float64).reshape(-1, 2)
                self.goal[e, k] = g
                self.path_xy[e, k, :len(a)] = a
                self.path_n[e, k] = len(a)
        self.path_out = np.zeros((n, M, 2))
        self.path_out_n = np.zeros(n, np.int32)


def oracle_sampler(use_libm):
    def sample(path, x, y, ts, speed, cap):
        return global_ref_traj(path, x, y, ts, speed, cap, use_libm=use_libm)
    return sample


def _view(fh, e):
    """A one-robot FleetHostK whose arrays are views of robot e's rows (writes go through)."""
    v = copy.copy(fh)
    v.n = 1
    sl = slice(e, e + 1)
    for name in ("state", "goal", "last_u", "idx_ref", "status", "ref_traj", "ref_len", "other", "dyn_cur",
                 "dyn_last", "dyn_disp", "hint", "use_hint", "sw_state"):
        a = getattr(fh, name)
        if a is not None:
            setattr(v, name, a[sl])
    if not fh.stc_shared:
        v.stc = fh.stc[sl]
    if fh.sw_poly_xy is not None and fh.sw_poly_xy.shape[0] != 1:
        v.sw_poly_xy, v.sw_poly_nv = fh.sw_poly_xy[sl], fh.sw_poly_nv[sl]
    return v


def pack_tasks(fh: FleetHostK, tq: TaskQueues, prev_u, use_libm: bool, sampler=None):
    """The pack kernel of the task step.  Returns (p, took): took[e] is True where robot e took a
    task in this step.  sampler(path, x, y, ts, speed, cap) -> rows or None (default: the oracle's)."""
    sampler = sampler or oracle_sampler(use_libm)
    sw = fh.sw_state is not None and fh.hint is not None
    if sw:
        fh.sw_state = np.ascontiguousarray(fh.sw_state, dtype=np.int32)
        fh.use_hint = np.ascontiguousarray(fh.use_hint, dtype=np.int32)
        pre = (fh.sw_state.copy(), fh.use_hint.copy())
    prev_u = np.asarray(prev_u, dtype=np.float64)
    p = fleet_pack_k(fh, prev_u, use_libm)
    took = np.zeros(fh.n, bool)
    ts = fh.cfg.ts
    for e in np.flatnonzero((fh.status == REACHED) & (tq.next < tq.count)):
        v = _view(fh, e)
        while fh.status[e] == REACHED and tq.next[e] < tq.count[e]:
            t = tq.next[e]
            tq.next[e] += 1
            path = tq.path_xy[e, t, :tq.path_n[e, t]]
            rows = sampler(path, fh.state[e, 0], fh.state[e, 1], ts, fh.base_speed, fh.ref_traj.shape[1])
            if rows is None:
                fh.status[e] = BAD_TASK
                break
            fh.ref_traj[e, :len(rows)] = rows
            fh.ref_len[e] = len(rows)
            fh.goal[e] = tq.goal[e, t]
            fh.last_u[e] = 0.0
            fh.idx_ref[e] = 0
            fh.status[e] = RUNNING
            tq.path_out[e, :len(path)] = path
            tq.path_out_n[e] = len(path)
            took[e] = True
            if sw:
                fh.sw_state[e], fh.use_hint[e] = pre[0][e], pre[1][e]
            p[e] = fleet_pack_k(v, prev_u[e:e + 1], use_libm)[0]
        if took[e] and fh.status[e] != RUNNING:
            if sw:
                fh.sw_state[e], fh.use_hint[e] = pre[0][e], pre[1][e]
            p[e] = fleet_pack_k(v, prev_u[e:e + 1], use_libm)[0]   # not RUNNING: no search, no switch
    return p, took


class OracleFleetTasks(OracleFleetK):
    """The closed loop of FleetPlanner.step(keep_multipliers=True, warm_start, skip_stopped) with task
    queues, on an oracle FleetHostK."""

    def __init__(self, fh, cfg, tq: TaskQueues, threads=8):
        super().__init__(fh, cfg, threads)
        self.tq = tq
        self.took = None

    def step(self, warm=False, skip=False):
        fh, r, k = self.fh, self.res, self.fh.action_steps
        self.p, self.took = pack_tasks(fh, self.tq, r["u"], use_libm=False)
        if warm:
            u0 = warm_start_k(fh.status, r["u"], r["exit_status"], k)
            u0[self.took & (fh.status == RUNNING)] = 0.0
        else:
            u0 = np.zeros_like(r["u"])
        idx = np.flatnonzero(fh.status == RUNNING) if skip else np.arange(fh.n)
        self.solved = idx
        if len(idx):
            s = O.solve_batch(self.cfg, self.p[idx], u0=u0[idx], y0=r["y"][idx], threads=self.threads, warp=True)
            for name in self.FIELDS:
                r[name][idx] = s[name]
        fleet_advance_k(fh, r["u"], r["exit_status"], use_libm=False)
