"""Task queues of the fleet step (ttmpc_fleet_step_tasks_device) on the CPU: tt_atan2 against
mpmath, the oracle's get_global_ref_traj sampler against the reference's own trajectories, the
mission step of tests/fleet_tasks_ref.py against the single-robot host mirror ``InterfaceMpc``
driven as a mission loop (solver replaced by a recorder), the ctypes layout of struct
ttmpc_fleet_tasks and the argument checks of the new entry point."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.fleet import BAD_TASK, GOAL_REACH, work_mode
from trajtrack_mpcndqn_rlboost_b200.planner import TrajectoryGenerator
from tests.fleet_action_steps_ref import FleetHostK, fleet_advance_k
from tests import fleet_tasks_ref as R
from tests.fleet_tasks_ref import TaskQueues, pack_tasks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ulps(a, b):
    a, b = np.float64(a), np.float64(b)
    if a == b:
        return 0
    if np.sign(a) != np.sign(b):
        return 1 << 62
    return abs(int(a.view(np.int64)) - int(b.view(np.int64)))


def test_tt_atan2_within_one_ulp_of_mpmath():
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.prec = 120
    rng = np.random.default_rng(11)
    ang = rng.uniform(-np.pi, np.pi, 100_000)
    mag = np.exp(rng.uniform(-8.0, 8.0, 100_000))
    pairs = list(zip(mag * np.sin(ang), mag * np.cos(ang)))
    tiny, huge = 1e-300, 1e300
    for sy in (1.0, -1.0):
        for sx in (1.0, -1.0):   # four quadrants, axes, ratios near 0 and infinity
            pairs += [(sy * 1.0, sx * 1.0), (sy * 0.0, sx * 1.0), (sy * 1.0, sx * 0.0), (sy * 0.0, sx * 0.0),
                      (sy * tiny, sx * 1.0), (sy * 1.0, sx * tiny), (sy * 1e-20, sx * 3.0), (sy * 3.0, sx * 1e-20),
                      (sy * huge, sx * 1.0), (sy * 1.0, sx * huge), (sy * 0.5, sx * 1.0), (sy * 1.5, sx * 1.0),
                      (sy * 2.4375, sx * 1.0), (sy * 0.4375, sx * 1.0), (sy * 0.6875, sx * 1.0), (sy * 1.1875, sx * 1.0),
                      (sy * math.inf, sx * 1.0), (sy * 1.0, sx * math.inf), (sy * math.inf, sx * math.inf)]
    worst = 0
    for y, x in pairs:
        got = R.atan2(y, x)
        if math.isinf(x) or math.isinf(y) or x == 0.0 or y == 0.0:   # IEEE 754 special values, signed zeros
            want = math.atan2(y, x)
            assert got == want and math.copysign(1, got) == math.copysign(1, want), (y, x, got)
            continue
        want = float(mpmath.atan2(mpmath.mpf(y), mpmath.mpf(x)))
        d = _ulps(got, want)
        assert d <= 1, (y, x, got, want)
        worst = max(worst, d)
    assert math.isnan(R.atan2(math.nan, 1.0)) and math.isnan(R.atan2(1.0, math.nan))


def test_oracle_sampler_reproduces_reference_trajectories():
    g = np.load(os.path.join(ROOT, "tests", "golden", "host_logic.npz"))
    names = sorted(k for k in g.files if k.startswith("gref_") and k.count("_") == 2)
    assert len(names) == 9
    for k in names:
        want = g[k]
        st, speed = g[k + "_state"], float(g[k + "_speed"])
        got = R.global_ref_traj(g[k + "_path"], st[0], st[1], 0.2, speed, 100_000, use_libm=True)
        assert got is not None and got.shape == want.shape, k
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-12, err_msg=k)
        # too small a cap, and the device arithmetic within ulps of libm's
        assert R.global_ref_traj(g[k + "_path"], st[0], st[1], 0.2, speed, len(want) - 1) is None
        dev = R.global_ref_traj(g[k + "_path"], st[0], st[1], 0.2, speed, len(want), use_libm=False)
        np.testing.assert_allclose(dev, want, rtol=0, atol=1e-12, err_msg=k)
    assert R.global_ref_traj(np.zeros((0, 2)), 1.0, 1.0, 0.2, 1.0, 100) is None
    # the walk the reference indexes past the last node in: starting on the only node, a duplicated last node
    assert R.global_ref_traj([(1.0, 2.0)], 1.0, 2.0, 0.2, 1.0, 100) is None
    assert R.global_ref_traj([(0.0, 0.0), (1.0, 0.0), (1.0, 0.0)], 0.0, 0.0, 0.2, 1.0, 100) is None
    with pytest.raises(IndexError):
        TrajectoryGenerator.get_global_ref_traj(0.2, [(0.0, 0.0), (1.0, 0.0), (1.0, 0.0)], (0.0, 0.0), 1.0)


# ------------------------------------------------------------------ mission loop against the mirror
class _Sol:
    def __init__(self, u):
        self.solution = list(u); self.cost = 1.25; self.exit_status = "Converged"; self.solve_time_ms = 0.5


class _Recorder:
    """Stands in for the mirror's Solver: records p and returns a steering law's controls, computed
    from the mirror's state and current goal when the solve is called."""
    def __init__(self, mirror, N):
        self.m, self.N, self.p_log, self.u_log = mirror, N, [], []

    def run(self, p, initial_guess=None):
        self.p_log.append(np.array(p, dtype=np.float64))
        x, y, th = self.m.state
        gx, gy = self.m.goal[:2]
        d = math.hypot(gx - x, gy - y)
        a = math.atan2(gy - y, gx - x) - th
        a = math.atan2(math.sin(a), math.cos(a))
        v = min(1.0, 2.0 * d) * max(0.0, math.cos(a))
        w = max(-1.5, min(1.5, a / 0.2))
        u = np.tile([v, w], self.N)
        self.u_log.append(u)
        return _Sol(u)


def _host_sampler(path, x, y, ts, speed, cap):
    try:
        rows = TrajectoryGenerator.get_global_ref_traj(ts, [tuple(q) for q in path], (x, y), speed)
    except IndexError:
        return None
    return rows if 0 < len(rows) <= cap else None


def _missions(n):
    """Three tasks per robot after the first, 1-2 m legs.  Robot 1 has two goals 3 cm apart (it
    takes two tasks in one step); robot 2's second task repeats its last node (the reference's
    walk indexes past it: BAD_TASK)."""
    rng = np.random.default_rng(8)
    init = np.zeros((n, 3)); goal = np.zeros((n, 3)); paths = []; tg = []; tp = []
    for e in range(n):
        x, y, h = rng.uniform(5, 15), rng.uniform(5, 15), rng.uniform(-np.pi, np.pi)
        init[e] = (x, y, h)
        pts = [(x, y)]
        for _ in range(4):
            h += rng.uniform(-1.2, 1.2)
            L = rng.uniform(1.0, 2.0)
            pts.append((pts[-1][0] + L * math.cos(h), pts[-1][1] + L * math.sin(h)))
        goal[e] = (*pts[1], 0.0)
        paths.append([pts[0], pts[1]])
        tg.append([(*pts[i + 1], 0.0) for i in range(1, 4)])
        tp.append([[pts[i], pts[i + 1]] for i in range(1, 4)])
    g1 = tg[1][0]
    tg[1][1] = (g1[0] + 0.03, g1[1] - 0.01, 0.0)
    tp[1][1] = [g1[:2], tg[1][1][:2]]
    tp[1][2] = [tg[1][1][:2], tg[1][2][:2]]
    tp[2][1] = [tp[2][1][0], tp[2][1][1], tp[2][1][1]]
    return init, goal, paths, tg, tp


@pytest.mark.parametrize("k", [1, 2])
def test_mission_reference_matches_interface_mpc(k):
    n, steps = 7, 90
    mc = t.Configurator()
    mc.action_steps = k
    cfg = mc.to_ttmpc()
    N = cfg.N_hor
    off = t.param_offsets(cfg)
    init, goal, paths, tg, tp = _missions(n)
    fp = t.FleetPlanner(mc, init, goal, paths, mode="work", device="cpu", action_steps=k)
    fp.set_tasks(tg, tp)
    tuning, base = work_mode(mc, "work")
    fh = FleetHostK(cfg, init, goal, fp.ref_traj.numpy(), fp.ref_len.numpy(), np.zeros(cfg.Nstcobs * cfg.nstcobs),
                    tuning, base, mc.low_speed, action_steps=k)
    tq = TaskQueues(tg, tp)
    mirrors, recs, left = [], [], []
    for e in range(n):
        m = t.InterfaceMpc(mc)
        m._traj_gen.solver = rec = _Recorder(m, N)
        m.initialization(init[e].copy(), goal[e].copy(), paths[e], mode="work")
        mirrors.append(m); recs.append(rec); left.append(list(zip(tg[e], tp[e])))
    prev_u = np.zeros((n, 2 * N))
    done, switches_ref, switches_mirror, multi = {}, [], [], set()
    for s in range(steps):
        nxt = tq.next.copy()
        p, took = pack_tasks(fh, tq, prev_u, use_libm=True, sampler=_host_sampler)
        switches_ref += [(e, s) for e in np.flatnonzero(tq.next > nxt) for _ in range(tq.next[e] - nxt[e])]
        U = np.zeros((n, 2 * N))
        for e, m in enumerate(mirrors):
            if e in done:
                continue
            n_before, taken = len(recs[e].p_log), 0
            ref_local, _ = m.get_local_ref_traj()
            ret = m.get_action(ref_local, mode="work")
            while ret is None and left[e]:
                (g, q), left[e] = left[e][0], left[e][1:]
                switches_mirror.append((e, s)); taken += 1
                try:
                    m.initialization(m.state, np.array(g), q, mode="work")
                except IndexError:
                    done[e] = "bad"
                    break
                ref_local, _ = m.get_local_ref_traj()
                ret = m.get_action(ref_local, mode="work")
            if taken > 1:
                multi.add(e)
            if e in done:
                assert fh.status[e] == BAD_TASK, f"robot {e} step {s}"
                continue
            assert int(fh.idx_ref[e]) == m._traj_gen.idx_ref, f"idx_ref of robot {e} at step {s}"
            assert np.array_equal(fh.goal[e], m.goal), f"goal of robot {e} at step {s}"
            if ret is None:
                done[e] = "reached"
                assert fh.status[e] == 1, f"robot {e} should stop at step {s}"
                continue
            assert fh.status[e] == 0, f"robot {e} should drive on at step {s}"
            gp = recs[e].p_log[n_before]
            mask = np.ones(len(gp), bool)
            mask[off["vref"]:off["c"]] = False
            assert np.array_equal(p[e][mask], gp[mask]), f"packed vector of robot {e} at step {s}"
            np.testing.assert_allclose(p[e][~mask], gp[~mask], rtol=4e-16, atol=0)
            U[e] = recs[e].u_log[-1]
        fleet_advance_k(fh, U, np.zeros(n, np.int32), use_libm=True)
        prev_u = np.where((fh.status == 0)[:, None], U, prev_u)
        for e, m in enumerate(mirrors):
            if done.get(e) != "bad":
                np.testing.assert_allclose(fh.state[e], m.state, rtol=0, atol=2e-15, err_msg=f"robot {e} step {s}")
        if len(done) == n:
            break
    assert switches_ref == switches_mirror
    assert len(switches_ref) >= 2 * n                      # switches happened, for every robot
    assert 1 in multi and done.get(2) == "bad" and fh.status[2] == BAD_TASK
    assert sum(v == "reached" for v in done.values()) == n - 1, done
    assert np.array_equal(tq.next, [3, 3, 2, 3, 3, 3, 3])


# ------------------------------------------------------------------ C-ABI
def test_fleet_tasks_struct_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    fields = [f for f, _ in _lib.TtmpcFleetTasks._fields_]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "ttmpc.h"\nint main(void) {\n'
                   '  printf("%zu %d", sizeof(ttmpc_fleet_tasks), TTMPC_FLEET_BAD_TASK);\n'
                   + "".join(f'  printf(" %zu", offsetof(ttmpc_fleet_tasks, {f}));\n' for f in fields)
                   + '  printf("\\n"); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    vals = list(map(int, subprocess.check_output([str(exe)]).split()))
    assert C.sizeof(_lib.TtmpcFleetTasks) == vals[0]
    assert BAD_TASK == vals[1]
    assert [getattr(_lib.TtmpcFleetTasks, f).offset for f in fields] == vals[2:]


def test_step_tasks_argument_checks():
    lib = _lib.load()
    mc = t.Configurator()
    cfg = mc.to_ttmpc()
    n, N = 4, cfg.N_hor
    tuning, base = work_mode(mc, "work")
    fh = FleetHostK(cfg, np.zeros((n, 3)), np.ones((n, 3)), np.zeros((n, 8, 3)), [8] * n,
                    np.zeros(cfg.Nstcobs * cfg.nstcobs), tuning, base, mc.low_speed)
    f = fh.struct()
    p = np.zeros((n, lib.ttmpc_num_params(C.byref(cfg)))); u = np.zeros((n, 2 * N)); es = np.zeros(n, np.int32)
    res = _lib.TtmpcResult(u=u.ctypes.data, exit_status=es.ctypes.data)
    cnt = np.ones(n, np.int32); nxt = np.zeros(n, np.int32); g = np.zeros((n, 1, 3)); xy = np.zeros((n, 1, 2, 2))
    pn = np.full((n, 1), 2, np.int32)

    def tasks(**kw):
        tk = _lib.TtmpcFleetTasks(max_tasks=1, max_nodes=2, count=cnt.ctypes.data, next=nxt.ctypes.data,
                                  goal=g.ctypes.data, path_xy=xy.ctypes.data, path_n=pn.ctypes.data)
        for key, v in kw.items():
            setattr(tk, key, v)
        return tk

    def call(tk):
        return lib.ttmpc_fleet_step_tasks_device(C.byref(cfg), C.byref(f), tk, p.ctypes.data, 1, C.byref(res), None)

    BAD_ARG = -2
    assert call(None) == BAD_ARG
    for kw in (dict(max_tasks=-1), dict(max_nodes=0), dict(count=None), dict(next=None), dict(goal=None),
               dict(path_xy=None), dict(path_n=None), dict(path_out=xy.ctypes.data)):
        assert call(C.byref(tasks(**kw))) == BAD_ARG, kw
        assert "tasks" in lib.ttmpc_last_error().decode()
    assert not p.any() and not fh.status.any() and not nxt.any()


# ------------------------------------------------------------------ host side
def test_set_tasks_grows_stride_to_cover_every_task():
    mc = t.Configurator()
    m = t.scenes.make_missions(12, 4, seed=3)
    fp = t.FleetPlanner(mc, m["init"], m["goal"], m["paths"], mode="work", device="cpu")
    rows0, len0, stride0 = fp.ref_traj.numpy().copy(), fp.ref_len.numpy().copy(), fp.ref_stride
    # a long last task: the stride must grow
    goals = [list(g) for g in m["task_goals"]]; paths = [list(q) for q in m["task_paths"]]
    gx, gy, _ = goals[0][-1]
    goals[0].append((gx + 30.1, gy, 0.0)); paths[0].append([(gx, gy), (gx + 30.1, gy)])
    fp.set_tasks(goals, paths)
    assert fp.ref_stride > stride0 and fp.tasks.max_tasks == 4 and fp.tasks.max_nodes == 3
    assert np.array_equal(fp.ref_traj.numpy()[:, :stride0], rows0) and not fp.ref_traj.numpy()[:, stride0:].any()
    assert np.array_equal(fp.ref_len.numpy(), len0)
    assert fp.task_count.tolist() == [4] + [3] * 11 and not fp.task_next.any()
    rng = np.random.default_rng(0)
    base = fp.base_speed
    for e in range(12):
        prev = m["goal"][e]
        for g, q in zip(goals[e], paths[e]):
            for _ in range(5):   # starts within GOAL_REACH of the previous goal
                a, r = rng.uniform(-np.pi, np.pi), GOAL_REACH * np.sqrt(rng.uniform())
                st = (prev[0] + r * np.cos(a), prev[1] + r * np.sin(a))
                assert len(TrajectoryGenerator.get_global_ref_traj(mc.ts, q, st, base)) <= fp.ref_stride
            prev = g
    fp.set_tasks([[] for _ in range(12)], [[] for _ in range(12)])
    assert fp.tasks is None
    with pytest.raises(ValueError):
        fp.set_tasks(goals[:3], paths[:3])


def test_make_missions_chains_tasks():
    m = t.scenes.make_missions(20, 4, seed=1000)
    assert t.scenes.make_missions(20, 4, seed=1000)["init"].tolist() == m["init"].tolist()
    for e in range(20):
        goals = [m["goal"][e]] + list(m["task_goals"][e])
        paths = [m["paths"][e]] + list(m["task_paths"][e])
        assert len(goals) == len(paths) == 4
        assert np.allclose(paths[0][0], m["init"][e][:2], atol=0.5)
        for i in range(4):
            assert np.array_equal(paths[i][-1], goals[i][:2])
            if i:
                assert np.array_equal(paths[i][0], goals[i - 1][:2])
        assert len(m["static_polys"][e]) == 8
    assert m["moving_pos"].shape == (20, 2, 2) and m["moving_disp"].shape == (20, 2, 2)
