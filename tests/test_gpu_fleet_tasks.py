"""Task queues of the fleet step on the GPU (FleetPlanner.set_tasks -> ttmpc_fleet_step_tasks_device)
against the WARP-order oracle reference of tests/fleet_tasks_ref.py, bit for bit."""
import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.fleet import BAD_TASK, REACHED, RUNNING, work_mode
from tests import fleet_tasks_ref as R
from tests.fleet_action_steps_ref import FleetHostK
from tests.fleet_tasks_ref import OracleFleetTasks, TaskQueues

pytestmark = pytest.mark.gpu

SOLVER = dict(max_inner_iterations=40, max_outer_iterations=3)
OPTIONS = dict(none=(False, False), warm=(True, False), skip=(False, True), warm_skip=(True, True))


def _short_missions(n, tasks, seed, scale=0.15):
    """make_missions shrunk about every robot's start: 1-2.5 m per task, so that robots finish
    several tasks in a few dozen steps.  The first goal is 2 cm from the start: every robot takes
    its second task in the first step."""
    m = t.scenes.make_missions(n, tasks, seed=seed)
    for e in range(n):
        o = m["init"][e, :2].copy()
        sx = lambda q: tuple(o + scale * (np.asarray(q[:2], np.float64) - o))
        m["paths"][e] = [sx(q) for q in m["paths"][e]]
        m["goal"][e, :2] = m["paths"][e][-1]
        m["task_paths"][e] = [[sx(q) for q in path] for path in m["task_paths"][e]]
        m["task_goals"][e] = [(*sx(g), 0.0) for g in m["task_goals"][e]]
        m["static_polys"][e] = [[sx(q) for q in poly] for poly in m["static_polys"][e]]
        m["moving_pos"][e] = o + scale * (m["moving_pos"][e] - o)
        m["init"][e, :2] = m["goal"][e, :2] + 0.02
    return m


def _make(m, k=1, dqn_paths=None, **solver):
    mc = t.Configurator()
    fp = t.FleetPlanner(mc, m["init"], m["goal"], m["paths"], mode="work", action_steps=k, **solver)
    fp.update_static_constraints(m["static_polys"], per_robot=True)
    fp.set_moving_obstacles(m["moving_pos"], m["moving_disp"])
    fp.set_tasks(m["task_goals"], m["task_paths"], dqn_paths=dqn_paths)
    tuning, base = work_mode(mc, "work")
    fh = FleetHostK(fp.cfg, m["init"], m["goal"], fp.ref_traj.cpu().numpy(), fp.ref_len.cpu().numpy(),
                    fp.stc.cpu().numpy(), tuning, base, mc.low_speed, dyn_cur=m["moving_pos"],
                    dyn_disp=m["moving_disp"], action_steps=k)
    tq = TaskQueues(m["task_goals"], m["task_paths"], max_nodes=fp.tasks.max_nodes)
    return fp, OracleFleetTasks(fh, fp.cfg, tq)


def _assert_step_equal(fp, of, s):
    fh = of.fh
    assert np.array_equal(fp.p.cpu().numpy(), of.p), f"packed parameters differ at step {s}"
    dev = dict(u=fp.u.cpu().numpy(), y=fp.y.cpu().numpy(), cost=fp.cost.cpu().numpy(),
               exit_status=fp.exit_status.cpu().numpy(), inner=fp.inner.cpu().numpy(),
               pred=fp.pred_states.cpu().numpy())
    for name, ref in of.res.items():
        assert np.array_equal(dev[name], ref), f"{name} differs at step {s}"
    for name in ("state", "last_u", "idx_ref", "status", "goal", "ref_len", "ref_traj", "dyn_cur"):
        assert np.array_equal(getattr(fp, name).cpu().numpy(), getattr(fh, name)), f"{name} differs at step {s}"
    assert np.array_equal(fp.task_next.cpu().numpy(), of.tq.next), f"task cursor differs at step {s}"


@pytest.mark.parametrize("option", list(OPTIONS))
def test_task_closed_loop_bit_exact(option):
    warm, skip = OPTIONS[option]
    fp, of = _make(_short_missions(32, 3, seed=21), **SOLVER)
    for s in range(40):
        fp.step(warm_start=warm, skip_stopped=skip); fp.torch.cuda.synchronize()
        of.step(warm=warm, skip=skip)
        _assert_step_equal(fp, of, s)
    nxt = of.tq.next
    assert (nxt >= 1).all() and (nxt == 2).sum() >= 8, nxt          # every robot switched, many twice
    assert (of.fh.status == RUNNING).sum() >= 1


def test_task_closed_loop_k2_bit_exact():
    fp, of = _make(_short_missions(32, 3, seed=22), k=2, **SOLVER)
    for s in range(40):
        fp.step(warm_start=True, skip_stopped=True); fp.torch.cuda.synchronize()
        of.step(warm=True, skip=True)
        _assert_step_equal(fp, of, s)
    assert (of.tq.next >= 1).all() and (of.tq.next == 2).sum() >= 4, of.tq.next


def test_task_hybrid_loop_with_hint_switch_bit_exact():
    import torch
    m = _short_missions(32, 3, seed=23)
    xy, cnt = t.dqn.pack_paths(m["paths"], max_nodes=3)
    path_xy, path_n = torch.tensor(xy).cuda(), torch.tensor(cnt).cuda()
    fp, of = _make(m, dqn_paths=(path_xy, path_n), **SOLVER)
    fp.enable_hint_switch(m["static_polys"], per_robot=True)
    fh, n = of.fh, fp.n
    fh.sw_state = np.zeros((n, 2), np.int32)
    fh.sw_poly_xy, fh.sw_poly_nv = fp.sw_poly_xy.cpu().numpy(), fp.sw_poly_nv.cpu().numpy()
    fh.use_hint = np.zeros(n, np.int32)
    g = torch.Generator(device="cpu").manual_seed(0)
    seen_on = 0
    for s in range(30):
        agent5 = torch.cat([fp.state, fp.last_u], 1).contiguous()
        act = torch.randint(0, 9, (n,), generator=g, dtype=torch.int32).cuda()
        rl = t.dqn.rl_ref_device(agent5, act)
        fp.set_hint(rl, fp.use_hint)
        fh.hint = rl.cpu().numpy()
        fp.step(); torch.cuda.synchronize()
        of.step()
        assert np.array_equal(fp.use_hint.cpu().numpy(), fh.use_hint), f"switch decision differs at step {s}"
        assert np.array_equal(fp.sw_state.cpu().numpy(), fh.sw_state)
        _assert_step_equal(fp, of, s)
        seen_on += int(fh.use_hint.sum())
    assert seen_on > 0 and (of.tq.next >= 1).all()
    # path_out: every robot's current path, which internal_obs_device reads like an explicit path
    cur = [m["task_paths"][e][of.tq.next[e] - 1] for e in range(n)]
    exy, ecnt = t.dqn.pack_paths(cur, max_nodes=3)
    assert np.array_equal(path_n.cpu().numpy(), ecnt) and np.array_equal(path_xy.cpu().numpy(), exy)
    agent5 = torch.cat([fp.state, fp.last_u], 1).contiguous()
    a, pa = t.dqn.internal_obs_device(agent5, path_xy, path_n)
    b, pb = t.dqn.internal_obs_device(agent5, torch.tensor(exy).cuda(), torch.tensor(ecnt).cuda())
    assert torch.equal(a, b) and torch.equal(pa, pb)


def test_task_one_step_2048_robots_rolled_build():
    """One warm, skip-stopped step of 2048 robots: half are at their goals at rest and switch."""
    n = 2048
    m = t.scenes.make_missions(n, 3, seed=31)
    at_goal = np.arange(n) % 2 == 0
    m["init"][at_goal, :2] = m["goal"][at_goal, :2] + 0.01
    fp, of = _make(m, **SOLVER)
    fp.step(warm_start=True, skip_stopped=True); fp.torch.cuda.synchronize()
    of.step(warm=True, skip=True)
    _assert_step_equal(fp, of, 0)
    assert np.array_equal(of.tq.next, at_goal.astype(np.int32)) and (of.fh.status == RUNNING).all()


def test_zero_counts_equal_fleet_step_device():
    """Queues with every count zero: ttmpc_fleet_step_tasks_device computes what
    ttmpc_fleet_step_device computes, output for output."""
    m = t.scenes.make_missions(64, 3, seed=41)
    m["init"][:8, :2] = m["goal"][:8, :2] + 0.01                      # robots that stop in the first step
    fps = []
    for _ in range(2):
        fp, _of = _make(m, **SOLVER)
        fp.task_count.zero_()
        fps.append(fp)
    fps[1].tasks = None                                                 # the entry point without queues
    for s in range(6):
        for fp in fps:
            fp.step(warm_start=True, skip_stopped=True)
        fps[0].torch.cuda.synchronize()
        for name in ("p", "u", "y", "cost", "exit_status", "inner", "pred_states", "state", "last_u", "idx_ref",
                     "status", "goal", "ref_traj", "ref_len", "dyn_cur"):
            assert fps[0].torch.equal(getattr(fps[0], name), getattr(fps[1], name)), f"{name} at step {s}"
    assert (fps[0].status[:8] == REACHED).all() and not fps[0].task_next.any()


def test_sampled_trajectories_equal_oracle_sampler():
    """>= 1000 seeded paths (2-8 nodes, speeds 0.3-1.5, a third starting exactly on node 0): after the
    switch, ref_traj / ref_len equal the oracle's sampler in device mode."""
    import torch
    rng = np.random.default_rng(5)
    checked = bad = 0
    for speed in (0.3, 0.6, 0.9, 1.2, 1.5):
        n = 220
        paths, init = [], np.zeros((n, 3))
        for e in range(n):
            k = int(rng.integers(2, 9))
            pts = np.cumsum(rng.uniform(-2.0, 2.0, (k, 2)), axis=0) + rng.uniform(10, 30, 2)
            paths.append([tuple(q) for q in pts])
            init[e, :2] = pts[0] if e % 3 == 0 else pts[0] + rng.normal(0.0, 0.03, 2)
            init[e, 2] = rng.uniform(-np.pi, np.pi)
        mc = t.Configurator()
        fp = t.FleetPlanner(mc, init, init, [[tuple(init[e, :2]), tuple(init[e, :2] + 0.01)] for e in range(n)],
                            mode="work", **SOLVER)
        fp.base_speed = speed
        fp.set_tasks([[(*p[-1], 0.0)] for p in paths], [[p] for p in paths])
        fp.step(); torch.cuda.synchronize()
        ref, L, st = fp.ref_traj.cpu().numpy(), fp.ref_len.cpu().numpy(), fp.status.cpu().numpy()
        assert (fp.task_next.cpu().numpy() == 1).all()
        for e in range(n):
            want = R.global_ref_traj(paths[e], init[e, 0], init[e, 1], mc.ts, speed, fp.ref_stride, use_libm=False)
            if want is None:
                assert st[e] == BAD_TASK
                bad += 1
                continue
            assert st[e] != BAD_TASK and L[e] == len(want), e
            assert np.array_equal(ref[e, :L[e]], want), e
            checked += 1
    assert checked >= 1000, (checked, bad)
