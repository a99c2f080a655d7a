"""The k-step fleet step on the GPU (FleetPlanner(action_steps=k).step(...), i.e.
ttmpc_fleet.action_steps = k > 1 in ttmpc_fleet_step_device) against the k-step form of the
WARP-order oracle (tests/fleet_action_steps_ref.py), bit for bit."""
import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.fleet import work_mode
from tests.fleet_action_steps_ref import FleetHostK, OracleFleetK

pytestmark = pytest.mark.gpu

SOLVER = dict(max_inner_iterations=40, max_outer_iterations=3)  # some solves end NotConvergedIterations
ARRIVE_AT = 3      # before this step, robots 0-3 are put next to their goals at rest: they stop there
OPTIONS = dict(none=(False, False), warm=(True, False), skip=(False, True), warm_skip=(True, True))


def _make(n, seed, k, fl=None, **solver):
    mc = t.Configurator()
    fl = fl or t.scenes.make_fleet(n, seed=seed)
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", action_steps=k, **solver)
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    fp.set_moving_obstacles(fl["moving_pos"], fl["moving_disp"])
    tuning, base = work_mode(mc, "work")
    fh = FleetHostK(fp.cfg, fl["init"], fl["goal"], fp.ref_traj.cpu().numpy(), fp.ref_len.cpu().numpy(),
                    fp.stc.cpu().numpy(), tuning, base, mc.low_speed, dyn_cur=fl["moving_pos"],
                    dyn_disp=fl["moving_disp"], action_steps=k)
    return fp, OracleFleetK(fh, fp.cfg)


def _arrive(fp, of, robots=slice(0, 4)):
    """Next to the goal, and at rest: with k > 1 the goal test reads u[0] of the previous solution."""
    fp.state[robots, :2] = fp.goal[robots, :2] + 0.01; fp.u[robots] = 0.0
    of.fh.state[robots, :2] = of.fh.goal[robots, :2] + 0.01; of.res["u"][robots] = 0.0


def _assert_step_equal(fp, of, s):
    fh = of.fh
    assert np.array_equal(fp.p.cpu().numpy(), of.p), f"packed parameters differ at step {s}"
    dev = dict(u=fp.u.cpu().numpy(), y=fp.y.cpu().numpy(), cost=fp.cost.cpu().numpy(),
               exit_status=fp.exit_status.cpu().numpy(), inner=fp.inner.cpu().numpy(),
               pred=fp.pred_states.cpu().numpy())
    for name, ref in of.res.items():
        assert np.array_equal(dev[name], ref), f"{name} differs at step {s}"
    assert np.array_equal(fp.state.cpu().numpy(), fh.state), f"states differ at step {s}"
    assert np.array_equal(fp.last_u.cpu().numpy(), fh.last_u), f"last_u differs at step {s}"
    assert np.array_equal(fp.idx_ref.cpu().numpy(), fh.idx_ref), f"idx_ref differs at step {s}"
    assert np.array_equal(fp.status.cpu().numpy(), fh.status), f"status differs at step {s}"
    assert np.array_equal(fp.dyn_cur.cpu().numpy(), fh.dyn_cur), f"obstacles differ at step {s}"


@pytest.mark.parametrize("option", list(OPTIONS))
@pytest.mark.parametrize("k", [2, 3])
def test_k_step_closed_loop_bit_exact(k, option):
    warm, skip = OPTIONS[option]
    n, steps = 32, 8
    fp, of = _make(n, seed=9, k=k, **SOLVER)
    for s in range(steps):
        if s == ARRIVE_AT:
            _arrive(fp, of)
        fp.step(warm_start=warm, skip_stopped=skip); fp.torch.cuda.synchronize()
        of.step(warm=warm, skip=skip)
        _assert_step_equal(fp, of, s)
    assert (of.fh.status[:4] == 1).all() and (of.fh.status[4:] == 0).sum() > 0
    # last_u is the LAST applied control of the last solve
    run = of.fh.status == 0
    assert np.array_equal(of.fh.last_u[run], of.res["u"][run][:, 2 * (k - 1):2 * k])


def test_k_step_hybrid_loop_with_hint_switch_bit_exact():
    """Hybrid loop at k = 2: the DQN hint from [state, last_u], HintSwitcher in the pack kernel."""
    import torch
    n, k = 48, 2
    fl = t.scenes.make_fleet(n, seed=17)
    for i in range(n):   # the first rectangle of every robot sits on its path: the switch has something to see
        (ax, ay), (bx, by) = fl["paths"][i][0], fl["paths"][i][1]
        cx, cy = ax + 0.35 * (bx - ax), ay + 0.35 * (by - ay)
        fl["static_polys"][i][0] = [(cx - 0.6, cy - 0.6), (cx + 0.6, cy - 0.6), (cx + 0.6, cy + 0.6), (cx - 0.6, cy + 0.6)]
    fp, of = _make(n, seed=None, k=k, fl=fl, **SOLVER)
    fp.enable_hint_switch(fl["static_polys"], per_robot=True)
    fh = of.fh
    fh.sw_state = np.zeros((n, 2), np.int32)
    fh.sw_poly_xy, fh.sw_poly_nv = fp.sw_poly_xy.cpu().numpy(), fp.sw_poly_nv.cpu().numpy()
    fh.use_hint = np.zeros(n, np.int32)
    g = torch.Generator(device="cpu").manual_seed(0)
    seen_on = 0
    for s in range(5):
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
    assert seen_on > 0


def test_k_step_one_step_2048_robots_rolled_build():
    """One warm, skip-stopped step of 2048 robots at k = 2 from a prescribed previous solution.
    2048 robots exceed the resident warps: the rolled build with the dispatch order.  A quarter of
    the robots sit at their goals, half of those with a first control below the 0.05 threshold and a
    last one above it (they stop), half the other way round (they drive on)."""
    n, k = 2048, 2
    fp, of = _make(n, seed=12, k=k, **SOLVER)
    rng = np.random.default_rng(4)
    N = fp.N
    u = np.stack([rng.uniform(-0.5, 1.5, (n, N)), rng.uniform(-0.5, 0.5, (n, N))], -1).reshape(n, 2 * N)
    at_goal = np.arange(n) % 4 == 0
    stops = at_goal & (np.arange(n) % 8 == 0)
    drives_on = at_goal & ~stops
    u[stops, 0], u[stops, 2 * (k - 1)] = 0.01, 0.3
    u[drives_on, 0], u[drives_on, 2 * (k - 1)] = 0.3, 0.01
    exit_status = rng.integers(0, 2, n).astype(np.int32)
    last_u = u[:, 2 * (k - 1):2 * k].copy()
    state = of.fh.state.copy()
    state[at_goal, :2] = of.fh.goal[at_goal, :2] + 0.01
    for a, b in ((fp.u, u), (fp.exit_status, exit_status), (fp.last_u, last_u), (fp.state, state)):
        a.copy_(fp.torch.from_numpy(b))
    of.res["u"][:], of.res["exit_status"][:] = u, exit_status
    of.fh.last_u[:], of.fh.state[:] = last_u, state
    fp.step(warm_start=True, skip_stopped=True); fp.torch.cuda.synchronize()
    of.step(warm=True, skip=True)
    _assert_step_equal(fp, of, 0)
    assert (of.fh.status[stops] == 1).all() and (of.fh.status[drives_on] == 0).all()
    assert (of.fh.status[~at_goal] == 0).all()
    # skipped robots keep their previous rows: the prescribed solution, unshifted
    assert np.array_equal(fp.u.cpu().numpy()[stops], u[stops])
