"""The k-step fleet step (config.action_steps = k > 1) on the CPU: the k-step form of the fleet
oracle (tests/fleet_action_steps_ref.py) against the single-robot host mirror
``planner.InterfaceMpc``, whose solver is replaced by a recorder that returns prescribed controls
(as tools/gen_golden_fleet.py does with the reference's own Python); and the argument checks of
the C-ABI, which run before any device work."""
import ctypes as C

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.fleet import DYN_OBS_SIZE, work_mode
from tests.fleet_action_steps_ref import FleetHostK, fleet_advance_k, fleet_pack_k, warm_start_k
from tests.fleet_options_ref import warm_start

N_ROBOTS, N_STEPS = 6, 10
STOPS, DRIVES_ON = 4, 5    # robots whose first and last controls straddle the 0.05 goal threshold


class _Sol:
    def __init__(self, u):
        self.solution = list(u); self.cost = 1.25; self.exit_status = "Converged"; self.solve_time_ms = 0.5


class _Recorder:
    """Stands in for the mirror's Solver: records p, returns the next prescribed u."""
    def __init__(self):
        self.p_log, self.u_next = [], None

    def run(self, p, initial_guess=None):
        self.p_log.append(np.array(p, dtype=np.float64))
        return _Sol(self.u_next)


def _est_dyn_obs_positions(last, cur, N):
    """main.py:80-89: N steps of constant-velocity extrapolation, ellipse rx = ry = DYN_OBS_SIZE."""
    dx, dy = cur[0] - last[0], cur[1] - last[1]
    return [[cur[0] + dx * (i + 1), cur[1] + dy * (i + 1), DYN_OBS_SIZE, DYN_OBS_SIZE, 0.0, 1.0] for i in range(N)]


def _fleet():
    fl = t.scenes.make_fleet(N_ROBOTS, seed=5)
    # two robots just outside the 5 cm box around their goals, heading at them: after one step
    # they are inside it
    for e, gap in ((STOPS, 0.08), (DRIVES_ON, 0.0515)):
        gx, gy = fl["goal"][e, :2]
        fl["init"][e] = (gx + gap, gy, np.pi)
        fl["paths"][e] = [(gx + gap, gy), (gx, gy)]
    return fl


def _controls(k, N, steps, seed=3):
    """Prescribed solutions [steps][n][2N].  Robot STOPS has first speed 0.01 and last 0.21 (it
    moves 4.2 cm per step), robot DRIVES_ON the reverse (0.2 cm per step)."""
    rng = np.random.default_rng(seed)
    U = np.stack([rng.uniform(0.2, 1.4, (steps, N_ROBOTS, N)), rng.uniform(-0.4, 0.4, (steps, N_ROBOTS, N))], -1)
    U[:, (STOPS, DRIVES_ON)] = 0.0
    U[:, (STOPS, DRIVES_ON), :k, 0] = 0.21
    U[:, STOPS, 0, 0] = 0.01
    U[:, DRIVES_ON, k - 1, 0] = 0.01
    return U.reshape(steps, N_ROBOTS, 2 * N)


@pytest.mark.parametrize("k", [2, 3])
def test_k_step_oracle_matches_interface_mpc(k):
    mc = t.Configurator()
    mc.action_steps = k
    cfg = mc.to_ttmpc()
    N = cfg.N_hor
    off = t.param_offsets(cfg)
    fl = _fleet()
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", device="cpu", action_steps=k)
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    tuning, base = work_mode(mc, "work")
    fh = FleetHostK(cfg, fl["init"], fl["goal"], fp.ref_traj.numpy(), fp.ref_len.numpy(), fp.stc.numpy(), tuning,
                    base, mc.low_speed, dyn_cur=fl["moving_pos"], dyn_disp=fl["moving_disp"], action_steps=k)
    mirrors, recorders = [], []
    for e in range(N_ROBOTS):
        m = t.InterfaceMpc(mc)
        m._traj_gen.solver = rec = _Recorder()
        m.initialization(fl["init"][e].copy(), fl["goal"][e].copy(), fl["paths"][e], mode="work")
        m.update_static_constraints(fl["static_polys"][e])
        mirrors.append(m); recorders.append(rec)
    obs_last = fl["moving_pos"].copy(); obs_cur = fl["moving_pos"].copy()
    U = _controls(k, N, N_STEPS)
    prev_u = np.zeros((N_ROBOTS, 2 * N))
    reached_at = {}
    for s in range(N_STEPS):
        p = fleet_pack_k(fh, prev_u, use_libm=True)
        for e, m in enumerate(mirrors):
            if e in reached_at:
                continue
            m.update_dynamic_constraints([_est_dyn_obs_positions(obs_last[e, j], obs_cur[e, j], N)
                                          for j in range(len(obs_cur[e]))])
            ref_local, _ = m.get_local_ref_traj()
            recorders[e].u_next = U[s, e]
            n_before = len(recorders[e].p_log)
            ret = m.get_action(ref_local, mode="work")
            assert int(fh.idx_ref[e]) == m._traj_gen.idx_ref, f"idx_ref of robot {e} at step {s}"
            if ret is None:
                reached_at[e] = s
                assert fh.status[e] == 1, f"robot {e} should stop at step {s}"
                continue
            assert fh.status[e] == 0, f"robot {e} should drive on at step {s}"
            gp = recorders[e].p_log[n_before]
            mask = np.ones(len(gp), bool)
            mask[off["vref"]:off["c"]] = False
            assert np.array_equal(p[e][mask], gp[mask]), f"packed vector of robot {e} at step {s}"
            # speed reference: hypot may differ from CPython's by an ulp
            np.testing.assert_allclose(p[e][~mask], gp[~mask], rtol=4e-16, atol=0)
            assert np.array_equal(gp[6:8], U[s - 1, e, 2 * (k - 1):2 * k] if s else np.zeros(2)), "v_init, w_init"
        fleet_advance_k(fh, U[s], np.zeros(N_ROBOTS, np.int32), use_libm=True)
        prev_u = U[s].copy()
        for e, m in enumerate(mirrors):
            np.testing.assert_allclose(fh.state[e], m.state, rtol=0, atol=2e-15, err_msg=f"robot {e} step {s}")
            if e not in reached_at:
                assert np.array_equal(fh.last_u[e], U[s, e, 2 * (k - 1):2 * k])
        obs_last = obs_cur.copy()
        obs_cur = obs_cur + fl["moving_disp"]
        np.testing.assert_array_equal(fh.dyn_cur, obs_cur)
    # the straddling robots: the goal test reads the FIRST control of the previous solution
    assert reached_at.get(STOPS) == 1, reached_at
    assert DRIVES_ON not in reached_at, reached_at
    assert len(reached_at) == 1


@pytest.mark.parametrize("k", [1, 2, 3, 20])
def test_warm_start_shift_by_k(k):
    N = 20
    u = np.arange(3 * 2 * N, dtype=np.float64).reshape(3, 2 * N) + 0.5
    status = np.array([0, 0, 1], np.int32)
    exit_status = np.array([0, 1, 0], np.int32)
    out = warm_start_k(status, u, exit_status, k)
    pairs = u[0].reshape(N, 2)
    expect = np.concatenate([pairs[k:], np.repeat(pairs[-1:], k, axis=0)]).reshape(-1)
    assert np.array_equal(out[0], expect)
    assert not out[1].any() and np.array_equal(out[2], u[2])
    if k == 1:
        assert np.array_equal(out, warm_start(status, u, exit_status))


def _host_call_args(k, n=4):
    """A ttmpc_fleet over host buffers: argument checks return before anything touches them."""
    mc = t.Configurator()
    cfg = mc.to_ttmpc()
    N = cfg.N_hor
    tuning, base = work_mode(mc, "work")
    ref = np.zeros((n, 8, 3))
    fh = FleetHostK(cfg, np.zeros((n, 3)), np.ones((n, 3)), ref, [8] * n, np.zeros(cfg.Nstcobs * cfg.nstcobs),
                    tuning, base, mc.low_speed, action_steps=k)
    bufs = dict(p=np.zeros((n, _lib.load().ttmpc_num_params(C.byref(cfg)))), u=np.zeros((n, 2 * N)),
                es=np.zeros(n, np.int32))
    res = _lib.TtmpcResult(u=bufs["u"].ctypes.data, exit_status=bufs["es"].ctypes.data)
    return cfg, fh, fh.struct(), res, bufs


def test_action_steps_argument_checks():
    lib = _lib.load()
    N = t.Configurator().N_hor
    BAD_ARG, UNSUPPORTED = -2, -4
    for k in (0, -1, N + 1):
        cfg, fh, f, res, b = _host_call_args(k)
        assert lib.ttmpc_fleet_step_device(C.byref(cfg), C.byref(f), b["p"].ctypes.data, 1, C.byref(res), None) == BAD_ARG, k
        assert "action_steps" in lib.ttmpc_last_error().decode()
    for k in (0, 2, N):
        cfg, fh, f, res, b = _host_call_args(k)
        assert lib.ttmpc_fleet_pack_device(C.byref(cfg), C.byref(f), b["p"].ctypes.data, None) == UNSUPPORTED, k
        assert lib.ttmpc_fleet_advance_device(C.byref(cfg), C.byref(f), b["u"].ctypes.data, b["es"].ctypes.data,
                                              None) == UNSUPPORTED, k
    # nothing was written
    assert not b["p"].any() and not fh.status.any() and not fh.state.any()


def test_fleet_planner_pack_and_advance_refuse_k_steps():
    mc = t.Configurator()
    fl = t.scenes.make_fleet(2, seed=1)
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], device="cpu", action_steps=2)
    assert fp._fleet_struct().action_steps == 2
    with pytest.raises(_lib.TtmpcError, match="action_steps"):
        fp.pack(stream=0)
    with pytest.raises(_lib.TtmpcError, match="action_steps"):
        fp.advance(stream=0)
    assert t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], device="cpu")._fleet_struct().action_steps == 1
