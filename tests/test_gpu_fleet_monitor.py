"""Obstacle-contact and tracking monitor on the GPU (FleetPlanner.enable_monitor ->
ttmpc_fleet_monitor_device) against the oracle of tests/fleet_monitor_ref.py, bit for bit: on random
robots through the C entry point, and after every step of closed loops composed from the
WARP-order fleet oracles."""
import ctypes as C

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.fleet import COLLIDED, DYN_OBS_SIZE, RUNNING, work_mode
from tests.fleet_action_steps_ref import FleetHostK, OracleFleetK
from tests.fleet_monitor_ref import BUFFERS, MonitorHost
from tests.test_gpu_fleet_tasks import _make as _make_tasks, _short_missions

pytestmark = pytest.mark.gpu

SOLVER = dict(max_inner_iterations=40, max_outer_iterations=3)
OPTIONS = dict(none=(False, False), warm=(True, False), skip=(False, True), warm_skip=(True, True))
FLEET = ("state", "last_u", "idx_ref", "status", "goal", "ref_len", "ref_traj", "dyn_cur", "dyn_last")


# ------------------------------------------------------------------ the entry point on random robots
def _random_robots(rng, n, shared, n_dyn, k, stride=30):
    mc = t.Configurator()
    cfg = mc.to_ttmpc()
    tuning, base = work_mode(mc, "work")
    centre = rng.uniform(-20, 20, (n, 2))
    P, V = 5, 8
    rows = 1 if shared else n
    xy = np.zeros((rows, P, V, 2)); nv = np.zeros((rows, P), np.int32)
    for r in range(rows):
        c = np.zeros(2) if shared else centre[r]
        for j in range(P):
            m = int(rng.choice([0, 2, 3, 4, 5, 6, 7, 8]))            # 0 and 2: unused slots
            ang = np.sort(rng.uniform(0, 2 * np.pi, V))
            rad = rng.uniform(0.2, 1.2, V) * (1.0 if rng.uniform() < 0.5 else rng.uniform(0.3, 1.0, V))  # non-convex rings
            xy[r, j] = c + rng.uniform(-2, 2, 2) + np.stack([rad * np.cos(ang), rad * np.sin(ang)], 1)
            nv[r, j] = m
    if shared:
        centre = rng.uniform(-3, 3, (n, 2))
    start = centre + rng.uniform(-2.5, 2.5, (n, 2))
    ref = np.zeros((n, stride, 3)); ref[:, :, :2] = start[:, None] + np.cumsum(rng.normal(0, 0.2, (n, stride, 2)), 1)
    ref_len = rng.integers(1, stride + 1, n).astype(np.int32)
    state = np.zeros((n, 3)); state[:, :2] = start
    dyn = None
    if n_dyn:
        dyn = start[:, None] + rng.uniform(-3, 3, (n, n_dyn, 2))
    fh = FleetHostK(cfg, state, np.zeros((n, 3)), ref, ref_len, np.zeros(cfg.Nstcobs * cfg.nstcobs), tuning, base,
                    mc.low_speed, dyn_cur=dyn, dyn_disp=None if dyn is None else np.zeros_like(dyn), action_steps=k)
    fh.idx_ref[:] = (rng.uniform(0, 1, n) * ref_len).astype(np.int32)
    return fh, xy, nv


def _move(rng, fh):
    """The next step: robots move by up to 0.4 m (a fifth not at all), obstacles by up to 0.5 m, some
    robots change status."""
    n = fh.n
    d = rng.uniform(-0.4, 0.4, (n, 2)) * (rng.uniform(0, 1, (n, 1)) > 0.2)
    fh.state[:, :2] += d
    if fh.dyn_cur is not None:
        fh.dyn_last[:] = fh.dyn_cur
        fh.dyn_cur += rng.uniform(-0.5, 0.5, fh.dyn_cur.shape)
    flip = rng.uniform(0, 1, n) < 0.1
    fh.status[flip] = rng.integers(0, 5, int(flip.sum()))


@pytest.mark.parametrize("case", [
    dict(shared=True, n_dyn=0, k=1, robot_radius=0.0, moving_radius=1.6, stop=False),
    dict(shared=False, n_dyn=3, k=2, robot_radius=0.3, moving_radius=0.5, stop=True),
    dict(shared=False, n_dyn=0, k=3, robot_radius=0.0, moving_radius=0.0, stop=True),
    dict(shared=None, n_dyn=4, k=1, robot_radius=0.2, moving_radius=0.0, stop=False),   # no polygons
])
def test_monitor_kernel_equals_oracle_on_random_robots(case):
    import torch
    rng = np.random.default_rng(7)
    n = 1200
    fh, xy, nv = _random_robots(rng, n, bool(case["shared"]), case["n_dyn"], case["k"])
    fh.status[:] = np.where(rng.uniform(0, 1, n) < 0.7, RUNNING, rng.integers(1, 5, n))
    polys = case["shared"] is not None
    mh = MonitorHost(fh.state, xy if polys else None, nv if polys else None, case["robot_radius"],
                     case["moving_radius"], case["stop"])
    names = ["state", "goal", "last_u", "idx_ref", "status", "ref_traj", "ref_len", "stc", "dyn_cur", "dyn_last",
             "dyn_disp"]
    dev = {}
    for name in names + ["mon_" + b for b in BUFFERS] + ["poly_xy", "poly_nv"]:
        a = getattr(mh, name[4:]) if name.startswith("mon_") else getattr(mh if name.startswith("poly") else fh, name)
        if a is not None:
            dev[name] = (a, torch.from_numpy(np.ascontiguousarray(a)).cuda())
    by_id = {id(a): d.data_ptr() for a, d in dev.values()}
    lib = _lib.load()
    contacts = collided = 0
    for s in range(3):
        if s:
            _move(rng, fh)
            for name in ("state", "status", "dyn_cur", "dyn_last"):
                if name in dev:
                    dev[name][1].copy_(torch.from_numpy(getattr(fh, name)))
        f = fh.struct()
        for name in names:
            if name in dev:
                setattr(f, name, dev[name][1].data_ptr())
        m = mh.struct(step=10 + s, ptr=lambda a: by_id[id(a)])
        _lib.check(lib.ttmpc_fleet_monitor_device(C.byref(fh.cfg), C.byref(f), C.byref(m),
                                                  torch.cuda.current_stream().cuda_stream), "monitor")
        torch.cuda.synchronize()
        mh.run(fh, step=10 + s)
        for b in BUFFERS:
            assert np.array_equal(dev["mon_" + b][1].cpu().numpy(), getattr(mh, b)), f"{b} differs at call {s}"
        assert np.array_equal(dev["status"][1].cpu().numpy(), fh.status), f"status differs at call {s}"
        contacts += int((mh.clearance <= 0).sum())
        collided += int((fh.status == COLLIDED).sum())
    assert contacts > 50 and (mh.clearance > 0).sum() > 50, contacts            # both sides of the test drawn
    assert (mh.moved_steps > 0).sum() > n // 2 and not mh.deviation_max[mh.moved_steps == 0].any()
    if case["stop"]:
        assert collided > 0


# ------------------------------------------------------------------ closed loops
def _make_fleet(n, seed, k=1, robot_radius=0.3, stop=False):
    mc = t.Configurator()
    fl = t.scenes.make_fleet(n, seed=seed)
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", action_steps=k, **SOLVER)
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    fp.set_moving_obstacles(fl["moving_pos"], fl["moving_disp"])
    fp.enable_monitor(robot_radius=robot_radius, stop_on_contact=stop)
    tuning, base = work_mode(mc, "work")
    fh = FleetHostK(fp.cfg, fl["init"], fl["goal"], fp.ref_traj.cpu().numpy(), fp.ref_len.cpu().numpy(),
                    fp.stc.cpu().numpy(), tuning, base, mc.low_speed, dyn_cur=fl["moving_pos"],
                    dyn_disp=fl["moving_disp"], action_steps=k)
    return fp, OracleFleetK(fh, fp.cfg), _monitor_host(fp, robot_radius, stop)


def _monitor_host(fp, robot_radius, stop, moving_radius=DYN_OBS_SIZE):
    return MonitorHost(fp.state.cpu().numpy(), fp.mon_poly_xy.cpu().numpy(), fp.mon_poly_nv.cpu().numpy(),
                       robot_radius, moving_radius, stop)


def _assert_equal(fp, of, mh, s):
    fh = of.fh
    assert np.array_equal(fp.p.cpu().numpy(), of.p), f"packed parameters differ at step {s}"
    dev = dict(u=fp.u, y=fp.y, cost=fp.cost, exit_status=fp.exit_status, inner=fp.inner, pred=fp.pred_states)
    for name, ref in of.res.items():
        assert np.array_equal(dev[name].cpu().numpy(), ref), f"{name} differs at step {s}"
    for name in FLEET:
        assert np.array_equal(getattr(fp, name).cpu().numpy(), getattr(fh, name)), f"{name} differs at step {s}"
    for name in BUFFERS:
        assert np.array_equal(getattr(fp, name).cpu().numpy(), getattr(mh, name)), f"{name} differs at step {s}"


def _drive(fp, of, mh, steps, warm, skip, each=None):
    import torch
    for s in range(steps):
        fp.step(warm_start=warm, skip_stopped=skip); torch.cuda.synchronize()
        of.step(warm=warm, skip=skip)
        mh.run(of.fh, s)
        _assert_equal(fp, of, mh, s)
        if each:
            each(s)


@pytest.mark.parametrize("option", list(OPTIONS))
def test_monitor_closed_loop_bit_exact(option):
    warm, skip = OPTIONS[option]
    fp, of, mh = _make_fleet(32, seed=51)
    _drive(fp, of, mh, 40, warm, skip)
    assert (mh.moved_steps == 40).sum() >= 16 and (mh.contact_steps > 0).any(), mh.contact_steps


def test_monitor_closed_loop_k2_stop_on_contact_bit_exact():
    fp, of, mh = _make_fleet(32, seed=52, k=2, robot_radius=0.5, stop=True)
    _drive(fp, of, mh, 40, True, True)
    assert 1 <= (of.fh.status == COLLIDED).sum() < 32


def test_stop_on_contact_freezes_robots_with_task_queues():
    """Robots in contact become COLLIDED in the step of their first contact; from then on their
    state, last_u, idx_ref, task cursor and (skip-stopped) result rows stay as they were."""
    m = _short_missions(32, 3, seed=53)
    fp, of = _make_tasks(m, **SOLVER)
    # the missions are shrunk to 0.15 of their size: so are the moving obstacles' discs
    fp.enable_monitor(moving_radius=0.15 * DYN_OBS_SIZE, stop_on_contact=True)
    mh = _monitor_host(fp, 0.0, True, moving_radius=0.15 * DYN_OBS_SIZE)
    frozen = {}
    res_names = dict(u=fp.u, y=fp.y, cost=fp.cost, exit_status=fp.exit_status, inner=fp.inner, pred=fp.pred_states)

    def each(s):
        st = fp.status.cpu().numpy()
        fc = fp.first_contact.cpu().numpy()
        snap = dict(state=fp.state, last_u=fp.last_u, idx_ref=fp.idx_ref, task_next=fp.task_next, **res_names)
        snap = {k: v.cpu().numpy() for k, v in snap.items()}
        for e in np.flatnonzero(st == COLLIDED):
            if e not in frozen:
                assert fc[e] == s, (e, fc[e], s)           # stopped in the step of its first contact
                frozen[e] = {k: v[e].copy() for k, v in snap.items()}
            for k, v in frozen[e].items():
                assert np.array_equal(snap[k][e], v), (e, k, s)
        assert np.array_equal(fp.task_next.cpu().numpy(), of.tq.next)

    _drive(fp, of, mh, 40, True, True, each)
    assert 1 <= len(frozen) < 32 and (of.tq.next >= 1).all(), (len(frozen), of.tq.next)


def test_monitor_without_stop_changes_nothing():
    """40 steps with the monitor on (stop_on_contact off) leave every fleet tensor and every result
    array bit-identical to the same run without the monitor."""
    import torch
    m = t.scenes.make_missions(64, 3, seed=54)
    m["init"][:8, :2] = m["goal"][:8, :2] + 0.01                     # robots that switch tasks at once
    fps = [_make_tasks(m, **SOLVER)[0] for _ in range(2)]
    fps[0].enable_monitor(robot_radius=0.3)
    names = ("p", "u", "y", "cost", "exit_status", "inner", "pred_states", "state", "last_u", "idx_ref", "status",
             "goal", "ref_traj", "ref_len", "dyn_cur", "dyn_last", "task_next")
    for s in range(40):
        for fp in fps:
            fp.step(warm_start=True, skip_stopped=True)
        torch.cuda.synchronize()
        for name in names:
            assert torch.equal(getattr(fps[0], name), getattr(fps[1], name)), f"{name} at step {s}"
    assert int(fps[0].contact_steps.sum()) > 0 and int(fps[0].moved_steps.sum()) > 0
