"""Shared obstacle map on the GPU (ttmpc_fleet_world_select_device, FleetPlanner.set_world): the kernel
against the brute-force oracle of tests/fleet_world_ref.py bit for bit, and closed loops with a map
against the same loops with update_static_constraints or with the selection done on the host."""
import ctypes as C
import zlib

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.geometry import convex_hull
from tests.fleet_world_ref import WorldHost, distance
from tests.test_fleet_world import _quad, _random_quads, _world

pytestmark = pytest.mark.gpu

SOLVER = dict(max_inner_iterations=40, max_outer_iterations=3)
OPTIONS = dict(none=(False, False), warm=(True, False), skip=(False, True), warm_skip=(True, True))
RESULTS = ("p", "u", "y", "cost", "exit_status", "inner", "pred_states")
FLEET = ("state", "last_u", "idx_ref", "status", "goal", "ref_traj", "ref_len")


# ------------------------------------------------------------------ the kernel against the oracle
def _run_kernel(wh, cfg, state):
    import torch
    n, K = len(state), cfg.Nstcobs
    dev = {k: torch.from_numpy(np.ascontiguousarray(getattr(wh, k))).cuda()
           for k in ("poly_xy", "poly_nv", "rows", "bbox", "cell_start", "cell_items")}
    by_id = {id(getattr(wh, k)): v.data_ptr() for k, v in dev.items()}
    st = torch.from_numpy(np.ascontiguousarray(state)).cuda()
    f = _lib.TtmpcFleet()
    f.n, f.ref_stride, f.action_steps = n, 1, 1
    for name in ("state", "goal", "last_u", "idx_ref", "status", "ref_traj", "ref_len", "stc"):
        setattr(f, name, st.data_ptr())                 # only n and state are read; the others must be set
    stc = torch.full((n, K * cfg.nstcobs), np.nan, dtype=torch.float64, device="cuda")
    slots = torch.full((n, K), -7, dtype=torch.int32, device="cuda")
    reach = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    w = wh.struct(ptr=lambda a: by_id[id(a)])
    _lib.check(_lib.load().ttmpc_fleet_world_select_device(C.byref(cfg), C.byref(f), C.byref(w), stc.data_ptr(),
                                                           slots.data_ptr(), reach.data_ptr(),
                                                           torch.cuda.current_stream().cuda_stream), "world select")
    torch.cuda.synchronize()
    return stc.cpu().numpy(), slots.cpu().numpy(), reach.cpu().numpy()


def _cfg(K=10):
    cfg = t.Configurator().to_ttmpc()
    cfg.Nstcobs = K
    return cfg


def _robots(rng, n, lo, hi):
    s = np.zeros((n, 3))
    s[:, :2] = rng.uniform(lo, hi, (n, 2))
    s[:, 2] = rng.uniform(-np.pi, np.pi, n)
    return s


def _case(name):
    """(WorldHost, cfg, state [2048][3]) of one named case."""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    n = 2048
    if name == "empty":
        return _world([], 6.0), _cfg(), _robots(rng, n, -10, 10)
    if name == "few":                                                  # M < K
        return _world(_random_quads(rng, 5, 3.0), 6.0), _cfg(), _robots(rng, n, -12, 12)
    if name.startswith("random"):                                      # M up to 2e4, robots inside and outside the grid
        M, K, cell = dict(random2k=(2000, 10, None), random20k=(20_000, 10, None), random20k_k32=(20_000, 32, 2.0),
                          random5k_k4=(5000, 4, 12.0))[name]
        polys = _random_quads(rng, M, 150.0)
        return _world(polys, 6.0, cell), _cfg(K), _robots(rng, n, -170, 170)
    if name == "dense_cell":                                           # >= 1000 candidates in one cell
        polys = [_quad(x, y, 0.05, 0.05) for x, y in rng.uniform(-0.9, 0.9, (1500, 2))]
        polys += _random_quads(rng, 500, 20.0)
        wh = _world(polys, 6.0, cell=6.0)
        counts = np.diff(wh.cell_start)
        assert counts.max() >= 1000, counts.max()
        return wh, _cfg(), _robots(rng, n, -8, 8)
    if name == "ties_exact_reach":
        R = 2.0
        polys = []
        for cx in range(-10, 11, 5):                                   # stacks of identical squares: d ties everywhere
            for cy in range(-10, 11, 5):
                polys += [_quad(cx, cy, 0.5, 0.5)] * 3 + [_quad(cx + R + 1.0, cy, 0.5, 0.5)]
        wh = _world(polys, R, cell=1.0)
        s = np.zeros((n, 3))
        s[:, :2] = rng.integers(-10, 11, (n, 2)).astype(np.float64) * 0.5   # centres, edges, cell corners
        k = n // 4                                                     # exactly R from the right square's left edge
        s[:k, 0] = rng.choice(np.arange(-10, 11, 5), k) + 0.5
        s[:k, 1] = rng.choice(np.arange(-10, 11, 5), k)
        assert sum(distance(wh.poly_xy[o], *s[0, :2]) == R for o in range(wh.M)) >= 1
        return wh, _cfg(4), s
    raise KeyError(name)


@pytest.mark.parametrize("name", ["empty", "few", "random2k", "random20k", "random20k_k32", "random5k_k4",
                                  "dense_cell", "ties_exact_reach"])
def test_world_select_kernel_equals_oracle(name):
    wh, cfg, state = _case(name)
    stc, slots, reach = _run_kernel(wh, cfg, state)
    ref = wh.select(cfg, state)
    assert np.array_equal(slots, ref[1]), f"slot_poly differs for {int((slots != ref[1]).any(1).sum())} robots"
    assert np.array_equal(reach, ref[2]), "n_reach differs"
    assert np.array_equal(stc, ref[0]), "stc_out differs"
    K = cfg.Nstcobs
    if wh.M:
        assert (reach > 0).sum() > 100
    if name in ("random20k", "dense_cell", "ties_exact_reach"):
        assert (reach > K).sum() > 50                                   # slots overflowed: the ranking decided
    if name == "dense_cell":
        assert reach.max() >= 1000
    if name.startswith("random20k"):
        assert (reach == 0).sum() > 50                                   # robots far from everything / off the grid


# ------------------------------------------------------------------ closed loops
def _missions(n, seed, k=1, tasks=True):
    mc = t.Configurator()
    m = t.scenes.make_missions(n, 3, seed=seed)
    polys = [m["static_polys"][e][0] for e in range(10)]               # 10 rectangles shared by everyone

    def make():
        fp = t.FleetPlanner(mc, m["init"], m["goal"], m["paths"], mode="work", action_steps=k, **SOLVER)
        fp.set_moving_obstacles(m["moving_pos"], m["moving_disp"])
        if tasks:
            fp.set_tasks(m["task_goals"], m["task_paths"])
        return fp
    return make, polys


def _same(a, b, s, names):
    import torch
    for name in names:
        x, y = getattr(a, name), getattr(b, name)
        assert torch.equal(x, y), f"{name} differs at step {s}"


@pytest.mark.parametrize("case", list(OPTIONS) + ["k2", "tasks_warm_skip"])
def test_small_map_equals_update_static_constraints(case):
    """A map of Nstcobs polygons, all within reach: 40 steps bit-identical to the same polygons given
    to update_static_constraints as one shared block."""
    import torch
    warm, skip = OPTIONS.get(case, (True, True))
    make, polys = _missions(32, seed=61, k=2 if case == "k2" else 1, tasks=case == "tasks_warm_skip")
    a, b = make(), make()
    a.set_world(polys, reach=1e3)
    b.update_static_constraints(polys)
    for s in range(40):
        for fp in (a, b):
            fp.step(warm_start=warm, skip_stopped=skip)
        torch.cuda.synchronize()
        _same(a, b, s, RESULTS + FLEET + ("dyn_cur", "dyn_last"))
        assert torch.equal(a.stc, b.stc.expand_as(a.stc)), f"stc differs at step {s}"
        assert (a.world_reach == 10).all() and (a.world_slots == torch.arange(10, device="cuda", dtype=torch.int32)).all()
        if case == "tasks_warm_skip":
            _same(a, b, s, ("task_next",))
    assert int((a.idx_ref > 20).sum()) == a.n                          # every robot drove along its path


def test_warehouse_equals_host_selection_loop():
    """make_warehouse map (M >> Nstcobs), task queues and the monitor on the map: 40 steps equal a loop
    that copies the states to the host, selects with the oracle, writes a per-robot stc and calls the
    unchanged step."""
    import torch
    mc = t.Configurator()
    w = t.scenes.make_warehouse(64, 3, seed=62, shelves=2000, aisle=2.6)
    hulls = [convex_hull(np.array(p)) for p in w["world_polys"]]

    def make():
        fp = t.FleetPlanner(mc, w["init"], w["goal"], w["paths"], mode="work", **SOLVER)
        fp.set_tasks(w["task_goals"], w["task_paths"])
        return fp
    a, b = make(), make()
    a.set_world(w["world_polys"])
    a.enable_monitor(robot_radius=0.2)
    b.enable_monitor(polygons=hulls, robot_radius=0.2)
    wh = WorldHost.from_planner(a)
    assert wh.M == len(w["world_polys"]) >= 2000
    for s in range(40):
        stc, slots, reach = wh.select(a.cfg, b.state.cpu().numpy())
        b.stc, b.stc_shared = torch.from_numpy(stc).cuda(), 0
        a.step(warm_start=True, skip_stopped=True)
        b.step(warm_start=True, skip_stopped=True)
        torch.cuda.synchronize()
        assert np.array_equal(a.world_slots.cpu().numpy(), slots) and np.array_equal(a.world_reach.cpu().numpy(), reach)
        assert torch.equal(a.stc, b.stc), f"stc differs at step {s}"
        _same(a, b, s, RESULTS + FLEET + ("task_next", "clearance", "min_clearance", "contact_steps", "first_contact",
                                          "deviation_max", "deviation_sum", "moved_steps"))
    assert int(a.task_next.sum()) > 0 and int(a.moved_steps.sum()) > 0
    assert int(a.world_reach.max()) > 0, "no shelf within reach"
