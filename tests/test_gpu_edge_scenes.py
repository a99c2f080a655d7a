"""GPU tests (-m gpu) of the solve and evaluation kernels on scene content scenes.make_scenes never
produces (tests/edge_scenes.py): other robots, static polygons of 3-8 edges in scattered slots,
dynamic obstacles in scattered slots up to 63, horizons 1-31, coordinates up to 1e5 m, rollouts that
leave the live box, and NaN / inf inputs.

Every solve is compared bit for bit with the WARP-order oracle, every evaluation bit for bit with
O.eval_warp and within a stated bound with the long-double reference edge_scenes.ref_eval.  Each test
also asserts that the content it adds changed something, so that none passes without testing it."""
import dataclasses
import os

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.mpc_config import param_offsets
from tests import edge_scenes as E
from tests import oracle_lib as O

pytestmark = pytest.mark.gpu
THREADS = os.cpu_count() or 1
CTRL_TOL, COST_RTOL = 1e-4, 1e-6
EPS = 2.0 ** -53


def assert_parity(sol, ref):
    assert np.array_equal(sol.exit_status, ref["exit_status"])
    assert np.abs(sol.solution - ref["u"]).max() <= CTRL_TOL
    assert np.all(np.abs(sol.cost - ref["cost"]) <= COST_RTOL * np.maximum(1.0, np.abs(ref["cost"])))
    # and in fact bit for bit
    assert np.array_equal(sol.solution, ref["u"])
    assert np.array_equal(sol.cost, ref["cost"])
    assert np.array_equal(sol.lagrange_multipliers, ref["y"])
    assert np.array_equal(sol.num_inner_iterations, ref["inner"])
    assert np.array_equal(sol.num_outer_iterations, ref["outer"])
    assert np.array_equal(sol.penalty, ref["pen"])
    assert np.array_equal(sol.f2_norm, ref["f2"])
    assert np.array_equal(sol.f1_infeasibility, ref["f1"])
    assert np.array_equal(sol.last_problem_norm_fpr, ref["fpr"])
    assert np.array_equal(sol.pred_states, ref["pred"])


def solve_parity(cfg, p, **kw):
    """GPU solve, checked bit for bit against the WARP-order oracle; returns the GPU solution."""
    sol = t.BatchSolver(cfg).run(p, **kw)
    ref = O.solve_batch(cfg, p, u0=kw.get("initial_guess"), threads=THREADS, warp=True)
    assert_parity(sol, ref)
    return sol


def changed(cfg, p, sol, block):
    """Fraction of scenes whose solution changes when the named parameter block is zeroed."""
    o = param_offsets(cfg)
    lo, hi = {"c": (o["c"], o["os"]), "os": (o["os"], o["od"]), "od": (o["od"], o["qstc"])}[block]
    q = p.copy()
    q[:, lo:hi] = 0.0
    other = t.BatchSolver(cfg).run(q)
    return float((sol.solution != other.solution).any(1).mean())


def controls(rng, cfg, n, scale=1.0):
    u = np.empty((n, 2 * cfg.N_hor))
    u[:, 0::2] = scale * rng.uniform(cfg.lin_vel_min, cfg.lin_vel_max, (n, cfg.N_hor))
    u[:, 1::2] = scale * rng.uniform(-cfg.ang_vel_max, cfg.ang_vel_max, (n, cfg.N_hor))
    return u


def robot_kinds(n_other):
    kinds = [E.ROBOT_KINDS[j % len(E.ROBOT_KINDS)] for j in range(n_other)]
    if n_other > 1:
        kinds[-1] = "crossing"      # the highest bit of the mask carries a robot that meets the path
    return kinds


def dyn_slots(rng, n, ndyn, lo=6, hi=12):
    """Per scene 6-12 live slots scattered over the range; half the scenes hold 31, 32, 63 and the last slot."""
    out = []
    for i in range(n):
        k = min(int(rng.integers(lo, hi + 1)), ndyn)
        must = sorted({s for s in (31, 32, 63, ndyn - 1) if s < ndyn}) if i % 2 == 0 else []
        rest = [s for s in rng.permutation(ndyn) if s not in must][:max(k - len(must), 0)]
        out.append(sorted(must + rest)[:max(k, len(must))])
    return out


def rich_scenes(cfg, n, seed):
    """Every kind of content at once: other robots, scattered static polygons, scattered dynamic
    obstacles, and (from N = 4 on) a folded reference path in every other scene."""
    rng = np.random.default_rng(seed)
    ne = cfg.nstcobs // 3
    p = t.scenes.make_scenes(n, cfg, seed=seed, n_static=0, n_dynamic=0)
    if cfg.N_hor >= 4:
        E.with_folded_reference(p[1::2], cfg)
    if cfg.Nother:
        E.with_other_robots(p, cfg, rng, robot_kinds(cfg.Nother))
    if cfg.Nstcobs:
        slots = sorted({1, cfg.Nstcobs - 1} | set(range(2, cfg.Nstcobs - 1, max(2, cfg.Nstcobs // 4))))
        E.with_static_polygons(p, cfg, rng, ne, slots[:6])
    if cfg.Ndynobs:
        E.with_dynamic_obstacles(p, cfg, rng, dyn_slots(rng, n, cfg.Ndynobs), boundary=(0, 1))
    return p


def eval_checks(cfg, p, u, c=None, y=None):
    """solver.evaluate against O.eval_warp (bit for bit) and against ref_eval.  The bound against the
    long double reference: the kernel forms positions X = x0 + (prefix sum of steps) in fp64, so each
    rolled-out position carries a rounding error up to eps |X| <= eps R (R = largest coordinate of the
    scene and its rollout, eps = 2^-53); centres and path points are exact inputs and their
    differences with nearby positions are exact (Sterbenz).  A term's error is then at most its
    position gradient times the position error: |df| <= 4 eps R lip_f (lip_f = sum over steps of
    |d f / d position|, computed by ref_eval; the 4 covers both coordinates and the roundings of the
    differences), plus 1e-12 relative for the operation order.  The same for F2 with lip_F2."""
    n, N = len(p), cfg.N_hor
    ev = t.BatchSolver(cfg).evaluate(p, u, c, y)
    for i in range(n):
        f, F2, ps, gr = O.eval_warp(cfg, u[i], p[i], 0.0 if c is None else c[i], None if y is None else y[i])
        assert f == ev["f"][i] and ps == ev["psi"][i], i
        assert np.array_equal(F2, ev["F2"][i]) and np.array_equal(gr, ev["grad"][i]), i
    f, F1, F2, parts = E.ref_eval(cfg, u, p, terms=True)
    xy = E.rollouts(cfg, u, p)
    R = np.maximum(np.abs(p[:, :2]).max(1), np.abs(xy).max((1, 2)))
    bf = 4 * EPS * R * np.asarray(parts["lip_f"], np.float64) + 1e-12 * np.maximum(1.0, np.abs(np.asarray(f, np.float64)))
    df = np.abs(ev["f"] - np.asarray(f, np.float64))
    print(f"f vs long double: max |df| {df.max():.3e}, max |df| / bound {(df / bf).max():.3f}")
    assert (df <= bf).all()
    assert np.abs(ev["F1"] - np.asarray(F1, np.float64)).max() <= 1e-12 * max(1.0, float(np.abs(ev["F1"]).max()))
    if cfg.Ndynobs:
        b2 = 4 * EPS * R[:, None] * np.asarray(parts["lip_F2"], np.float64) + \
            1e-12 * np.maximum(1.0, np.abs(np.asarray(F2, np.float64)).max(1, keepdims=True))
        d2 = np.abs(ev["F2"] - np.asarray(F2, np.float64))
        print(f"F2 vs long double: max |dF2| {d2.max():.3e}, max |dF2| / bound {(d2 / b2).max():.3f}")
        assert (d2 <= b2).all()
    return ev, parts


# ------------------------------------------------------------------ 1. other robots
@pytest.mark.parametrize("code", ["small", "unrolled"])
def test_other_robots_default_shape(cfg, monkeypatch, code):
    """The specialised Dims<20,10,10,4,15,10> kernel with every kind of other robot, both builds."""
    monkeypatch.setenv("TTMPC_CODE", code)
    rng = np.random.default_rng(101)
    p = t.scenes.make_scenes(128, cfg, seed=101, n_static=4, n_dynamic=3, blocking_fraction=0.2)
    E.with_other_robots(p, cfg, rng, ["headon", "crossing", "parallel", "parked_in", "parked_out",
                                      "headon", "crossing", "empty", "parked_in", "crossing"])
    sol = solve_parity(cfg, p)
    assert changed(cfg, p, sol, "c") >= 0.5
    parts = E.ref_eval(cfg, sol.solution, p, terms=True)[3]
    assert (parts["contacts"] > 0).mean() >= 0.25


@pytest.mark.parametrize("n_other", [1, 31, 32])
def test_other_robots_runtime_shapes(n_other):
    mc = t.Configurator(Nother=n_other)
    c = mc.to_ttmpc()
    rng = np.random.default_rng(110 + n_other)
    p = t.scenes.make_scenes(48, c, seed=110 + n_other, n_static=3, n_dynamic=2, mpc=mc)
    E.with_other_robots(p, c, rng, ["headon"] if n_other == 1 else robot_kinds(n_other))
    sol = solve_parity(c, p)
    assert changed(c, p, sol, "c") >= 0.5
    # the last slot's robot meets the rollout of the solution in some scenes
    parts = E.ref_eval(c, sol.solution, p, terms=True)[3]
    assert (parts["robot_contacts"][:, -1] > 0).sum() >= 3


# ------------------------------------------------------------------ 2. dynamic-obstacle slots
@pytest.mark.parametrize("ndyn", [15, 32, 33, 64])
def test_dynamic_obstacle_slots(ndyn):
    """6-12 live obstacles per scene in scattered slots (31, 32, 63 included): the 32 / 64-bit live
    mask, the popcount slot arithmetic, shared-memory rows (the first DYN_SLOTS live ones) and
    global-scratch rows (the rest).  Slots 0 and 1 are parked at the live box's edge when drawn."""
    mc = t.Configurator(Ndynobs=ndyn)
    c = mc.to_ttmpc()
    rng = np.random.default_rng(120 + ndyn)
    p = t.scenes.make_scenes(64, c, seed=120 + ndyn, n_static=3, n_dynamic=0, mpc=mc)
    E.with_dynamic_obstacles(p, c, rng, dyn_slots(rng, 64, ndyn), boundary=(0, 1))
    sol = solve_parity(c, p)
    assert changed(c, p, sol, "od") >= 0.3
    # obstacles held in global scratch (live rank >= DYN_SLOTS) and in slots >= 32 touched the solve
    u0 = np.zeros((64, 2 * c.N_hor)); u0[:, 0::2] = 0.5
    parts = E.ref_eval(c, u0, p, terms=True)[3]
    live = E.dyn_live(p, c)
    rank = np.cumsum(live, 1) - 1
    hit = (np.asarray(parts["dyn_soft"]) > 0) & live
    assert (hit & (rank >= E.DYN_SLOTS)).any(1).sum() >= 3
    if ndyn > 32:
        assert hit[:, 32:].any(1).sum() >= 3


# ------------------------------------------------------------------ 3. static edge counts
@pytest.mark.parametrize("ne", [3, 5, 8])
@pytest.mark.parametrize("nstc", [10, 32])
def test_static_edge_counts(ne, nstc):
    """Regular ne-gons in slots with zero slots between them; the same obstacles compacted into the
    first slots give the same bits (stage_part1 drops zero slots, order kept)."""
    mc = t.Configurator(nstcobs=3 * ne, Nstcobs=nstc)
    c = mc.to_ttmpc()
    rng = np.random.default_rng(130 + ne + nstc)
    p = t.scenes.make_scenes(48, c, seed=130 + ne + nstc, n_dynamic=2, mpc=mc)
    slots = [1, 3, 4, 7, 8, 9] if nstc == 10 else [0, 5, 11, 17, 30, 31]
    E.with_static_polygons(p, c, rng, ne, slots)
    sol = solve_parity(c, p)
    assert changed(c, p, sol, "os") >= 0.25
    comp = t.BatchSolver(c).run(E.compact_static(p, c))
    for f in dataclasses.fields(sol):
        if f.name not in ("evals", "solve_time_ms"):
            assert np.array_equal(getattr(sol, f.name), getattr(comp, f.name)), f.name


# ------------------------------------------------------------------ 4. horizons
@pytest.mark.parametrize("N", [1, 2, 3, 7, 16, 17, 21, 22, 24, 31])
def test_horizons(N):
    """Horizons around the helper-lane split of the path deviation (nh = 32 - N helper lanes; for
    N >= 22 the loop runs N - nh trips), with static, dynamic and other-robot content."""
    mc = t.Configurator(N_hor=N)
    c = mc.to_ttmpc()
    p = rich_scenes(c, 48, 140 + N)
    sol = solve_parity(c, p)
    assert changed(c, p, sol, "c") >= 0.25


@pytest.mark.parametrize("N,mem", [(7, 1), (24, 3)])
def test_horizons_short_lbfgs_memory(N, mem):
    mc = t.Configurator(N_hor=N)
    c = mc.to_ttmpc(lbfgs_memory=mem)
    solve_parity(c, rich_scenes(c, 48, 150 + N))


# ------------------------------------------------------------------ 5. far coordinates
@pytest.mark.parametrize("offset", [(1e3, -1e3), (1e4, 1e4), (-3e4, 5e4), (1e5, 0.0)])
def test_far_coordinates_solve(cfg, offset):
    rng = np.random.default_rng(160)
    p = t.scenes.make_scenes(48, cfg, seed=160, n_static=4, n_dynamic=3, blocking_fraction=0.3)
    E.with_other_robots(p, cfg, rng, ["headon", "crossing", "parallel", "parked_in", "parked_out",
                                      "crossing", "headon", "empty", "empty", "crossing"])
    q = E.translate(p, cfg, *offset)
    sol = solve_parity(cfg, q)
    parts = E.ref_eval(cfg, sol.solution, q, terms=True)[3]
    assert (parts["contacts"] > 0).mean() >= 0.25


@pytest.mark.parametrize("shape", ["default", "runtime"])
def test_far_coordinates_eval_near_contacts(shape):
    """Other robots at d (1 +- delta) and ellipses with the rollout point on their axes at
    R (1 +- delta) from it, delta in {1e-3, 1e-5, 1e-7}, at coordinates up to 1e5 m, where one fp32
    ulp is ~8 mm: the fp32 prefilters must never reject a contact the fp64 test accepts."""
    mc = t.Configurator() if shape == "default" else t.Configurator(Nother=32, Ndynobs=64, N_hor=16)
    c = mc.to_ttmpc()
    n, N = 24, c.N_hor
    o = param_offsets(c)
    rng = np.random.default_rng(170)
    base = t.scenes.make_scenes(n, c, seed=170, n_static=2, n_dynamic=0, mpc=mc)
    u = np.tile(np.ravel(np.column_stack([np.full(N, 0.8), np.full(N, 0.15)])), (n, 1))
    deltas = np.array([1e-3, 1e-5, 1e-7])
    for off in [(0.0, 0.0), (1e3, -1e3), (1e4, 1e4), (-3e4, 5e4), (1e5, 0.0)]:
        p = E.translate(base, c, *off)
        xy = E.rollouts(c, u, p)
        cb = p[:, o["c"]:o["os"]].reshape(n, c.Nother, N, 3)
        for j in range(c.Nother):
            d = c.vehicle_width * (1 + rng.choice([-1, 1], (n, N)) * deltas[rng.integers(0, 3, (n, N))])
            phi = rng.uniform(0, 2 * np.pi, (n, N))
            cb[:, j, :, 0] = xy[..., 0] + d * np.cos(phi)
            cb[:, j, :, 1] = xy[..., 1] + d * np.sin(phi)
        p[:, o["c"]:o["os"]] = cb.reshape(n, -1)
        od = p[:, o["od"]:o["qstc"]].reshape(n, c.Ndynobs, N, 6)
        for j in range(c.Ndynobs):
            rx, ry = rng.uniform(0.5, 0.8, (n, 1)), rng.uniform(0.2, 0.45, (n, 1))
            ang = rng.uniform(0, np.pi, (n, 1))
            outer = rng.random((n, N)) < 0.5          # on the margin ellipse's major axis, else the inner one's minor axis
            s = 1 + rng.choice([-1, 1], (n, N)) * deltas[rng.integers(0, 3, (n, N))]
            dist = np.where(outer, (rx + c.social_margin + 1e-6) * s, (ry + 1e-6) * s)
            ax = np.where(outer, ang, ang + np.pi / 2)
            od[:, j, :, 0] = xy[..., 0] - dist * np.cos(ax)
            od[:, j, :, 1] = xy[..., 1] - dist * np.sin(ax)
            od[:, j, :, 2], od[:, j, :, 3], od[:, j, :, 4], od[:, j, :, 5] = rx, ry, ang, 1.0
        p[:, o["od"]:o["qstc"]] = od.reshape(n, -1)
        print("offset", off)
        _, parts = eval_checks(c, p, u, np.full(n, 10.0), rng.uniform(-1, 1, (n, 2 * N)))
        assert (parts["contacts"] > 0).all() and (np.asarray(parts["dyn_soft"]) > 0).any(1).all()
        assert (np.asarray(parts["D"]) > 0).any(1).all()


# ------------------------------------------------------------------ 6. out of the box
@pytest.mark.parametrize("speed", [10.0, 100.0])
def test_out_of_box_eval(cfg, speed):
    """Controls of +-10 and +-100 m/s take the rollout out of the live box: every robot and obstacle
    slot is scanned, and robots / obstacles parked beside the far part of the rollout (not live) count."""
    n, N = 32, cfg.N_hor
    rng = np.random.default_rng(180)
    p = t.scenes.make_scenes(n, cfg, seed=180, n_static=cfg.Nstcobs, n_dynamic=cfg.Ndynobs, blocking_fraction=0.3)
    E.with_other_robots(p, cfg, rng, robot_kinds(cfg.Nother))
    u = controls(rng, cfg, n)
    u[:, 0::2] = speed * rng.choice([-1.0, 1.0], (n, 1)) * rng.uniform(0.5, 1.0, (n, N))
    xy = E.rollouts(cfg, u, p)
    far = np.maximum(np.abs(xy[..., 0] - p[:, 0, None]), np.abs(xy[..., 1] - p[:, 1, None]))
    assert (far.max(1) > E.box_half(cfg)).all()        # every rollout left the box
    E.park_on_rollout(p, cfg, xy, robot_slots=[7, 9], dyn_slots=[5, 14], rng=rng)
    _, parts = eval_checks(cfg, p, u, np.full(n, 10.0), rng.uniform(-1, 1, (n, 2 * N)))
    live_dyn = E.dyn_live(p, cfg)
    assert not live_dyn[:, [5, 14]].any()
    assert (parts["robot_contacts"][:, [7, 9]] > 0).any(1).mean() >= 0.5
    assert (np.asarray(parts["dyn_soft"])[:, [5, 14]] > 0).any(1).mean() >= 0.5


def test_out_of_box_warm_start(cfg):
    """A warm start outside the control bounds: its rollout leaves the box."""
    n, N = 48, cfg.N_hor
    rng = np.random.default_rng(190)
    p = t.scenes.make_scenes(n, cfg, seed=190, n_static=4, n_dynamic=3, blocking_fraction=0.2)
    E.with_other_robots(p, cfg, rng, robot_kinds(cfg.Nother))
    u0 = controls(rng, cfg, n)
    u0[:, 0::2] = rng.choice([-1.0, 1.0], (n, 1)) * rng.uniform(5.0, 12.0, (n, N))
    xy = E.rollouts(cfg, u0, p)
    assert (np.maximum(np.abs(xy[..., 0] - p[:, 0, None]), np.abs(xy[..., 1] - p[:, 1, None])).max(1)
            > E.box_half(cfg)).all()
    solve_parity(cfg, p, initial_guess=u0)


# ------------------------------------------------------------------ 7. non-finite inputs
def test_non_finite_scenes_in_a_finite_batch(cfg, monkeypatch):
    """Six scenes with NaN / inf inputs among 300 finite ones, on the device path with and without tail
    helpers: the finite scenes get exactly the results of the batch without the bad ones, the bad
    ones the oracle's status, iteration counts, controls and cost (NaN where the oracle has NaN)."""
    import torch
    o = param_offsets(cfg)
    rng = np.random.default_rng(200)
    good = t.scenes.make_scenes(300, cfg, seed=200, n_static=4, n_dynamic=3, blocking_fraction=0.2)
    E.with_other_robots(good, cfg, rng, robot_kinds(cfg.Nother))
    bad = good[[3, 50, 100, 150, 200, 250]].copy()
    bad[0, 0] = np.nan                                 # start x
    bad[1, 0] = np.inf                                 # start x
    bad[2, o["vref"] + 4] = np.nan                     # speed reference
    bad[3, o["od"] + 6 * 5] = np.nan                   # a dynamic centre x (obstacle 0, step 5)
    bad[4, o["os"]] = np.nan                           # a static b (obstacle 0, edge 0)
    bad[5, o["r"] + 3 * 3] = np.nan                    # a reference x (step 3)
    ref = O.solve_batch(cfg, bad, threads=THREADS, warp=True)
    # the first three never converge (cost NaN or inf after every iteration), as the reference-order oracle does too
    assert (ref["exit_status"][:3] == 1).all() and not np.isfinite(ref["cost"][:3]).any()
    assert np.isfinite(ref["u"]).all() and np.isfinite(ref["cost"][3:]).all()
    pos = np.array([0, 31, 32, 97, 180, 299]) + np.arange(6)   # among finite scenes, in shared CTAs
    allp = np.insert(good, pos - np.arange(6), bad, axis=0)
    assert np.array_equal(np.flatnonzero(~np.isfinite(allp).all(1)), pos)
    fin = np.setdiff1d(np.arange(len(allp)), pos)

    def solve(p):
        sol = t.BatchSolver(cfg).run_device(torch.from_numpy(p).cuda(), t.BatchSolver(cfg).alloc_device(len(p)))
        torch.cuda.synchronize()
        return {f.name: getattr(sol, f.name).cpu().numpy() for f in dataclasses.fields(sol)
                if f.name not in ("evals", "solve_time_ms")}

    for helpers in (True, False):
        if not helpers:
            monkeypatch.setenv("TTMPC_NO_HELPERS", "1")
        a, b = solve(allp), solve(good)
        for name in a:
            assert np.array_equal(a[name][fin], b[name]), (helpers, name)
        assert np.array_equal(a["exit_status"][pos], ref["exit_status"])
        assert np.array_equal(a["num_inner_iterations"][pos], ref["inner"])
        assert np.array_equal(a["num_outer_iterations"][pos], ref["outer"])
        assert np.array_equal(a["solution"][pos], ref["u"], equal_nan=True)
        assert np.array_equal(a["cost"][pos], ref["cost"], equal_nan=True)


# ------------------------------------------------------------------ 8. evaluation at every new shape
SHAPES = [dict(Nother=1), dict(Nother=31), dict(Nother=32), dict(Ndynobs=32), dict(Ndynobs=33),
          dict(Ndynobs=64), dict(nstcobs=9), dict(nstcobs=15, Nstcobs=32), dict(nstcobs=24, Nstcobs=32)] + \
         [dict(N_hor=N) for N in (1, 2, 3, 7, 16, 17, 21, 22, 24, 31)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: ",".join(f"{k}={v}" for k, v in s.items()))
def test_eval_new_shapes(shape):
    """eval_kernel<DimsRuntime> at the new shapes: in-bound and 3x out-of-bound controls, with
    multipliers and a penalty (psi, grad psi)."""
    mc = t.Configurator(**shape)
    c = mc.to_ttmpc()
    n, N = 48, c.N_hor
    rng = np.random.default_rng(210)
    p = rich_scenes(c, n, 210)
    u = controls(rng, c, n, 1.0)
    u[n // 2:] *= 3.0
    _, parts = eval_checks(c, p, u, rng.uniform(1.0, 50.0, n), rng.uniform(-1, 1, (n, 2 * N)))
    assert (parts["contacts"] > 0).sum() >= 3
    assert (np.asarray(parts["S"]) > 0).sum() >= 3
    assert (np.asarray(parts["dyn_soft"]) > 0).any(1).sum() >= 3
    nh = 32 - N
    if N - nh - 1 > (N + 1) // 2:   # steps k >= nh scan their whole range alone, in N - nh trips (the last
        # segment is the duplicated end point, never a strict minimum: from N = 23 on, more than half remain)
        k = np.arange(N)[None, :]
        assert ((parts["jmin"] >= k + (N + 1) // 2) & (k >= nh)).any(1).sum() >= 3
