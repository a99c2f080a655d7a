"""CPU checks of the edge-scene builders (tests/edge_scenes.py), of the long-double reference
ref_eval, and of scenes.make_scenes at short horizons and on the benchmark workloads."""
import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.geometry import polygon_halfspace_representation
from trajtrack_mpcndqn_rlboost_b200.mpc_config import param_offsets
from tests import edge_scenes as E
from tests import oracle_lib as O


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(1.0, np.abs(b).max()))


def controls(rng, cfg, n, scale=1.0):
    u = np.empty((n, 2 * cfg.N_hor))
    u[:, 0::2] = scale * rng.uniform(cfg.lin_vel_min, cfg.lin_vel_max, (n, cfg.N_hor))
    u[:, 1::2] = scale * rng.uniform(-cfg.ang_vel_max, cfg.ang_vel_max, (n, cfg.N_hor))
    return u


def edge_batches():
    """One batch per scene kind the GPU tests build (tests/test_gpu_edge_scenes.py), 24 scenes each."""
    rng = np.random.default_rng(5)
    out = []
    cfg = t.Configurator().to_ttmpc()
    p = t.scenes.make_scenes(24, cfg, seed=1, n_static=4, n_dynamic=3)
    out.append(("robots", cfg, E.with_other_robots(p, cfg, rng, (list(E.ROBOT_KINDS) * 2)[:10])))
    for ndyn in (15, 33, 64):
        c = t.Configurator(Ndynobs=ndyn).to_ttmpc()
        p = t.scenes.make_scenes(24, c, seed=ndyn, n_static=2)
        slots = [sorted(rng.choice(ndyn, 8, replace=False)) for _ in range(24)]
        out.append((f"dyn{ndyn}", c, E.with_dynamic_obstacles(p, c, rng, slots, boundary=slots[0][:2])))
    for ne in (3, 5, 8):
        c = t.Configurator(nstcobs=3 * ne, Nstcobs=32).to_ttmpc()
        p = t.scenes.make_scenes(24, c, seed=ne, n_dynamic=2)
        out.append((f"static{ne}", c, E.with_static_polygons(p, c, rng, ne, [1, 6, 7, 20, 31])))
    for N in (1, 2, 3, 24):
        c = t.Configurator(N_hor=N).to_ttmpc()
        p = t.scenes.make_scenes(24, c, seed=N, n_static=3, n_dynamic=3)
        p = E.with_other_robots(p, c, rng, ["headon", "crossing", "parallel"])
        out.append((f"N{N}", c, E.with_folded_reference(p, c) if N > 3 else p))
    return out


def test_ref_eval_matches_reference_goldens(cfg, golden_problem):
    """The long-double restatement against the reference's own MpcModule.build values
    (the bars of test_eval_matches_reference_goldens)."""
    g = golden_problem
    f, F1, F2 = E.ref_eval(cfg, g["u"], g["p"])
    assert rel(f, g["f"]) <= 1e-12
    assert np.abs(np.asarray(F1, np.float64) - g["F1"]).max() <= 1e-12
    assert rel(F2, g["F2"]) <= 1e-12


@pytest.mark.parametrize("offset", [(0.0, 0.0), (100.0, -100.0), (-60.0, 80.0)])
def test_ref_eval_matches_oracle_on_edge_scenes(offset):
    """ref_eval against the reference-order oracle (O.evaluate) on every kind of edge scene, at
    in-bound controls and at 10x out-of-bound ones, moved by up to 100 m."""
    rng = np.random.default_rng(9)
    for name, c, p in edge_batches():
        q = E.translate(p, c, *offset)
        for scale in (1.0, 10.0):
            u = controls(rng, c, len(q), scale)
            f, F1, F2 = E.ref_eval(c, u, q)
            ev = [O.evaluate(c, u[i], q[i]) for i in range(len(q))]
            assert rel(f, [e[0] for e in ev]) <= 1e-12, name
            assert np.abs(np.asarray(F1, np.float64) - np.array([e[1] for e in ev])).max() <= 1e-12, name
            if c.Ndynobs:
                assert rel(F2, np.array([e[2] for e in ev])) <= 1e-12, name


def test_builders_fill_what_they_claim():
    """Robots, polygons and ellipses land in the slots asked for; live-box edges are 1e-3 m away."""
    rng = np.random.default_rng(2)
    cfg = t.Configurator().to_ttmpc()
    o = param_offsets(cfg)
    N = cfg.N_hor
    p = t.scenes.make_scenes(16, cfg, seed=2, n_static=0)
    E.with_other_robots(p, cfg, rng, ["headon", "parked_in", "parked_out", "empty", "parallel"])
    c = p[:, o["c"]:o["os"]].reshape(16, cfg.Nother, N, 3)
    assert not c[:, 3:4].any() and not c[:, 5:].any()
    edge = E.box_half(cfg) + E.robot_pad(cfg)
    for j, sgn in ((1, -1), (2, 1)):
        far = np.maximum(np.abs(c[:, j, :, 0] - p[:, None, 0]), np.abs(c[:, j, :, 1] - p[:, None, 1]))
        assert np.allclose(far, edge + sgn * 1e-3, rtol=0, atol=1e-9)
    r = p[:, o["r"]:o["r"] + 3 * N].reshape(16, N, 3)
    lat = np.hypot(c[:, 4, :, 0] - r[..., 0], c[:, 4, :, 1] - r[..., 1])
    assert (lat < cfg.vehicle_width).all()
    # polygons: rows of geometry.polygon_halfspace_representation, edge for edge
    b, a0, a1 = E.regular_polygon_rows(3.0, -2.0, 0.7, 0.4, 5)
    ang = 0.4 + 2 * np.pi * np.arange(5) / 5
    gb, ga0, ga1 = polygon_halfspace_representation(np.stack([3.0 + 0.7 * np.cos(ang), -2.0 + 0.7 * np.sin(ang)], 1))
    key = lambda x, y, z: sorted(zip(np.round(x, 12), np.round(y, 12), np.round(z, 12)))
    assert np.allclose(np.array(key(b, a0, a1)), np.array(key(gb, ga0, ga1)), rtol=0, atol=1e-12)
    c5 = t.Configurator(nstcobs=15).to_ttmpc()
    p5 = E.with_static_polygons(t.scenes.make_scenes(4, c5, seed=3), c5, rng, 5, [2, 7])
    blk = p5[:, param_offsets(c5)["os"]:param_offsets(c5)["od"]].reshape(4, c5.Nstcobs, 15)
    assert (blk.any(-1) == np.isin(np.arange(c5.Nstcobs), [2, 7])[None]).all()
    comp = E.compact_static(p5, c5)[:, param_offsets(c5)["os"]:param_offsets(c5)["od"]].reshape(4, c5.Nstcobs, 15)
    assert np.array_equal(comp[:, :2], blk[:, [2, 7]]) and not comp[:, 2:].any()
    # dynamic: slots >= 32 and per-scene slot lists
    c64 = t.Configurator(Ndynobs=64).to_ttmpc()
    p64 = E.with_dynamic_obstacles(t.scenes.make_scenes(2, c64, seed=4), c64, rng, [[3, 40, 63], [31, 32]])
    od = p64[:, param_offsets(c64)["od"]:param_offsets(c64)["qstc"]].reshape(2, 64, c64.N_hor, 6)
    assert np.flatnonzero(od[0].any((1, 2))).tolist() == [3, 40, 63]
    assert np.flatnonzero(od[1].any((1, 2))).tolist() == [31, 32]


def test_translate_moves_every_block_rigidly():
    """Each term of the cost depends only on differences of positions: after a rigid move by
    (37, -21) m the long-double f and F2 stay the same to rounding of the moved inputs."""
    rng = np.random.default_rng(4)
    for name, c, p in edge_batches():
        u = controls(rng, c, len(p))
        f0, _, F20 = E.ref_eval(c, u, p)
        f1, _, F21 = E.ref_eval(c, u, E.translate(p, c, 37.0, -21.0))
        assert rel(f1, f0) <= 1e-11, name
        if c.Ndynobs:
            assert rel(F21, F20) <= 1e-11, name


@pytest.mark.parametrize("N", [1, 2, 3])
def test_make_scenes_short_horizons(N):
    c = t.Configurator(N_hor=N).to_ttmpc()
    p = t.scenes.make_scenes(64, c, seed=N, n_static=4, n_dynamic=3)
    o = param_offsets(c)
    assert p.shape == (64, o["np"]) and np.isfinite(p).all()
    r = p[:, o["r"]:o["r"] + 3 * N].reshape(64, N, 3)
    assert np.array_equal(p[:, 3:6], r[:, -1])
    f, F1, F2 = O.evaluate(c, np.zeros(2 * N), p[0])
    assert np.isfinite(f) and F1.shape == (2 * N,)


# ---- make_scenes as of the commit before short horizons were allowed: the benchmark inputs
def _make_scenes_before(n, cfg, seed=0, n_static=4, n_dynamic=0, mode_speed=1.2, blocking_fraction=0.1, mpc=None):
    rng = np.random.default_rng(seed)
    mpc = mpc or t.Configurator()
    N, ts = cfg.N_hor, cfg.ts
    off = param_offsets(cfg)
    p = np.zeros((n, off["np"]))
    x0 = rng.uniform(8.0, 32.0, n)
    y0 = rng.uniform(8.0, 32.0, n)
    heading = rng.uniform(-np.pi, np.pi, n)
    th0 = heading + rng.normal(0.0, 0.25, n)
    lateral = rng.normal(0.0, 0.15, n)
    px = x0 - lateral * np.sin(heading)
    py = y0 + lateral * np.cos(heading)
    leg1 = rng.uniform(2.0, 6.0, n)
    turn = rng.uniform(-0.9, 0.9, n)
    step = mode_speed * ts
    k = np.arange(1, N + 1)[None, :] * step
    on1 = k <= leg1[:, None]
    h2 = heading + turn
    rx = np.where(on1, px[:, None] + k * np.cos(heading)[:, None],
                  px[:, None] + leg1[:, None] * np.cos(heading)[:, None] + (k - leg1[:, None]) * np.cos(h2)[:, None])
    ry = np.where(on1, py[:, None] + k * np.sin(heading)[:, None],
                  py[:, None] + leg1[:, None] * np.sin(heading)[:, None] + (k - leg1[:, None]) * np.sin(h2)[:, None])
    rth = np.where(on1, heading[:, None], h2[:, None])
    short = rng.random(n) < 0.15
    n_keep = np.where(short, rng.integers(3, N, n), N)
    idx = np.minimum(np.arange(N)[None, :], n_keep[:, None] - 1)
    rx = np.take_along_axis(rx, idx, 1); ry = np.take_along_axis(ry, idx, 1)
    rth = np.take_along_axis(rth, idx, 1)
    p[:, 0], p[:, 1], p[:, 2] = x0, y0, th0
    p[:, 3], p[:, 4], p[:, 5] = rx[:, -1], ry[:, -1], rth[:, -1]
    p[:, 6] = rng.uniform(0.0, mode_speed, n)
    p[:, 7] = rng.uniform(-0.3, 0.3, n)
    q = [mpc.qpos, mpc.qvel, mpc.qtheta, mpc.lin_vel_penalty, mpc.ang_vel_penalty,
         mpc.qpN, mpc.qthetaN, mpc.qrpd, mpc.lin_acc_penalty, mpc.ang_acc_penalty]
    p[:, off["q"]:off["q"] + 10] = np.asarray(q, dtype=np.float64)
    p[:, off["r"]:off["r"] + 3 * N] = np.stack([rx, ry, rth], axis=-1).reshape(n, 3 * N)
    dist_goal = np.hypot(x0 - rx[:, -1], y0 - ry[:, -1])
    vref = np.where(dist_goal >= mode_speed * N * ts, mode_speed, np.maximum(dist_goal / N / ts, mpc.low_speed))
    p[:, off["vref"]:off["vref"] + N] = vref[:, None]
    ns_use = min(n_static, cfg.Nstcobs)
    if ns_use and cfg.nstcobs // 3 == 4:
        along = rng.uniform(1.5, 5.5, (n, ns_use))
        blocking = rng.random((n, ns_use)) < blocking_fraction
        side = np.where(blocking, rng.normal(0.0, 0.4, (n, ns_use)),
                        rng.choice([-1.0, 1.0], (n, ns_use)) * rng.uniform(1.2, 3.0, (n, ns_use)))
        cx = px[:, None] + along * np.cos(heading)[:, None] - side * np.sin(heading)[:, None]
        cy = py[:, None] + along * np.sin(heading)[:, None] + side * np.cos(heading)[:, None]
        hx = rng.uniform(0.3, 1.0, (n, ns_use)); hy = rng.uniform(0.3, 1.0, (n, ns_use))
        ang = rng.uniform(0, np.pi, (n, ns_use))
        b, a0, a1 = t.scenes._rect_halfspaces(cx, cy, hx, hy, ang)
        p[:, off["os"]:off["os"] + ns_use * cfg.nstcobs] = np.concatenate([b, a0, a1], axis=-1).reshape(n, -1)
    nd_use = min(n_dynamic, cfg.Ndynobs)
    if nd_use:
        along = rng.uniform(1.0, 5.0, (n, nd_use))
        side = rng.uniform(-2.5, 2.5, (n, nd_use))
        ox = px[:, None] + along * np.cos(heading)[:, None] - side * np.sin(heading)[:, None]
        oy = py[:, None] + along * np.sin(heading)[:, None] + side * np.cos(heading)[:, None]
        vdir = rng.uniform(-np.pi, np.pi, (n, nd_use)); vmag = rng.uniform(0.0, 1.0, (n, nd_use))
        steps = np.arange(1, N + 1)[None, None, :]
        ex = ox[..., None] + vmag[..., None] * np.cos(vdir)[..., None] * ts * steps
        ey = oy[..., None] + vmag[..., None] * np.sin(vdir)[..., None] * ts * steps
        rxy = rng.uniform(0.2, 0.8, (n, nd_use, 2))
        ang = rng.uniform(0, np.pi, (n, nd_use))
        rec = np.stack([ex, ey, np.broadcast_to(rxy[..., 0:1], ex.shape), np.broadcast_to(rxy[..., 1:2], ex.shape),
                        np.broadcast_to(ang[..., None], ex.shape), np.ones_like(ex)], axis=-1)
        p[:, off["od"]:off["od"] + nd_use * 6 * N] = rec.reshape(n, -1)
    p[:, off["qstc"]:off["qstc"] + N] = 1e3
    p[:, off["qdyn"]:off["qdyn"] + N] = 1e3
    return p


@pytest.mark.parametrize("name", ["static4096", "mixed4096", "dynamic8192", "sweep:N=10,Nstc=10,Ndyn=15"])
def test_make_scenes_benchmark_inputs_unchanged(name):
    """The benchmark's seeded inputs (bench.py: seeds 1000 + 100 j) are what they were."""
    if name.startswith("sweep:"):
        mc = t.Configurator(N_hor=10, Nstcobs=10, Ndynobs=15)
        w = dict(n=4096, n_static=4, n_dynamic=3, blocking_fraction=0.1)
    else:
        mc, w = t.Configurator(), t.scenes.WORKLOADS[name]
    c = mc.to_ttmpc()
    for seed in (1000, 1100):
        kw = dict(seed=seed, n_static=w["n_static"], n_dynamic=w["n_dynamic"],
                  blocking_fraction=w["blocking_fraction"], mpc=mc)
        assert np.array_equal(t.scenes.make_scenes(w["n"], c, **kw), _make_scenes_before(w["n"], c, **kw))
