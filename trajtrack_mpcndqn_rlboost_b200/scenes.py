"""Synthetic scenes of the shapes BASELINE.json names, packed exactly like the
reference packs one robot's parameters (trajectory_generator.py:251-254).

A scene = one robot at a random pose in a 40 m x 40 m world (kept away from the
origin, where the reference's zero-padded obstacle / other-robot slots live), a
polyline reference path sampled at base_speed*ts like
``get_global_ref_traj`` does, rectangles as static obstacles (half-space form)
and, optionally, ellipses moving at constant velocity as dynamic obstacles with
their N-step prediction (main.py:80-88 est_dyn_obs_positions).
"""
from __future__ import annotations

import numpy as np

from ._lib import TtmpcConfig
from .mpc_config import Configurator, param_offsets


def _rect_halfspaces(cx, cy, hx, hy, ang):
    """Half-space rows (b, a0, a1)[4] of rectangles, scaled like
    polygon_halfspace_representation: a.(v - centre) = 1 on each edge."""
    ca, sa = np.cos(ang), np.sin(ang)
    # outward unit normals of the 4 edges and their distance from the centre
    nx = np.stack([ca, -sa, -ca, sa], axis=-1)
    ny = np.stack([sa, ca, -sa, -ca], axis=-1)
    dist = np.stack([hx, hy, hx, hy], axis=-1)
    a0 = nx / dist
    a1 = ny / dist
    b = a0 * cx[..., None] + a1 * cy[..., None] + 1.0
    return b, a0, a1


def make_scenes(n: int, cfg: TtmpcConfig, seed: int = 0, n_static: int = 4, n_dynamic: int = 0,
                mode_speed: float = 1.2, blocking_fraction: float = 0.1, mpc: Configurator = None):
    """Returns p [n, np] float64.

    Static obstacles are only placed when the configuration has 4-edge slots (nstcobs = 12);
    with any other edge count the static block stays zero.  Other robots are never placed: the
    c block is all zeros.  Live obstacles always fill the first slots."""
    rng = np.random.default_rng(seed)
    mpc = mpc or Configurator()
    N, ts = cfg.N_hor, cfg.ts
    off = param_offsets(cfg)
    p = np.zeros((n, off["np"]))
    # ---- start pose and a two-leg reference path
    x0 = rng.uniform(8.0, 32.0, n)
    y0 = rng.uniform(8.0, 32.0, n)
    heading = rng.uniform(-np.pi, np.pi, n)
    th0 = heading + rng.normal(0.0, 0.25, n)
    lateral = rng.normal(0.0, 0.15, n)          # robot starts slightly off the path
    px = x0 - lateral * np.sin(heading)
    py = y0 + lateral * np.cos(heading)
    leg1 = rng.uniform(2.0, 6.0, n)
    turn = rng.uniform(-0.9, 0.9, n)
    step = mode_speed * ts
    k = np.arange(1, N + 1)[None, :] * step                     # arc length of sample k
    on1 = k <= leg1[:, None]
    h2 = heading + turn
    rx = np.where(on1, px[:, None] + k * np.cos(heading)[:, None],
                  px[:, None] + leg1[:, None] * np.cos(heading)[:, None]
                  + (k - leg1[:, None]) * np.cos(h2)[:, None])
    ry = np.where(on1, py[:, None] + k * np.sin(heading)[:, None],
                  py[:, None] + leg1[:, None] * np.sin(heading)[:, None]
                  + (k - leg1[:, None]) * np.sin(h2)[:, None])
    rth = np.where(on1, heading[:, None], h2[:, None])
    # some scenes end their path early (goal inside the horizon): tail padded with the last state
    # (at least 3 samples kept; horizons of 3 or less keep 1..N-1, and a horizon of 1 cannot end early)
    short = rng.random(n) < 0.15
    lo = min(3, N - 1)
    n_keep = np.where(short, rng.integers(lo, N, n), N) if lo >= 1 else np.full(n, N)
    idx = np.minimum(np.arange(N)[None, :], n_keep[:, None] - 1)
    rx = np.take_along_axis(rx, idx, 1); ry = np.take_along_axis(ry, idx, 1)
    rth = np.take_along_axis(rth, idx, 1)
    # ---- s block
    p[:, 0], p[:, 1], p[:, 2] = x0, y0, th0
    p[:, 3], p[:, 4], p[:, 5] = rx[:, -1], ry[:, -1], rth[:, -1]      # finish_state
    p[:, 6] = rng.uniform(0.0, mode_speed, n)                          # last action v
    p[:, 7] = rng.uniform(-0.3, 0.3, n)                                # last action w
    # ---- q block (set_work_mode, mode != aligning)
    q = [mpc.qpos, mpc.qvel, mpc.qtheta, mpc.lin_vel_penalty, mpc.ang_vel_penalty,
         mpc.qpN, mpc.qthetaN, mpc.qrpd, mpc.lin_acc_penalty, mpc.ang_acc_penalty]
    p[:, off["q"]:off["q"] + 10] = np.asarray(q, dtype=np.float64)
    # ---- r block
    ref = np.stack([rx, ry, rth], axis=-1).reshape(n, 3 * N)
    p[:, off["r"]:off["r"] + 3 * N] = ref
    dist_goal = np.hypot(x0 - rx[:, -1], y0 - ry[:, -1])
    vref = np.where(dist_goal >= mode_speed * N * ts, mode_speed,
                    np.maximum(dist_goal / N / ts, mpc.low_speed))
    p[:, off["vref"]:off["vref"] + N] = vref[:, None]
    # ---- static obstacles: rectangles near the path, a fraction of them straddling it
    ns_use = min(n_static, cfg.Nstcobs)
    ne = cfg.nstcobs // 3
    if ns_use and ne == 4:
        along = rng.uniform(1.5, 5.5, (n, ns_use))
        blocking = rng.random((n, ns_use)) < blocking_fraction
        side = np.where(blocking, rng.normal(0.0, 0.4, (n, ns_use)),
                        rng.choice([-1.0, 1.0], (n, ns_use)) * rng.uniform(1.2, 3.0, (n, ns_use)))
        cx = px[:, None] + along * np.cos(heading)[:, None] - side * np.sin(heading)[:, None]
        cy = py[:, None] + along * np.sin(heading)[:, None] + side * np.cos(heading)[:, None]
        hx = rng.uniform(0.3, 1.0, (n, ns_use)); hy = rng.uniform(0.3, 1.0, (n, ns_use))
        ang = rng.uniform(0, np.pi, (n, ns_use))
        b, a0, a1 = _rect_halfspaces(cx, cy, hx, hy, ang)
        blk = np.concatenate([b, a0, a1], axis=-1)                     # [n, ns_use, 12]
        p[:, off["os"]:off["os"] + ns_use * cfg.nstcobs] = blk.reshape(n, -1)
    # ---- dynamic obstacles: constant-velocity ellipses crossing the path
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
        rec = np.stack([ex, ey, np.broadcast_to(rxy[..., 0:1], ex.shape),
                        np.broadcast_to(rxy[..., 1:2], ex.shape),
                        np.broadcast_to(ang[..., None], ex.shape), np.ones_like(ex)], axis=-1)
        p[:, off["od"]:off["od"] + nd_use * 6 * N] = rec.reshape(n, -1)
    # ---- obstacle weights (set_obstacle_weights(1e3, 1e3), trajectory_generator.py:58)
    p[:, off["qstc"]:off["qstc"] + N] = 1e3
    p[:, off["qdyn"]:off["qdyn"] + N] = 1e3
    return p


WORKLOADS = {
    # BASELINE.json configs[1]: 4096 scenes, default horizon, static polygon obstacles
    "static4096": dict(n=4096, n_static=4, n_dynamic=0, blocking_fraction=0.1, solver={}),
    # default shapes with both obstacle kinds active (diagnostics / sweep reference point)
    "mixed4096": dict(n=4096, n_static=4, n_dynamic=3, blocking_fraction=0.1, solver={}),
    # configs[2] per-GPU shard: moving ellipses, long iteration limits
    "dynamic8192": dict(n=8192, n_static=3, n_dynamic=4, blocking_fraction=0.1,
                        solver=dict(max_inner_iterations=2000, max_outer_iterations=20)),
}


def make_fleet(n: int, seed: int = 0, n_static: int = 4, n_moving: int = 2):
    """Synthetic closed-loop fleet for FleetPlanner: every robot gets a start pose, a three-node
    reference path (10-20 m), its own rectangles near the path and obstacles crossing it at
    constant velocity.  Returns a dict of numpy arrays / lists."""
    rng = np.random.default_rng(seed)
    x0 = rng.uniform(8.0, 32.0, n); y0 = rng.uniform(8.0, 32.0, n)
    heading = rng.uniform(-np.pi, np.pi, n)
    leg1 = rng.uniform(4.0, 9.0, n); leg2 = rng.uniform(4.0, 9.0, n)
    h2 = heading + rng.uniform(-0.9, 0.9, n)
    mx, my = x0 + leg1 * np.cos(heading), y0 + leg1 * np.sin(heading)
    gx, gy = mx + leg2 * np.cos(h2), my + leg2 * np.sin(h2)
    lateral = rng.normal(0.0, 0.1, n)
    init = np.stack([x0 - lateral * np.sin(heading), y0 + lateral * np.cos(heading),
                     heading + rng.normal(0.0, 0.2, n)], axis=1)
    goal = np.stack([gx, gy, np.zeros(n)], axis=1)
    paths = [[(x0[i], y0[i]), (mx[i], my[i]), (gx[i], gy[i])] for i in range(n)]
    along = rng.uniform(2.0, 8.0, (n, n_static))
    side = rng.choice([-1.0, 1.0], (n, n_static)) * rng.uniform(1.3, 3.0, (n, n_static))
    cx = x0[:, None] + along * np.cos(heading)[:, None] - side * np.sin(heading)[:, None]
    cy = y0[:, None] + along * np.sin(heading)[:, None] + side * np.cos(heading)[:, None]
    hx = rng.uniform(0.3, 0.9, (n, n_static)); hy = rng.uniform(0.3, 0.9, (n, n_static))
    polys = [[[(cx[i, j] - hx[i, j], cy[i, j] - hy[i, j]), (cx[i, j] + hx[i, j], cy[i, j] - hy[i, j]),
               (cx[i, j] + hx[i, j], cy[i, j] + hy[i, j]), (cx[i, j] - hx[i, j], cy[i, j] + hy[i, j])]
              for j in range(n_static)] for i in range(n)]
    a = rng.uniform(3.0, 9.0, (n, n_moving)); s = rng.choice([-1.0, 1.0], (n, n_moving)) * rng.uniform(3.0, 5.0, (n, n_moving))
    ox = x0[:, None] + a * np.cos(heading)[:, None] - s * np.sin(heading)[:, None]
    oy = y0[:, None] + a * np.sin(heading)[:, None] + s * np.cos(heading)[:, None]
    vdir = rng.uniform(-np.pi, np.pi, (n, n_moving)); vmag = rng.uniform(0.0, 0.05, (n, n_moving))
    return dict(init=init, goal=goal, paths=paths, static_polys=polys,
                moving_pos=np.stack([ox, oy], axis=-1),
                moving_disp=np.stack([vmag * np.cos(vdir), vmag * np.sin(vdir)], axis=-1))


def make_missions(n: int, tasks: int, seed: int = 0, n_moving: int = 2, max_static: int = 10):
    """Synthetic missions for FleetPlanner.set_tasks: every robot gets a chain of ``tasks`` tasks,
    each a two-leg path (4-8 m per leg) that starts at the goal of the task before it (the first at
    the robot's start), one rectangle beside every leg while the ``max_static`` static slots last, and
    obstacles crossing its first leg at constant velocity as in ``make_fleet``.

    Returns make_fleet's keys for the first task (init, goal, paths, static_polys, moving_pos,
    moving_disp) and task_goals / task_paths: per robot, the goals [3] and paths of the other
    ``tasks - 1`` tasks, in the form ``FleetPlanner.set_tasks`` takes."""
    rng = np.random.default_rng(seed)
    x0 = rng.uniform(8.0, 32.0, n); y0 = rng.uniform(8.0, 32.0, n)
    heading = rng.uniform(-np.pi, np.pi, n)
    lateral = rng.normal(0.0, 0.1, n)
    init = np.stack([x0 - lateral * np.sin(heading), y0 + lateral * np.cos(heading),
                     heading + rng.normal(0.0, 0.2, n)], axis=1)
    goals, paths, polys = [[] for _ in range(n)], [[] for _ in range(n)], [[] for _ in range(n)]
    ax, ay, h = x0.copy(), y0.copy(), heading.copy()
    for k in range(tasks):
        if k:
            h = h + rng.uniform(-2.5, 2.5, n)                  # the next task leaves in a new direction
        leg1 = rng.uniform(4.0, 8.0, n); leg2 = rng.uniform(4.0, 8.0, n)
        h2 = h + rng.uniform(-0.9, 0.9, n)
        mx, my = ax + leg1 * np.cos(h), ay + leg1 * np.sin(h)
        gx, gy = mx + leg2 * np.cos(h2), my + leg2 * np.sin(h2)
        for (sx, sy, lh, ll) in ((ax, ay, h, leg1), (mx, my, h2, leg2)):
            along = rng.uniform(0.25, 0.75, n) * ll
            side = rng.choice([-1.0, 1.0], n) * rng.uniform(1.3, 3.0, n)
            cx = sx + along * np.cos(lh) - side * np.sin(lh)
            cy = sy + along * np.sin(lh) + side * np.cos(lh)
            hx = rng.uniform(0.3, 0.9, n); hy = rng.uniform(0.3, 0.9, n)
            for i in range(n):
                if len(polys[i]) < max_static:
                    polys[i].append([(cx[i] - hx[i], cy[i] - hy[i]), (cx[i] + hx[i], cy[i] - hy[i]),
                                     (cx[i] + hx[i], cy[i] + hy[i]), (cx[i] - hx[i], cy[i] + hy[i])])
        for i in range(n):
            goals[i].append((gx[i], gy[i], 0.0))
            paths[i].append([(ax[i], ay[i]), (mx[i], my[i]), (gx[i], gy[i])])
        ax, ay, h = gx, gy, h2
    a = rng.uniform(3.0, 9.0, (n, n_moving)); s = rng.choice([-1.0, 1.0], (n, n_moving)) * rng.uniform(3.0, 5.0, (n, n_moving))
    ox = x0[:, None] + a * np.cos(heading)[:, None] - s * np.sin(heading)[:, None]
    oy = y0[:, None] + a * np.sin(heading)[:, None] + s * np.cos(heading)[:, None]
    vdir = rng.uniform(-np.pi, np.pi, (n, n_moving)); vmag = rng.uniform(0.0, 0.05, (n, n_moving))
    return dict(init=init, goal=np.array([g[0] for g in goals]), paths=[p[0] for p in paths],
                static_polys=polys, task_goals=[g[1:] for g in goals], task_paths=[p[1:] for p in paths],
                moving_pos=np.stack([ox, oy], axis=-1),
                moving_disp=np.stack([vmag * np.cos(vdir), vmag * np.sin(vdir)], axis=-1))


def make_warehouse(n: int, tasks: int, seed: int = 0, shelves: int = 10_000, shelf=(1.0, 4.0), aisle: float = 3.0,
                   hops: int = 4):
    """A warehouse floor for FleetPlanner.set_world: about ``shelves`` rectangular shelves (shelf =
    width x depth, m) on a lattice with aisles ``aisle`` m wide between them, so the floor's density
    stays the same at any size.  Robots start at random aisle crossings; every task is a Manhattan
    route along aisle centre lines (x first or y first, at random) to a random other crossing at most
    ``hops`` crossings away in each direction, ending 2-20 cm short of it.  A route keeps aisle / 2
    from every shelf; a robot starts within 5 cm of its first route's first crossing.

    Returns the keys of make_missions with the shared map in place of per-robot obstacles: init,
    goal, paths (the first task), world_polys (every shelf, CCW rectangles), task_goals / task_paths
    (the other ``tasks - 1`` tasks), moving_pos / moving_disp ([n][0][2]: no moving obstacles)."""
    rng = np.random.default_rng(seed)
    sw, sd = float(shelf[0]), float(shelf[1])
    gx = int(np.ceil(np.sqrt(shelves)))
    gy = int(np.ceil(shelves / gx))
    px, py = sw + aisle, sd + aisle
    x0 = aisle + px * np.arange(gx)[:, None] + np.zeros(gy)[None]
    y0 = aisle + py * np.arange(gy)[None, :] + np.zeros(gx)[:, None]
    x0, y0 = x0.ravel(), y0.ravel()
    world = [[(a, b), (a + sw, b), (a + sw, b + sd), (a, b + sd)] for a, b in zip(x0.tolist(), y0.tolist())]

    def crossing(i, j):
        return float(i * px + 0.5 * aisle), float(j * py + 0.5 * aisle)

    ci, cj = rng.integers(0, gx + 1, n), rng.integers(0, gy + 1, n)
    pos = [crossing(i, j) for i, j in zip(ci, cj)]
    goals, paths = [[] for _ in range(n)], [[] for _ in range(n)]
    for _ in range(max(tasks, 1)):
        di, dj = rng.integers(-hops, hops + 1, n), rng.integers(-hops, hops + 1, n)
        ni, nj = np.clip(ci + di, 0, gx), np.clip(cj + dj, 0, gy)
        same = (ni == ci) & (nj == cj)
        ni = np.where(same, np.where(ci < gx, ci + 1, ci - 1), ni)
        x_first = rng.random(n) < 0.5
        short = rng.uniform(0.02, 0.2, n)
        for e in range(n):
            # from where the robot stands (on the aisle into its crossing) to the crossing, along one
            # aisle and the other, and to a stop 2-20 cm short of the target crossing: a sampled
            # reference never lands on a route's last node, which get_global_ref_traj cannot walk past
            a, b = crossing(ci[e], cj[e]), crossing(ni[e], nj[e])
            corner = (b[0], a[1]) if x_first[e] else (a[0], b[1])
            nodes = [pos[e]]
            for q in (a, corner, b):
                if q != nodes[-1]:
                    nodes.append(q)
            (px_, py_), (bx, by) = nodes[-2], nodes[-1]
            L = float(np.hypot(bx - px_, by - py_))
            nodes[-1] = (bx - (bx - px_) / L * short[e], by - (by - py_) / L * short[e])
            pos[e] = nodes[-1]
            paths[e].append(nodes)
            goals[e].append((nodes[-1][0], nodes[-1][1], 0.0))
        ci, cj = ni, nj
    first = [p[0] for p in paths]
    off = rng.uniform(-0.05, 0.05, (n, 2))  # a parked robot stands a few cm off its spot
    init = np.array([[p[0][0] + off[e, 0], p[0][1] + off[e, 1], np.arctan2(p[1][1] - p[0][1], p[1][0] - p[0][0])]
                     for e, p in enumerate(first)])
    return dict(init=init, goal=np.array([g[0] for g in goals]), paths=first, world_polys=world,
                task_goals=[g[1:tasks] for g in goals], task_paths=[p[1:tasks] for p in paths],
                moving_pos=np.zeros((n, 0, 2)), moving_disp=np.zeros((n, 0, 2)))
