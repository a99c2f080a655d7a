"""Scene content that ``scenes.make_scenes`` never produces, and a high-precision restatement of the
problem functions -- TEST INFRASTRUCTURE (a helper module, not a test file).

The builders take a parameter block ``p [n, np]`` (usually from ``make_scenes``), fill one block of it
in place and return it:

- ``with_other_robots``: predicted trajectories of other robots (the c block, robot-major,
  (x, y, theta) per step) -- head-on, crossing, parallel, parked at the live box, empty.
- ``with_static_polygons``: regular ne-gons in chosen slots of the static block, zero slots between.
- ``with_dynamic_obstacles``: constant-velocity ellipses in chosen slots of the dynamic block.
- ``with_folded_reference``: a reference path that turns back on itself.
- ``translate``: moves a whole scene rigidly.

``ref_eval`` computes f, F1 and F2 in ``np.longdouble`` (64-bit mantissa on x86), vectorised over
scenes: a plain restatement of oracle/ttmpc_oracle.c:forward(), i.e. of mpc_generator.py:155-283.
"""
from __future__ import annotations

import numpy as np

from trajtrack_mpcndqn_rlboost_b200.mpc_config import param_offsets

DYN_SLOTS = 4  # csrc/ttmpc_device.cuh: live dynamic obstacles whose table rows sit in shared memory


# ------------------------------------------------------------------ the kernel's live box
def box_half(cfg):
    """Half-width of the box around the start that every rollout with in-bounds controls stays in."""
    return 2.0 * cfg.N_hor * cfg.ts * max(abs(cfg.lin_vel_max), abs(cfg.lin_vel_min)) + 1.0


def robot_pad(cfg):
    """How far beyond the box an other robot still counts as live."""
    return cfg.vehicle_width * 1.001 + 1e-3


def ellipse_pad(cfg, rx, ry):
    """How far beyond the box a dynamic-obstacle record still counts as live."""
    m = cfg.social_margin
    return max(abs(rx + 1e-6), abs(ry + 1e-6), abs(rx + m + 1e-6), abs(ry + m + 1e-6)) * 1.001 + 1e-3


def _path(p, cfg):
    o = param_offsets(cfg)
    N = cfg.N_hor
    r = p[:, o["r"]:o["r"] + 3 * N].reshape(-1, N, 3)
    return r[..., 0], r[..., 1], r[..., 2]


# ------------------------------------------------------------------ builders
ROBOT_KINDS = ("headon", "crossing", "parallel", "parked_in", "parked_out", "empty")


def with_other_robots(p, cfg, rng, kinds):
    """Slot j of the c block gets a robot of kind kinds[j] (ROBOT_KINDS) in every scene:
    headon -- drives the reference path backwards from its end;
    crossing -- crosses the path at right angles, at a random sample, at that sample's step;
    parallel -- follows the path at a lateral offset below vehicle_width (contact at every step);
    parked_in / parked_out -- stands still just inside / just outside the live box (1e-3 m from it);
    empty -- left at the origin (zeros)."""
    assert len(kinds) <= cfg.Nother
    n, N = p.shape[0], cfg.N_hor
    o = param_offsets(cfg)
    rx, ry, rth = _path(p, cfg)
    x0, y0 = p[:, 0], p[:, 1]
    k = np.arange(N)[None, :]
    c = p[:, o["c"]:o["os"]].reshape(n, cfg.Nother, N, 3)
    for j, kind in enumerate(kinds):
        if kind == "headon":
            idx = np.broadcast_to(N - 1 - k, (n, N))
            lat = rng.normal(0.0, 0.1, (n, 1))
            h = np.take_along_axis(rth, idx, 1)
            x = np.take_along_axis(rx, idx, 1) - lat * np.sin(h)
            y = np.take_along_axis(ry, idx, 1) + lat * np.cos(h)
            th = h + np.pi
        elif kind == "crossing":
            m = rng.integers(0, N, n)
            mx, my, mh = rx[np.arange(n), m], ry[np.arange(n), m], rth[np.arange(n), m]
            speed = rng.uniform(0.8, 1.5, n) * cfg.ts * rng.choice([-1.0, 1.0], n)
            s = (k - m[:, None]) * speed[:, None]
            x = mx[:, None] - s * np.sin(mh)[:, None]
            y = my[:, None] + s * np.cos(mh)[:, None]
            th = np.broadcast_to((mh + np.pi / 2)[:, None], (n, N))
        elif kind == "parallel":
            lat = rng.choice([-1.0, 1.0], (n, 1)) * rng.uniform(0.3, 0.9, (n, 1)) * cfg.vehicle_width
            x = rx - lat * np.sin(rth)
            y = ry + lat * np.cos(rth)
            th = rth
        elif kind in ("parked_in", "parked_out"):
            edge = box_half(cfg) + robot_pad(cfg) + (-1e-3 if kind == "parked_in" else 1e-3)
            side = rng.choice([-1.0, 1.0], n) * edge
            along = rng.uniform(-0.5, 0.5, n) * box_half(cfg)
            on_x = rng.random(n) < 0.5
            x = np.broadcast_to((x0 + np.where(on_x, side, along))[:, None], (n, N))
            y = np.broadcast_to((y0 + np.where(on_x, along, side))[:, None], (n, N))
            th = np.zeros((n, N))
        elif kind == "empty":
            x = y = th = np.zeros((n, N))
        else:
            raise ValueError(kind)
        c[:, j, :, 0], c[:, j, :, 1], c[:, j, :, 2] = x, y, th
    p[:, o["c"]:o["os"]] = c.reshape(n, -1)
    return p


def regular_polygon_rows(cx, cy, R, phi, ne):
    """Half-space rows (b, a0, a1)[ne] of regular ne-gons (centre, circumradius R, first vertex at
    angle phi), scaled like geometry.polygon_halfspace_representation: a.(v - centre) = 1 on each
    edge, b - a0 x - a1 y > 0 inside.  Edges in counter-clockwise order from vertex 0."""
    cx, cy, R, phi = (np.asarray(v, np.float64)[..., None] for v in (cx, cy, R, phi))
    psi = phi + np.pi * (2 * np.arange(ne) + 1) / ne          # outward normal of edge e
    apothem = R * np.cos(np.pi / ne)
    a0, a1 = np.cos(psi) / apothem, np.sin(psi) / apothem
    return a0 * cx + a1 * cy + 1.0, a0, a1


def with_static_polygons(p, cfg, rng, ne, slots, straddle_fraction=0.35):
    """Regular ne-gons (circumradius 0.4-1.0 m) in the given static slots of every scene, the other
    slots left as they are (zero).  Centres lie near the reference path; a fraction of them straddle it.
    The obstacles come in overlapping triples (slots[0:3], slots[3:6], ...: centres within ~0.2 m),
    so that positions inside several obstacles at once make the order of their sums matter."""
    assert cfg.nstcobs == 3 * ne and max(slots) < cfg.Nstcobs
    n, N, ns = p.shape[0], cfg.N_hor, len(slots)
    o = param_offsets(cfg)
    rx, ry, rth = _path(p, cfg)
    m = rng.integers(min(2, N - 1), N, (n, ns))
    mx, my, mh = (np.take_along_axis(a, m, 1) for a in (rx, ry, rth))
    straddle = rng.random((n, ns)) < straddle_fraction
    side = np.where(straddle, rng.normal(0.0, 0.3, (n, ns)),
                    rng.choice([-1.0, 1.0], (n, ns)) * rng.uniform(1.0, 2.5, (n, ns)))
    cx = mx - side * np.sin(mh)
    cy = my + side * np.cos(mh)
    lead = np.arange(ns) // 3 * 3
    cx = cx[:, lead] + np.where(lead == np.arange(ns), 0.0, rng.normal(0.0, 0.15, (n, ns)))
    cy = cy[:, lead] + np.where(lead == np.arange(ns), 0.0, rng.normal(0.0, 0.15, (n, ns)))
    b, a0, a1 = regular_polygon_rows(cx, cy, rng.uniform(0.4, 1.0, (n, ns)), rng.uniform(0, 2 * np.pi, (n, ns)), ne)
    blk = p[:, o["os"]:o["od"]].reshape(n, cfg.Nstcobs, 3 * ne)
    blk[:, slots] = np.concatenate([b, a0, a1], axis=-1)
    p[:, o["os"]:o["od"]] = blk.reshape(n, -1)
    return p


def compact_static(p, cfg):
    """The same static obstacles moved to the first slots, order kept, zero slots after them."""
    o = param_offsets(cfg)
    n = p.shape[0]
    blk = p[:, o["os"]:o["od"]].reshape(n, cfg.Nstcobs, cfg.nstcobs)
    out = np.zeros_like(blk)
    for i in range(n):
        live = blk[i][np.any(blk[i] != 0.0, axis=1)]
        out[i, :len(live)] = live
    q = p.copy()
    q[:, o["os"]:o["od"]] = out.reshape(n, -1)
    return q


def with_dynamic_obstacles(p, cfg, rng, slots, boundary=()):
    """Constant-velocity ellipses (alpha = 1) in the given dynamic slots.  ``slots`` is one list for
    every scene or one list per scene.  The obstacles start 1-5 m along the path, up to 2.5 m to
    either side (closer for horizons under 14 steps).  Slots in ``boundary`` instead get an obstacle parked at the edge of the live
    box: alternately just inside and just outside it (1e-3 m from the edge, along x or y)."""
    n, N, ts = p.shape[0], cfg.N_hor, cfg.ts
    per_scene = [list(slots)] * n if np.ndim(slots[0]) == 0 else [list(s) for s in slots]
    o = param_offsets(cfg)
    od = p[:, o["od"]:o["qstc"]].reshape(n, cfg.Ndynobs, N, 6)
    _, _, rth = _path(p, cfg)
    x0, y0, h = p[:, 0], p[:, 1], rth[:, 0]
    steps = np.arange(1, N + 1)
    bh = box_half(cfg)
    reach = min(5.0, 1.0 + 1.5 * N * ts)       # 1-5 m ahead, +-2.5 m aside at the default horizon
    nb = 0
    for i in range(n):
        for j in per_scene[i]:
            rx_, ry_ = rng.uniform(0.2, 0.8, 2)
            ang = rng.uniform(0, np.pi)
            if j in boundary:
                edge = bh + ellipse_pad(cfg, rx_, ry_) + (-1e-3 if nb % 2 == 0 else 1e-3)
                nb += 1
                s = rng.choice([-1.0, 1.0]) * edge
                t = rng.uniform(-0.5, 0.5) * bh
                ex, ey = (x0[i] + s, y0[i] + t) if rng.random() < 0.5 else (x0[i] + t, y0[i] + s)
                ex, ey = np.full(N, ex), np.full(N, ey)
            else:
                along, side = rng.uniform(0.2 * reach, reach), rng.uniform(-0.5, 0.5) * reach
                ox = x0[i] + along * np.cos(h[i]) - side * np.sin(h[i])
                oy = y0[i] + along * np.sin(h[i]) + side * np.cos(h[i])
                vdir, vmag = rng.uniform(-np.pi, np.pi), rng.uniform(0.0, 1.0)
                ex = ox + vmag * np.cos(vdir) * ts * steps
                ey = oy + vmag * np.sin(vdir) * ts * steps
            od[i, j] = np.stack([ex, ey, np.full(N, rx_), np.full(N, ry_), np.full(N, ang), np.ones(N)], -1)
    p[:, o["od"]:o["qstc"]] = od.reshape(n, -1)
    return p


def with_folded_reference(p, cfg, lateral=0.25):
    """The reference path runs out along its first heading for half the horizon and comes back,
    ``lateral`` metres to the side the robot starts on.  Late samples then lie closer to the early
    positions than the early samples do, so the minimum over the remaining segments of the
    reference-path deviation is taken at segments far beyond the step."""
    n, N = p.shape[0], cfg.N_hor
    o = param_offsets(cfg)
    rx, ry, rth = _path(p, cfg)
    h = rth[:, 0]
    nx, ny = -np.sin(h), np.cos(h)
    bx, by = rx[:, 0] - 1.2 * cfg.ts * np.cos(h), ry[:, 0] - 1.2 * cfg.ts * np.sin(h)  # sample "-1"
    side = np.sign((p[:, 0] - bx) * nx + (p[:, 1] - by) * ny)
    side = np.where(side == 0, 1.0, side)
    K = (N + 1) // 2
    k = np.arange(1, N + 1)
    s = np.where(k <= K, k, 2 * K - k).astype(np.float64) * 1.2 * cfg.ts
    lat = np.where(k <= K, 0.0, lateral)[None, :] * side[:, None]
    r = np.stack([bx[:, None] + s * np.cos(h)[:, None] + lat * nx[:, None],
                  by[:, None] + s * np.sin(h)[:, None] + lat * ny[:, None],
                  np.where(k <= K, 0.0, np.pi)[None, :] + h[:, None]], -1)
    p[:, o["r"]:o["r"] + 3 * N] = r.reshape(n, -1)
    p[:, 3], p[:, 4], p[:, 5] = r[:, -1, 0], r[:, -1, 1], r[:, -1, 2]
    return p


def rollouts(cfg, u, p):
    """Positions of the rollouts of controls u [n, 2N] from each scene's start (oracle, libm): [n, N, 2]."""
    from tests import oracle_lib as O
    return np.stack([O.rollout(cfg, u[i], p[i])[:, :2] for i in range(len(p))])


def dyn_live(p, cfg):
    """[n, Ndyn] the kernel's live mask: some record of obstacle j lies within the live box."""
    n, N = p.shape[0], cfg.N_hor
    o = param_offsets(cfg)
    od = p[:, o["od"]:o["qstc"]].reshape(n, cfg.Ndynobs, N, 6)
    m = cfg.social_margin
    pad = np.maximum(np.maximum(np.abs(od[..., 2] + 1e-6), np.abs(od[..., 3] + 1e-6)),
                     np.maximum(np.abs(od[..., 2] + m + 1e-6), np.abs(od[..., 3] + m + 1e-6))) * 1.001 + 1e-3
    lim = box_half(cfg) + pad
    inside = (np.abs(od[..., 0] - p[:, 0, None, None]) <= lim) & (np.abs(od[..., 1] - p[:, 1, None, None]) <= lim)
    return inside.any(-1) | ~np.isfinite(od[..., :4]).all(-1).all(-1)


def park_on_rollout(p, cfg, xy, robot_slots, dyn_slots, rng):
    """Parks other robots and dynamic obstacles (r = 0.3 m circles) 0.2 m beside rollout positions
    xy [n, N, 2] that lie outside the live box, for all N steps: none of them is live, and only the
    out-of-box path (every slot scanned) sees them."""
    n, N = p.shape[0], cfg.N_hor
    o = param_offsets(cfg)
    lim = box_half(cfg) + max(robot_pad(cfg), ellipse_pad(cfg, 0.3, 0.3)) + 0.5
    far = np.maximum(np.abs(xy[..., 0] - p[:, 0, None]), np.abs(xy[..., 1] - p[:, 1, None])) > lim
    c = p[:, o["c"]:o["os"]].reshape(n, cfg.Nother, N, 3)
    od = p[:, o["od"]:o["qstc"]].reshape(n, cfg.Ndynobs, N, 6)
    for i in range(n):
        ks = np.flatnonzero(far[i])
        if not len(ks):
            continue
        for j in robot_slots:
            k = rng.choice(ks)
            c[i, j, :, 0], c[i, j, :, 1], c[i, j, :, 2] = xy[i, k, 0] + 0.2, xy[i, k, 1], 0.0
        for j in dyn_slots:
            k = rng.choice(ks)
            od[i, j] = [xy[i, k, 0], xy[i, k, 1] + 0.2, 0.3, 0.3, 0.0, 1.0]
    p[:, o["c"]:o["os"]] = c.reshape(n, -1)
    p[:, o["od"]:o["qstc"]] = od.reshape(n, -1)
    return p


def translate(p, cfg, dx, dy):
    """The same scenes moved rigidly by (dx, dy): start, goal, reference path, other robots, static
    half-spaces (b += a0 dx + a1 dy; zero slots stay zero) and dynamic centres."""
    q = np.array(p, np.float64, copy=True)
    n, N = q.shape[0], cfg.N_hor
    o = param_offsets(cfg)
    q[:, 0] += dx; q[:, 1] += dy; q[:, 3] += dx; q[:, 4] += dy
    r = q[:, o["r"]:o["r"] + 3 * N].reshape(n, N, 3)
    r[..., 0] += dx; r[..., 1] += dy
    c = q[:, o["c"]:o["os"]].reshape(n, cfg.Nother, N, 3)
    c[..., 0] += dx; c[..., 1] += dy
    ne = cfg.nstcobs // 3
    if cfg.Nstcobs and ne:
        s = q[:, o["os"]:o["od"]].reshape(n, cfg.Nstcobs, 3, ne)
        s[:, :, 0] += s[:, :, 1] * dx + s[:, :, 2] * dy
    d = q[:, o["od"]:o["qstc"]].reshape(n, cfg.Ndynobs, N, 6)
    d[..., 0] += dx; d[..., 1] += dy
    return q


# ------------------------------------------------------------------ high-precision reference
def ref_eval(cfg, u, p, terms=False):
    """f [n], F1 [n, 2N], F2 [n, Ndyn] in np.longdouble: oracle/ttmpc_oracle.c:forward() restated
    (mpc_generator.py:124-139 path deviation, 203-204 speed and control, 207-211 fleet collision,
    214-220 static, 225-237 dynamic, 242 terminal, 250-264 accelerations; F2_j = S + D_j).
    fmin / fmax where the C code uses them, so NaN inputs behave alike.

    terms=True also returns a dict of per-scene pieces: 'path', 'fleet', 'dyn_soft' [n, Ndyn],
    'S', 'D' [n, Ndyn], 'contacts' (other-robot contacts), and Lipschitz bounds of f and of F2 with
    respect to the rolled-out positions: 'lip_f' [n] and 'lip_F2' [n, Ndyn] (sums over the steps of
    |d term / d position|)."""
    L = np.longdouble
    p = np.asarray(p, np.float64).astype(L)
    u = np.asarray(u, np.float64).astype(L)
    if p.ndim == 1:
        p, u = p[None], u[None]
    n, N, ns = p.shape[0], cfg.N_hor, cfg.ns
    o = param_offsets(cfg)
    ts = L(cfg.ts)
    s, q = p[:, 0:8], p[:, o["q"]:o["q"] + 10]
    qvel, rv, rw, qN, qthN, qrpd, accp, waccp = (q[:, i] for i in (1, 3, 4, 5, 6, 7, 8, 9))
    r = p[:, o["r"]:o["r"] + ns * N].reshape(n, N, ns)
    vref = p[:, o["vref"]:o["vref"] + N]
    c = p[:, o["c"]:o["os"]].reshape(n, cfg.Nother, N, ns)
    ne = cfg.nstcobs // 3
    st = p[:, o["os"]:o["od"]].reshape(n, cfg.Nstcobs, 3, max(ne, 1)) if cfg.Nstcobs else None
    od = p[:, o["od"]:o["qstc"]].reshape(n, cfg.Ndynobs, N, 6)
    qdyn = p[:, o["qdyn"]:o["qdyn"] + N]
    v, w = u[:, 0::2], u[:, 1::2]

    # rollout: unicycle_model with rk4 (motion_model.py:153-176)
    X, Y, TH = (np.zeros((n, N), L) for _ in range(3))
    x, y, th = s[:, 0], s[:, 1], s[:, 2]
    for k in range(N):
        vk, wk = v[:, k], w[:, k]
        kx, ky, kt = [], [], []
        for a in (L(0), L(0.5), L(0.5), L(1)):
            t_ = th + a * (kt[-1] if kt else L(0))
            kx.append(ts * (vk * np.cos(t_))); ky.append(ts * (vk * np.sin(t_))); kt.append(ts * wk)
        x = x + (kx[0] + 2 * kx[1] + 2 * kx[2] + kx[3]) / 6
        y = y + (ky[0] + 2 * ky[1] + 2 * ky[2] + ky[3]) / 6
        th = th + (kt[0] + 2 * kt[1] + 2 * kt[2] + kt[3]) / 6
        X[:, k], Y[:, k], TH[:, k] = x, y, th

    # reference-path deviation: min over the segments j >= k of the path (last point duplicated)
    j2 = np.minimum(np.arange(N) + 1, N - 1)
    s1x, s1y = r[:, :, 0], r[:, :, 1]
    sx, sy = r[:, j2, 0] - s1x, r[:, j2, 1] - s1y                        # [n, j]
    den = sx * sx + sy * sy + L(1e-16)
    PX, PY = X[:, :, None] - s1x[:, None, :], Y[:, :, None] - s1y[:, None, :]   # [n, k, j]
    t_hat = (PX * sx[:, None, :] + PY * sy[:, None, :]) / den[:, None, :]
    tt = np.fmin(np.fmax(t_hat, L(0)), L(1))
    cx_, cy_ = tt * sx[:, None, :] - PX, tt * sy[:, None, :] - PY
    d2 = cx_ * cx_ + cy_ * cy_
    d2 = np.where(np.arange(N)[None, None, :] >= np.arange(N)[None, :, None], d2, L(np.nan))
    dmin = np.fmin.reduce(d2, axis=2)
    path = (dmin * qrpd[:, None]).sum(1)
    cost = path + (qvel[:, None] * (v - vref) ** 2).sum(1) + (rv[:, None] * v * v + rw[:, None] * w * w).sum(1)

    # fleet collision, safe distance vehicle_width, weight 1000
    dveh = L(cfg.vehicle_width)
    ex, ey = X[:, None, :] - c[..., 0], Y[:, None, :] - c[..., 1]     # [n, j, k]
    dd = ex * ex + ey * ey
    fl = np.fmax(L(0), dveh * dveh - dd)
    fleet = 1000 * fl.sum((1, 2))
    cost = cost + fleet

    # static obstacles: S = sum_k sum_i max(0, prod_e max(0, b - a0 x - a1 y)^2)
    if st is not None and ne:
        res = st[:, :, 0, None, :] - st[:, :, 1, None, :] * X[:, None, :, None] - st[:, :, 2, None, :] * Y[:, None, :, None]
        m = np.fmax(L(0), res)                                           # [n, i, k, e]
        S = np.fmax(L(0), (m * m).prod(-1)).sum((1, 2))
    else:
        S = np.zeros(n, L)

    # dynamic obstacles
    dx_, dy_ = X[:, None, :] - od[..., 0], Y[:, None, :] - od[..., 1]   # [n, j, k]
    ca, sa = np.cos(od[..., 4]), np.sin(od[..., 4])
    A = dx_ * ca + dy_ * sa
    B = dx_ * sa - dy_ * ca
    Rx, Ry = od[..., 2] + L(1e-6), od[..., 3] + L(1e-6)
    Rxm, Rym = od[..., 2] + L(cfg.social_margin) + L(1e-6), od[..., 3] + L(cfg.social_margin) + L(1e-6)
    in1 = 1 - A * A / (Rx * Rx) - B * B / (Ry * Ry)
    in2 = 1 - A * A / (Rxm * Rxm) - B * B / (Rym * Rym)
    D = np.fmax(L(0), in1).sum(2)
    m2 = np.fmax(L(0), in2)
    soft = (m2 * m2 * od[..., 5]) * qdyn[:, None, :]
    dyn_soft = soft.sum(2)
    cost = cost + dyn_soft.sum(1)

    # terminal cost and accelerations
    cost = cost + qN * ((X[:, -1] - s[:, 3]) ** 2 + (Y[:, -1] - s[:, 4]) ** 2) + qthN * (TH[:, -1] - s[:, 5]) ** 2
    vp = np.concatenate([s[:, 6:7], v[:, :-1]], 1)
    wp = np.concatenate([s[:, 7:8], w[:, :-1]], 1)
    a, aw = (v - vp) / ts, (w - wp) / ts
    cost = cost + (a * a).sum(1) * accp + (aw * aw).sum(1) * waccp
    F1 = np.concatenate([a, aw], 1)
    F2 = S[:, None] + D
    if not terms:
        return cost, F1, F2

    # Lipschitz bounds with respect to the positions (for error bounds at large coordinates)
    with np.errstate(invalid="ignore", divide="ignore"):
        lip_f = (2 * qrpd[:, None] * np.sqrt(dmin)).sum(1)
        lip_f = lip_f + 2000 * (np.sqrt(dd) * (fl > 0)).sum((1, 2))
        g2 = 2 * np.sqrt((A / (Rxm * Rxm)) ** 2 + (B / (Rym * Rym)) ** 2)
        lip_f = lip_f + (2 * m2 * od[..., 5] * qdyn[:, None, :] * g2).sum((1, 2))
        lip_f = lip_f + 2 * np.abs(qN) * np.hypot(X[:, -1] - s[:, 3], Y[:, -1] - s[:, 4])
        g1 = 2 * np.sqrt((A / (Rx * Rx)) ** 2 + (B / (Ry * Ry)) ** 2)
        lip_D = (g1 * (in1 > 0)).sum(2)
        if st is not None and ne:
            prod = (m * m).prod(-1)                                       # [n, i, k]
            an = np.sqrt(st[:, :, 1] ** 2 + st[:, :, 2] ** 2)[:, :, None, :]
            gS = (2 * np.where(m > 0, prod[..., None] / m, 0) * an).sum(-1)
            lip_S = gS.sum((1, 2))
        else:
            lip_S = np.zeros(n, L)
    jmin = np.argmin(np.where(np.isnan(d2), L(np.inf), d2), axis=2)   # first minimum, as the fold takes it
    parts = dict(path=path, fleet=fleet, dyn_soft=dyn_soft, S=S, D=D, contacts=(fl > 0).sum((1, 2)),
                 robot_contacts=(fl > 0).sum(2), jmin=jmin, lip_f=lip_f, lip_F2=lip_S[:, None] + lip_D)
    return cost, F1, F2, parts
