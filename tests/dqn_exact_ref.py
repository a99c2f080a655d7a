"""References for the DQN kernels (csrc/ttdqn.cu) at every layout and network shape -- TEST
INFRASTRUCTURE; the package never imports this module.

  cr_net             the Q-network correctly rounded: each neuron is the exact dot product plus bias
                     (integers scaled by 2^SCALE_BITS, so exact), rounded once to fp32 (nearest, ties
                     to even), then ReLU.
  fma_net            replica of the FMA-pipe path (observe_act_body, oracle linear_f32): fp64
                     accumulation in input order (every fp32 x fp32 product is exact in fp64), one
                     rounding to fp32, ReLU as `a < 0 ? 0 : a`.  The kernel equals it bit for bit.
  tc_bound           running-error bound of the tensor-core path (qnet_mma_kernel) against cr_net.
  sector_ray_hp      sector / ray distances of one environment in extended precision, with the
                     sector directions from mpmath at 50 digits, and for each sector the margin by
                     which every decision (edge meets triangle, ray meets edge, agent in ring) is
                     clear of flipping.
  shape_scene        scenes with rings of 2..65 vertices, empty ring slots and obstacles in the band
                     between L cos(pi / ns) and L, where only the ray-length rule decides.
"""
from __future__ import annotations

import math

import mpmath
import numpy as np

import trajtrack_mpcndqn_rlboost_b200 as t

# ------------------------------------------------------------------ Q-network references
SCALE_BITS = 320          # fp32 x fp32 products are multiples of 2^-298: exact integers at this scale

# Constant of the tensor-core bound.  qnet_mma_kernel sums each 8-term k-step of six TF32 products in
# the tensor core (fp32, truncating) and the k-steps with round-to-nearest FADDs, so its error per
# neuron is a few units of 2^-24 of sum |w x| + |b| at worst.  Measured on one NVIDIA B200 (1000 W power
# limit) with tests/test_gpu_dqn_shapes.py::test_random_16_wide_networks_on_both_paths, which prints it:
# the largest |q_tc - q_cr| / tc_bound(kappa=1) over 6..248 inputs and 1..16 outputs was 0.26 (8 inputs).
KAPPA = 1.0


def _round_f32(num: int, exp: int) -> float:
    """num * 2^exp (integers) rounded once to fp32, nearest, ties to even."""
    if num == 0:
        return 0.0
    sign = -1.0 if num < 0 else 1.0
    m = abs(num)
    top = m.bit_length() - 1 + exp                      # exponent of the leading bit
    keep = 24 if top >= -126 else 24 - (-126 - top)     # subnormal: fewer significant bits
    shift = m.bit_length() - keep
    if shift > 0:
        q, r = m >> shift, m & ((1 << shift) - 1)
        half = 1 << (shift - 1)
        if r > half or (r == half and (q & 1)):
            q += 1
        m, exp = q, exp + shift
    v = math.ldexp(float(m), exp)
    if v > float(np.finfo(np.float32).max):
        return sign * math.inf
    return sign * v


def _exact_ints(a64: np.ndarray) -> np.ndarray:
    """fp64 values that are multiples of 2^-SCALE_BITS -> Python ints of value * 2^SCALE_BITS, exactly."""
    out = np.empty(a64.shape, dtype=object)
    for idx, v in np.ndenumerate(a64):
        n, d = float(v).as_integer_ratio()             # d is a power of two <= 2^SCALE_BITS
        out[idx] = (n << SCALE_BITS) // d
    return out


def cr_layer(w, b, x, relu):
    """One layer, correctly rounded: y[r, o] = fp32(sum_i w[o, i] x[r, i] + b[o]) (ReLU if relu)."""
    w = np.asarray(w, np.float32).astype(np.float64)
    b = np.asarray(b, np.float32).astype(np.float64)
    x = np.asarray(x, np.float32).astype(np.float64)
    bi = _exact_ints(b)
    y = np.empty((x.shape[0], w.shape[0]), np.float32)
    for r in range(x.shape[0]):
        p = _exact_ints(w * x[r][None, :])              # exact products
        for o in range(w.shape[0]):
            v = _round_f32(sum(p[o].tolist(), bi[o]), -SCALE_BITS)
            y[r, o] = 0.0 if (relu and v < 0.0) else v
    return y


def cr_net(weights, x):
    w0, b0, w1, b1, w2, b2 = weights.arrays
    h1 = cr_layer(w0, b0, x, True)
    h2 = cr_layer(w1, b1, h1, True)
    return cr_layer(w2, b2, h2, False), (h1, h2)


def fma_layer(w, b, x, relu):
    w = np.asarray(w, np.float32).astype(np.float64)
    x = np.asarray(x, np.float32).astype(np.float64)
    a = np.broadcast_to(np.asarray(b, np.float32).astype(np.float64), (x.shape[0], w.shape[0])).copy()
    for i in range(w.shape[1]):
        a = a + w[:, i][None, :] * x[:, i][:, None]
    y = a.astype(np.float32)
    return np.where(y < 0, np.float32(0), y) if relu else y


def fma_net(weights, x):
    w0, b0, w1, b1, w2, b2 = weights.arrays
    h1 = fma_layer(w0, b0, x, True)
    h2 = fma_layer(w1, b1, h1, True)
    return fma_layer(w2, b2, h2, False)


def first_argmax(q):
    """First maximum of each row (torch.argmax, the kernels and the oracle fold with `>`)."""
    return np.argmax(q, axis=1).astype(np.int32)


def tc_bound(weights, x, hidden, kappa=KAPPA):
    """|q_tc - q_cr| bound per element: |dh_k| <= |W_k| |dh_{k-1}| + kappa 2^-24 (|W_k| |h_{k-1}| + |b_k|),
    dh_0 = 0 (the inputs are exact), h the correctly rounded activations (ReLU is 1-Lipschitz)."""
    u = kappa * 2.0 ** -24
    ws = [np.abs(a.astype(np.float64)) for a in weights.arrays]
    acts = [np.abs(np.asarray(x, np.float64))] + [np.abs(h.astype(np.float64)) for h in hidden]
    d = np.zeros_like(acts[0])
    for k in range(3):
        W, B = ws[2 * k], ws[2 * k + 1]
        d = d @ W.T + u * (acts[k] @ W.T + B[None, :])
    return d


def random_weights(rng, n_in, n_h1, n_h2, n_out, scale=1.0):
    """Random fp32 weights with He-like scaling and small biases."""
    w = []
    for a, b in ((n_in, n_h1), (n_h1, n_h2), (n_h2, n_out)):
        w.append(rng.normal(0, scale * math.sqrt(2.0 / a), (b, a)).astype(np.float32))
        w.append(rng.normal(0, 0.1, b).astype(np.float32))
    return t.dqn.QNetWeights(*w)


# ------------------------------------------------------------------ sector / ray reference
LD = np.longdouble


def _cross(ax, ay, bx, by):
    return ax * by - ay * bx


def _pseg_dist(px, py, ax, ay, bx, by):
    """Distance of points p to segments a-b (broadcast)."""
    dx, dy = bx - ax, by - ay
    dd = dx * dx + dy * dy
    with np.errstate(invalid="ignore", divide="ignore"):
        tt = np.where(dd > 0, ((px - ax) * dx + (py - ay) * dy) / np.where(dd > 0, dd, 1), 0)
    tt = np.clip(tt, 0, 1)
    qx, qy = ax + tt * dx - px, ay + tt * dy - py
    return np.sqrt(qx * qx + qy * qy)


def _segseg_dist(a0x, a0y, a1x, a1y, b0x, b0y, b1x, b1y):
    """Distance of non-crossing segments a, b: the least of the four endpoint-to-segment distances."""
    return np.minimum.reduce([_pseg_dist(a0x, a0y, b0x, b0y, b1x, b1y), _pseg_dist(a1x, a1y, b0x, b0y, b1x, b1y),
                              _pseg_dist(b0x, b0y, a0x, a0y, a1x, a1y), _pseg_dist(b1x, b1y, a0x, a0y, a1x, a1y)])


def sector_ray_hp(lay, agent, rings, solid, ray_rule=True):
    """(seg [ns], ray [ns], margin [ns]) of one environment.  The sector directions come from mpmath at
    50 digits (the fp64 angle th + i * width is formed as the kernels form it), everything after in
    x87 extended precision (64-bit significand): 1e-19 relative, far below the 1e-12 the comparisons
    use.  margin[i]: the least distance by which a decision of sector i could flip (an edge touching
    or leaving the triangle, the ray meeting an edge's end or the ray's end, the agent on a ring).
    ray_rule=False: every ring's ray hit counts, whether or not the ring meets the triangle (the rule
    the kernels had before they followed the reference)."""
    assert np.finfo(LD).nmant >= 63, "extended precision needed"
    ns, L = lay.num_segments, LD(lay.ray_length)
    ax, ay, th = (LD(float(v)) for v in agent)
    width = 2 * math.pi / ns
    rings = [np.asarray(r, np.float64).reshape(-1, 2) for r in rings]
    live = [(r, s) for r, s in zip(rings, solid) if len(r) >= 2]
    seg, ray, margin = np.full(ns, np.inf), np.full(ns, np.inf), np.full(ns, np.inf)
    if not live:
        return seg, ray, margin
    P0 = np.concatenate([r for r, _ in live]).astype(LD)
    P1 = np.concatenate([np.roll(r, -1, axis=0) for r, _ in live]).astype(LD)
    rid = np.concatenate([np.full(len(r), k) for k, (r, _) in enumerate(live)])
    p0x, p0y, p1x, p1y = P0[:, 0], P0[:, 1], P1[:, 0], P1[:, 1]
    dx, dy = p1x - p0x, p1y - p0y
    dlen = np.sqrt(dx * dx + dy * dy)
    # agent in a solid ring (even-odd), and how far it is from every ring
    agent_d = _pseg_dist(ax, ay, p0x, p0y, p1x, p1y).min()
    for k, (r, s) in enumerate(live):
        if not s:
            continue
        e = rid == k
        yi, yj, xi, xj = p1y[e], p0y[e], p1x[e], p0x[e]
        with np.errstate(invalid="ignore", divide="ignore"):
            c = ((yi > ay) != (yj > ay)) & (ax < (xj - xi) * (ay - yi) / (yj - yi) + xi)
        if c.sum() % 2:
            return np.zeros(ns), np.zeros(ns), np.full(ns, float(agent_d))
    mp = mpmath.mp
    for i in range(ns):
        angle = float(agent[2]) + i * width                       # fp64, as the kernels form it
        a1, a2 = angle - width / 2, angle + width / 2
        with mpmath.workdps(50):
            cs = [(LD(str(mp.cos(mpmath.mpf(a)))), LD(str(mp.sin(mpmath.mpf(a))))) for a in (a1, a2, angle)]
        V = [(ax, ay), (ax + L * cs[0][0], ay + L * cs[0][1]), (ax + L * cs[1][0], ay + L * cs[1][1])]
        rx, ry = cs[2]
        # Liang-Barsky clip of every edge against the triangle
        lo, hi = np.zeros(len(P0), LD), np.ones(len(P0), LD)
        empty = np.zeros(len(P0), bool)
        for a in range(3):
            b = (a + 1) % 3
            ex, ey = V[b][0] - V[a][0], V[b][1] - V[a][1]
            f0 = _cross(ex, ey, p0x - V[a][0], p0y - V[a][1])
            f1 = _cross(ex, ey, dx, dy)
            with np.errstate(invalid="ignore", divide="ignore"):
                tt = -f0 / f1
            empty |= (f1 == 0) & (f0 < 0)
            lo = np.where(f1 > 0, np.maximum(lo, tt), lo)
            hi = np.where(f1 < 0, np.minimum(hi, tt), hi)
        touch = ~empty & (lo <= hi)
        dd = dx * dx + dy * dy
        with np.errstate(invalid="ignore", divide="ignore"):
            tc = np.where(dd > 0, ((ax - p0x) * dx + (ay - p0y) * dy) / np.where(dd > 0, dd, 1), lo)
        tc = np.minimum(np.maximum(tc, lo), hi)
        qx, qy = p0x + tc * dx - ax, p0y + tc * dy - ay
        dist = np.where(touch, np.sqrt(qx * qx + qy * qy), LD(np.inf))
        tri_d = np.minimum.reduce([_segseg_dist(V[a][0], V[a][1], V[(a + 1) % 3][0], V[(a + 1) % 3][1],
                                                p0x, p0y, p1x, p1y) for a in range(3)])
        m_touch = np.where(touch, (hi - lo) * dlen, tri_d)
        # centre ray, length L
        wx, wy = p0x - ax, p0y - ay
        den = _cross(rx, ry, dx, dy)
        with np.errstate(invalid="ignore", divide="ignore"):
            s_ = _cross(wx, wy, dx, dy) / den
            t_ = _cross(wx, wy, rx, ry) / den
        hit = (den != 0) & (t_ >= 0) & (t_ <= 1) & (s_ >= 0) & (s_ <= L)
        s_hit = np.where(hit, s_, LD(np.inf))
        ray_d = _segseg_dist(ax, ay, ax + L * rx, ay + L * ry, p0x, p0y, p1x, p1y)
        m_ray = np.where(hit, np.minimum.reduce([t_ * dlen, (1 - t_) * dlen, L - s_]), ray_d)
        m_ray = np.where(den == 0, LD(0), m_ray)                 # parallel: never clear of flipping
        cseg = cray = LD(np.inf)
        for k in range(len(live)):
            e = rid == k
            if touch[e].any():                                    # the ring meets the triangle
                cseg = min(cseg, dist[e].min())
            if touch[e].any() or not ray_rule:
                cray = min(cray, s_hit[e].min())
        seg[i], ray[i] = float(cseg), float(cray)
        margin[i] = float(min(m_touch.min(), m_ray.min(), agent_d))
    return seg, ray, margin


# ------------------------------------------------------------------ scenes
RING_SIZES = (2, 3, 31, 32, 33, 64, 65)


def _ring(rng, c, rad, nv):
    if nv == 2:
        a = rng.uniform(0, np.pi)
        return c + rad * np.array([(math.cos(a), math.sin(a)), (-math.cos(a), -math.sin(a))])
    s = np.sort(rng.uniform(0, 2 * np.pi, nv)) if nv > 3 else np.array([0.0, 2.1, 4.2]) + rng.uniform(0, 1)
    r = rad * rng.uniform(0.6, 1.0, nv)
    return c + np.c_[r * np.cos(s), r * np.sin(s)]


def band_square(agent, lay, sector, frac=0.3):
    """A solid square on sector `sector`'s centre ray, wholly between L cos(pi / ns) and L: outside
    every sector triangle, crossing the ray before its end."""
    ns, L = lay.num_segments, lay.ray_length
    near = L * math.cos(math.pi / ns)
    h = 0.2 * (L - near) / 2
    s0 = near + frac * (L - near)
    ang = agent[2] + sector * 2 * math.pi / ns
    c = np.array([agent[0] + (s0 + h) * math.cos(ang), agent[1] + (s0 + h) * math.sin(ang)])
    u, v = np.array([math.cos(ang), math.sin(ang)]), np.array([-math.sin(ang), math.cos(ang)])
    return np.array([c - h * u - h * v, c + h * u - h * v, c + h * u + h * v, c - h * u + h * v])


SCENE_MAX_POLY, SCENE_MAX_VERT = 14, 320


def shape_scene(rng, n, lay):
    """n environments for `lay` (max_poly / max_vert must be at least SCENE_MAX_POLY / SCENE_MAX_VERT):
    rings of every size in RING_SIZES, empty slots (0 and 1 vertices) between used ones, environments
    with no ring and with every slot used, a boundary ring, and band squares (band_square)."""
    scenes, solid, agent = [], [], []
    for e in range(n):
        ag = np.array([*rng.uniform(2, 18, 2), rng.uniform(-np.pi, np.pi)])
        kind = e % 8
        rings, sd = [], []
        if kind == 0:                                            # no ring at all
            pass
        else:
            sizes = list(RING_SIZES) if kind == 1 else list(rng.choice(RING_SIZES, int(rng.integers(1, 4)), replace=False))
            for nv in sizes:
                if rng.uniform() < 0.3:                          # empty slot: 0 or 1 vertex
                    rings.append(np.zeros((int(rng.integers(0, 2)), 2)) + ag[:2] + 1.0)
                    sd.append(True)
                rad = rng.uniform(0.2, 2.5)
                rings.append(_ring(rng, rng.uniform(1, 19, 2), rad, int(nv)))
                sd.append(bool(nv >= 3 and rng.uniform() < 0.8))
            for _ in range(int(rng.integers(1, 3))):
                rings.append(band_square(ag, lay, int(rng.integers(0, lay.num_segments)), rng.uniform(0.1, 0.7)))
                sd.append(True)
            if rng.uniform() < 0.5:
                rings.append(np.array([(0.0, 0.0), (20.0, 0.0), (20.0, 20.0), (0.0, 20.0)]) + rng.normal(0, 0.2, (4, 2)))
                sd.append(False)
            if kind == 1:                                        # every slot used
                while len(rings) < lay.max_poly:
                    rings.append(np.zeros((0, 2))); sd.append(False)
            rings, sd = rings[:lay.max_poly], sd[:lay.max_poly]
        if kind == 2 and rings and sd[0] and len(rings[0]) >= 3:   # agent inside a solid ring
            ag[:2] = rings[0].mean(axis=0) if len(rings[0]) == 3 else ag[:2]
        scenes.append(rings); solid.append(sd); agent.append(ag)
    return scenes, solid, np.array(agent)
