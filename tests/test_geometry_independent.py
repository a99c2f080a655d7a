"""Independent check of the shapely-dependent geometry (VERDICT r1 item 9).

shapely is absent here, so the sector / ray distances (csrc/ttdqn.cu, oracle/ttdqn_oracle.c:
edge clipping against the sector triangle, ray-edge intersection) and HintSwitcher's
`Polygon.contains` / `Polygon.distance` (csrc/ttmpc_fleet.cu, oracle/ttfleet_oracle.c: even-odd
crossing test, closest edge) were only ever compared with restatements by the same author.  These
tests use a DIFFERENT method -- dense sampling of the sets the reference intersects
(ext_obsv_sector_and_ray.py:44-66, main_pre.py:35-52) with a winding-number inside test -- and
compare to sampling accuracy.  The CUDA kernels equal the oracle functions checked here to 1e-9 /
bit for bit (tests/test_gpu_parity.py::test_dqn_observe_act_parity,
tests/test_gpu_fleet.py::test_hint_switch_on_device_matches_oracle).
"""
import math

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from tests import oracle_lib as O


def winding_inside(poly, pts):
    """Winding number != 0 (sum of signed angles), vectorised over points.  poly [nv,2], pts [m,2]."""
    a = poly[None, :, :] - pts[:, None, :]
    b = np.roll(poly, -1, axis=0)[None, :, :] - pts[:, None, :]
    ang = np.arctan2(a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0], a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1])
    return np.abs(ang.sum(axis=1)) > math.pi


def boundary_samples(poly, spacing):
    out = []
    for i in range(len(poly)):
        a, b = poly[i], poly[(i + 1) % len(poly)]
        m = max(2, int(np.linalg.norm(b - a) / spacing) + 2)
        out.append(a + (b - a) * np.linspace(0.0, 1.0, m)[:, None])
    return np.concatenate(out)


def brute_sector_ray(agent, rings, solid, ns=8, r_max=40.0, dr=2e-3, dth=2e-4, ray_length=None):
    """Reference semantics by sampling: segment i = wedge of half-width pi/ns around angle_i;
    closest point of wedge ^ geometry, first point of geometry along the centre ray.
    ray_length=L: segment i is the triangle with apex at the agent and far vertices at L (the wedge
    cut at L cos(pi/ns) along its centre line), the ray is L long, and a ring's ray hit counts only
    when the ring meets the triangle (ext_obsv_sector_and_ray.py looks for the ray hit only when the
    sector intersection is non-empty)."""
    ax, ay, ath = agent
    seg = np.full(ns, np.inf); ray = np.full(ns, np.inf)
    width = 2 * math.pi / ns
    rr = np.arange(dr, r_max if ray_length is None else ray_length, dr)
    for i in range(ns):
        ang = ath + i * width
        for poly, sd in zip(rings, solid):
            # ---- ray: first sample along the centre ray that is inside a solid polygon / crosses a ring
            pts = np.stack([ax + rr * math.cos(ang), ay + rr * math.sin(ang)], axis=1)
            ray_g = seg_g = np.inf
            inside = winding_inside(poly, pts)
            if sd:
                if winding_inside(poly, np.array([[ax, ay]]))[0]:
                    ray_g = 0.0
                elif inside.any():
                    ray_g = rr[np.argmax(inside)]
            else:  # LineString: the crossing of the boundary = a change of the inside flag
                start = winding_inside(poly, np.array([[ax, ay]]))[0]
                flips = np.nonzero(np.diff(np.concatenate([[start], inside]).astype(int)) != 0)[0]
                if len(flips):
                    ray_g = rr[flips[0]]
            # ---- sector: boundary points inside the wedge (the closest point of wedge ^ G lies on G's
            #      boundary when the agent is outside G) plus, for solid polygons, the wedge's own two
            #      edge rays entering the polygon
            if sd and winding_inside(poly, np.array([[ax, ay]]))[0]:
                seg_g = 0.0
            else:
                b = boundary_samples(poly, dr)
                rel = np.arctan2(b[:, 1] - ay, b[:, 0] - ax) - ang
                rel = (rel + math.pi) % (2 * math.pi) - math.pi
                inw = np.abs(rel) <= width / 2
                if ray_length is not None:      # the triangle: not beyond its far edge
                    inw &= (b[:, 0] - ax) * math.cos(ang) + (b[:, 1] - ay) * math.sin(ang) <= \
                        ray_length * math.cos(width / 2)
                if inw.any():
                    seg_g = np.hypot(b[inw, 0] - ax, b[inw, 1] - ay).min()
                if sd:
                    for edge_ang in (ang - width / 2, ang + width / 2):
                        e = np.stack([ax + rr * math.cos(edge_ang), ay + rr * math.sin(edge_ang)], axis=1)
                        ins = winding_inside(poly, e)
                        if ins.any():
                            seg_g = min(seg_g, rr[np.argmax(ins)])
            seg[i] = min(seg[i], seg_g)
            if ray_length is None or seg_g < np.inf:
                ray[i] = min(ray[i], ray_g)
    return seg, ray


def random_scene(rng):
    boundary = np.array([(0.0, 0.0), (20.0, 0.0), (20.0, 20.0), (0.0, 20.0)]) + rng.normal(0, 0.3, (4, 2))
    obs = []
    for _ in range(rng.integers(1, 4)):
        c = rng.uniform(4, 16, 2); h = rng.uniform(0.5, 2.0, 2); a = rng.uniform(0, np.pi)
        R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        sq = np.array([(-1, -1), (1, -1), (1, 1), (-1, 1)]) * h
        obs.append(t.geometry.pad_polygon_round(c + sq @ R.T, 0.5))
    # one concave (L-shaped) obstacle as well
    c = rng.uniform(5, 15, 2)
    L = np.array([(0, 0), (3, 0), (3, 1), (1, 1), (1, 3), (0, 3)], float) * rng.uniform(0.5, 1.0) + c
    obs.append(L)
    return obs + [boundary], [True] * len(obs) + [False]


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_sector_and_ray_distances_against_dense_sampling(seed):
    rng = np.random.default_rng(seed)
    rings, solid = random_scene(rng)
    lay = t.dqn.default_layout()
    # agents: free space, one inside an obstacle, one close to the boundary
    agents = [np.array([*rng.uniform(2, 18, 2), rng.uniform(-math.pi, math.pi)]) for _ in range(3)]
    agents.append(np.array([*rings[0].mean(axis=0), 0.3]))
    agents.append(np.array([0.8, 10.0, 1.0]))
    for e, ag in enumerate(agents):
        seg_o, ray_o = O.observe(lay, ag, rings, solid)
        seg_b, ray_b = brute_sector_ray(ag, rings, solid)
        tol = 6e-3 + 2e-4 * 40.0      # radial step + arc length of the angular step at r_max
        assert np.array_equal(np.isfinite(seg_o), np.isfinite(seg_b)), (seed, e, seg_o, seg_b)
        fin = np.isfinite(seg_o)
        assert np.abs(seg_o[fin] - seg_b[fin]).max() <= tol, (seed, e, seg_o, seg_b)
        assert np.array_equal(np.isfinite(ray_o), np.isfinite(ray_b)), (seed, e, ray_o, ray_b)
        finr = np.isfinite(ray_o)
        assert np.abs(ray_o[finr] - ray_b[finr]).max() <= tol, (seed, e, ray_o, ray_b)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_polygon_contains_and_distance_against_winding_number_and_sampling(seed):
    rng = np.random.default_rng(100 + seed)
    polys = [np.array([(0, 0), (4, 0), (4, 3), (0, 3)], float),
             np.array([(0, 0), (3, 0), (3, 1), (1, 1), (1, 3), (0, 3)], float),            # concave
             t.geometry.pad_polygon_round(np.array([(1., 1.), (1., 2.), (3., 2.), (3., 1.)]), 0.5)]
    for poly in polys:
        poly = poly + rng.uniform(-5, 5, 2)
        pts = rng.uniform(poly.min(axis=0) - 2.0, poly.max(axis=0) + 2.0, (400, 2))
        inside = winding_inside(poly, pts)
        b = boundary_samples(poly, 1e-3)
        for (px, py), ins in zip(pts, inside):
            d_b = 0.0 if ins else float(np.hypot(b[:, 0] - px, b[:, 1] - py).min())
            near_edge = float(np.hypot(b[:, 0] - px, b[:, 1] - py).min()) < 2e-3
            if not near_edge:
                assert O.poly_contains(poly, px, py) == bool(ins)
            assert abs(O.poly_distance(poly, px, py) - d_b) <= (2e-3 if not near_edge else 4e-3)
        # shapely: a point ON the boundary is not contained, its distance is 0
        v = poly[0]
        assert O.poly_distance(poly, *v) <= 1e-12


@pytest.mark.parametrize("ns", [3, 8])
def test_ray_length_rule_against_dense_sampling(ns):
    """Short rays (L = 3): obstacles on a centre ray between L cos(pi/ns) and L lie outside every
    sector triangle; the reference does not see them on the ray either.  Obstacles that reach into
    the triangle and cross the ray beyond it are seen on the ray."""
    from tests.dqn_exact_ref import band_square
    L = 3.0
    lay = t.dqn.default_layout()
    lay.num_segments, lay.ray_length = ns, L
    rng = np.random.default_rng(40 + ns)
    near = L * math.cos(math.pi / ns)
    seen_band = seen_reach = 0
    for k in range(3):
        ag = np.array([*rng.uniform(5, 15, 2), rng.uniform(-math.pi, math.pi)])
        rings = [band_square(ag, lay, s, 0.3 + 0.2 * k) for s in range(0, ns, 2)]
        # a thin bar from inside sector 1's triangle across its ray in the band
        a = ag[2] + 2 * math.pi / ns
        u, v = np.array([math.cos(a), math.sin(a)]), np.array([-math.sin(a), math.cos(a)])
        p1 = ag[:2] + u * (0.5 * (near + L))
        p2 = ag[:2] + u * (0.8 * near) + v * (0.3 * near * math.tan(math.pi / ns))
        p1 = p1 + 0.2 * (p1 - p2)
        nrm = np.array([-(p1 - p2)[1], (p1 - p2)[0]]) / np.hypot(*(p1 - p2)) * 0.01
        bar = np.array([p2 - nrm, p1 - nrm, p1 + nrm, p2 + nrm])
        rings.append(bar)
        solid = [True] * len(rings)
        seg_o, ray_o = O.observe(lay, ag, rings, solid)
        seg_b, ray_b = brute_sector_ray(ag, rings, solid, ns=ns, ray_length=L, dr=1e-3)
        tol = 3e-3 + 2e-4 * L
        for o, b in ((seg_o, seg_b), (ray_o, ray_b)):
            assert np.array_equal(np.isfinite(o), np.isfinite(b)), (ns, k, o, b)
            fin = np.isfinite(o)
            assert np.abs(o[fin] - b[fin]).max(initial=0.0) <= tol, (ns, k, o, b)
        seen_band += int(np.isinf(ray_o[0::2]).sum())
        seen_reach += int(np.isfinite(ray_o[1]) and ray_o[1] > near)
    assert seen_band >= 3 and seen_reach >= 1, (seen_band, seen_reach)
