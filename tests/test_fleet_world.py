"""Shared obstacle map of the fleet step (ttmpc_fleet_world_select_device) on the CPU: the ctypes layout
of struct ttmpc_fleet_world, the argument checks of the entry point, the grid builder and query rule
on random maps, the brute-force oracle's selection against an independent Python selection, and the
host side of FleetPlanner.set_world and scenes.make_warehouse."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.fleet import world_grid, work_mode
from trajtrack_mpcndqn_rlboost_b200.geometry import convex_hull, polygon_halfspace_representation
from tests import oracle_lib as O
from tests.fleet_action_steps_ref import FleetHostK
from tests.fleet_world_ref import WorldHost, distance, python_select

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_ARG = -2


def _quad(cx, cy, hx, hy):
    return [(cx - hx, cy - hy), (cx + hx, cy - hy), (cx + hx, cy + hy), (cx - hx, cy + hy)]


def _rows(polys):
    out = []
    for p in polys:
        b, a0, a1 = polygon_halfspace_representation(np.array(p))
        out.append(b + a0 + a1)
    return np.array(out).reshape(len(polys), -1)


def _world(polys, reach, cell=None):
    hulls = np.array([convex_hull(np.array(p)) for p in polys]).reshape(len(polys), 4, 2)
    return WorldHost.from_hulls(hulls, _rows(polys) if polys else np.zeros((0, 12)), reach, cell)


def _random_quads(rng, M, span):
    """Random convex quadrilaterals (rotated rectangles) over [-span, span]^2, some overlapping."""
    polys = []
    for _ in range(M):
        c = rng.uniform(-span, span, 2)
        hx, hy, a = rng.uniform(0.1, 1.5), rng.uniform(0.1, 1.5), rng.uniform(0, np.pi)
        R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        polys.append((c + np.array([(-hx, -hy), (hx, -hy), (hx, hy), (-hx, hy)]) @ R.T).tolist())
    return polys


# ------------------------------------------------------------------ C-ABI
def test_fleet_world_struct_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    fields = [f for f, _ in _lib.TtmpcFleetWorld._fields_]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "ttmpc.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(ttmpc_fleet_world));\n'
                   + "".join(f'  printf(" %zu", offsetof(ttmpc_fleet_world, {f}));\n' for f in fields)
                   + '  printf("\\n"); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    vals = list(map(int, subprocess.check_output([str(exe)]).split()))
    assert C.sizeof(_lib.TtmpcFleetWorld) == vals[0]
    assert [getattr(_lib.TtmpcFleetWorld, f).offset for f in fields] == vals[1:]
    assert _lib.load().ttmpc_version() == 102


def test_world_select_argument_checks():
    lib = _lib.load()
    mc = t.Configurator()
    cfg = mc.to_ttmpc()
    tuning, base = work_mode(mc, "work")
    n = 4
    fh = FleetHostK(cfg, np.zeros((n, 3)), np.zeros((n, 3)), np.zeros((n, 8, 3)), [8] * n,
                    np.zeros(cfg.Nstcobs * cfg.nstcobs), tuning, base, mc.low_speed)
    wh = _world([_quad(0, 0, 1, 1), _quad(3, 0, 1, 1)], 6.0)
    K = cfg.Nstcobs
    stc = np.full((n, K * cfg.nstcobs), 7.0)
    slots = np.full((n, K), 7, np.int32)
    reach = np.full(n, 7, np.int32)

    def call(fleet=fh.struct(), world="default", out=stc.ctypes.data, **kw):
        w = wh.struct()
        for key, v in kw.items():
            setattr(w, key, v)
        w = None if world is None else C.byref(w)
        return lib.ttmpc_fleet_world_select_device(C.byref(cfg), None if fleet is None else C.byref(fleet), w, out,
                                                   slots.ctypes.data, reach.ctypes.data, None)

    bad = [dict(world=None), dict(M=-1), dict(max_pv=2), dict(reach=0.0), dict(reach=-1.0), dict(reach=math.inf),
           dict(reach=math.nan), dict(cell=0.0), dict(cell=-2.0), dict(cell=math.inf), dict(cell=math.nan),
           dict(nx=0), dict(ny=0), dict(nx=1 << 16, ny=1 << 16), dict(out=None)]
    bad += [{name: None} for name in ("poly_xy", "poly_nv", "rows", "bbox", "cell_start", "cell_items")]
    for kw in bad:
        assert call(**kw) == BAD_ARG, kw
        assert "world" in lib.ttmpc_last_error().decode(), kw
    for key, v in (("n", -1), ("state", None), ("ref_stride", 0)):     # the fleet checks of the step
        g = fh.struct()
        setattr(g, key, v)
        assert call(fleet=g) == BAD_ARG, key
    assert call(fleet=None) == BAD_ARG
    assert (stc == 7.0).all() and (slots == 7).all() and (reach == 7).all()
    # no robot: nothing to do; an empty map needs no arrays
    g = fh.struct()
    g.n = 0
    assert call(fleet=g) == 0
    assert call(fleet=g, M=0, poly_xy=None, poly_nv=None, rows=None, bbox=None, cell_start=None, cell_items=None) == 0


# ------------------------------------------------------------------ grid builder and query rule
@pytest.mark.parametrize("seed,M,reach,cell_frac", [(1, 200, 6.0, 1.0), (2, 500, 2.0, 0.5), (3, 300, 3.0, 1 / 3),
                                                    (4, 50, 0.75, 0.25), (5, 400, 5.0, 2.0)])
def test_grid_lists_each_polygon_in_its_box_cells_and_the_query_misses_none(seed, M, reach, cell_frac):
    rng = np.random.default_rng(seed)
    polys = _random_quads(rng, M, 30.0)
    wh = _world(polys, reach, reach * cell_frac)
    ox, oy, cell, nx, ny = wh.origin_x, wh.origin_y, wh.cell, wh.nx, wh.ny
    assert ox == wh.bbox[:, 0].min() and oy == wh.bbox[:, 1].min()
    assert wh.bbox[:, 2].max() < ox + nx * cell and wh.bbox[:, 3].max() < oy + ny * cell
    # the grid: polygon o in exactly the cells its box overlaps, ascending within a cell
    listed = {}
    for c in range(nx * ny):
        items = wh.cell_items[wh.cell_start[c]:wh.cell_start[c + 1]].tolist()
        assert items == sorted(set(items))
        for o in items:
            listed.setdefault(o, set()).add(c)
    for o, bb in enumerate(wh.bbox):
        x0, x1 = (min(int(math.floor((v - ox) / cell)), nx - 1) for v in (bb[0], bb[2]))
        y0, y1 = (min(int(math.floor((v - oy) / cell)), ny - 1) for v in (bb[1], bb[3]))
        assert listed[o] == {cy * nx + cx for cy in range(y0, y1 + 1) for cx in range(x0, x1 + 1)}, o
    # query points: random, outside the grid, on cell boundaries (with R a multiple of the cell: also
    # the query square's edges), on polygon vertices
    pts = list(rng.uniform(-45, 45, (300, 2)))
    pts += [(ox + i * cell, oy + j * cell) for i in range(-2, nx + 3, 3) for j in range(-2, ny + 3, 3)]
    pts += [(ox - reach - cell * 1.5, 0.0), (ox + nx * cell + reach, oy), (1e6, -1e6)]
    pts += [tuple(p[0]) for p in polys[:20]]
    misses = found = 0
    for x, y in pts:
        q = wh.query(x, y)
        assert len(q) == len(set(q)), (x, y)                            # each polygon once
        near = {o for o in range(M) if distance(wh.poly_xy[o], x, y) <= reach}
        misses += len(near - set(q))
        found += len(near)
    assert misses == 0 and found > 100, (misses, found)


def test_grid_of_an_empty_map_and_of_one_point_sized_polygon():
    assert world_grid(np.zeros((0, 4)), 1.0)[2:4] == (1, 1)
    ox, oy, nx, ny, start, items = world_grid(np.array([[2.0, 3.0, 2.0, 3.0]]), 1.0)
    assert (ox, oy, nx, ny) == (2.0, 3.0, 1, 1) and start.tolist() == [0, 1] and items.tolist() == [0]
    with pytest.raises(ValueError):
        world_grid(np.array([[0.0, 0.0, 1e6, 1e6]]), 1e-3)


# ------------------------------------------------------------------ the oracle's selection
def _check_selection(wh, cfg, pts):
    state = np.zeros((len(pts), 3))
    state[:, :2] = pts
    stc, slots, n_reach = wh.select(cfg, state)
    K, ns = cfg.Nstcobs, cfg.nstcobs
    for e, (x, y) in enumerate(pts):
        dist = [distance(wh.poly_xy[o], x, y) for o in range(wh.M)]
        want, n_elig = python_select(dist, wh.reach, K)
        assert n_reach[e] == n_elig
        assert slots[e].tolist() == want + [-1] * (K - len(want)), (e, slots[e], want)
        rows = np.zeros((K, ns))
        for s, o in enumerate(want):
            rows[s] = wh.rows[o]
        assert np.array_equal(stc[e].reshape(K, ns), rows)
    return stc, slots, n_reach


def test_oracle_distance_is_the_fleet_oracles_polygon_distance():
    rng = np.random.default_rng(8)
    for p in _random_quads(rng, 50, 3.0):
        hull = convex_hull(np.array(p))
        for x, y in rng.uniform(-5, 5, (10, 2)):
            assert distance(hull, x, y) == O.poly_distance(hull, x, y)


def test_selection_ties_inside_overlapping_polygons():
    cfg = t.Configurator().to_ttmpc()
    cfg.Nstcobs = 2
    polys = [_quad(0, 0, 2, 2), _quad(5, 0, 1, 1), _quad(0.5, 0, 1, 1), _quad(-0.5, 0.2, 1, 1)]
    wh = _world(polys, 6.0)
    _, slots, n_reach = _check_selection(wh, cfg, [(0.0, 0.0)])
    assert slots[0].tolist() == [0, 2] and n_reach[0] == 4           # three at d = 0: the two lowest indices


def test_selection_symmetric_placements():
    cfg = t.Configurator().to_ttmpc()
    cfg.Nstcobs = 3
    polys = [_quad(3, 0, 1, 1), _quad(0, 3, 1, 1), _quad(-3, 0, 1, 1), _quad(0, -3, 1, 1), _quad(0, 0, 0.25, 0.25)]
    wh = _world(polys, 6.0)
    d = [distance(wh.poly_xy[o], 0.5, 0.5) for o in range(4)]
    assert d[0] == d[1] and d[2] == d[3] and d[0] < d[2]
    _, slots, _ = _check_selection(wh, cfg, [(0.5, 0.5), (0.0, 0.0), (-0.5, -0.5)])
    assert slots[0].tolist() == [0, 1, 4] and slots[2].tolist() == [2, 3, 4]
    assert slots[1].tolist() == [0, 1, 4]                               # four at the same distance: lowest indices


def test_selection_polygon_at_exactly_reach():
    cfg = t.Configurator().to_ttmpc()
    R = 2.0
    eps = 2.0 ** -20
    polys = [[(R, -0.5), (R + 1, -0.5), (R + 1, 0.5), (R, 0.5)],                     # d = R exactly
             [(-R - 1 - eps, -0.5), (-R - eps, -0.5), (-R - eps, 0.5), (-R - 1 - eps, 0.5)]]   # d = R + 2^-20
    wh = _world(polys, R, cell=0.5)
    assert distance(wh.poly_xy[0], 0.0, 0.0) == R and distance(wh.poly_xy[1], 0.0, 0.0) == R + eps
    _, slots, n_reach = _check_selection(wh, cfg, [(0.0, 0.0)])
    assert slots[0, 0] == 0 and slots[0, 1] == -1 and n_reach[0] == 1
    assert 0 in wh.query(0.0, 0.0)


@pytest.mark.parametrize("M", [0, 3, 400])
def test_selection_map_sizes(M):
    cfg = t.Configurator().to_ttmpc()
    rng = np.random.default_rng(M)
    polys = _random_quads(rng, M, 2.0 if M < 10 else 25.0)
    wh = _world(polys, 6.0)
    pts = rng.uniform(-30, 30, (120, 2))
    _, slots, n_reach = _check_selection(wh, cfg, pts)
    if M == 400:
        assert (n_reach > cfg.Nstcobs).sum() > 10 and (n_reach == 0).sum() > 0
        # the kernel's candidates: the grid query gives every eligible polygon
        for x, y in pts:
            q = set(wh.query(x, y))
            assert all(o in q for o in range(M) if distance(wh.poly_xy[o], x, y) <= 6.0)


# ------------------------------------------------------------------ host side
def _planner(n=6, device="cpu"):
    mc = t.Configurator()
    fl = t.scenes.make_fleet(n, seed=4)
    return t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", device=device), fl


def test_set_world_rows_grid_and_edge_count_check():
    fp, fl = _planner()
    polys = [_quad(10, 10, 1, 2), [(0, 0), (2, 0), (2, 1), (1, 1.5), (0, 1)], _quad(30, 5, 0.5, 0.5)]
    with pytest.raises(ValueError, match="5 edges"):
        fp.set_world(polys)
    with pytest.raises(ValueError, match="3 edges"):
        fp.set_world([[(0, 0), (1, 0), (0, 1)]])
    with pytest.raises(ValueError, match="3 edges"):                 # a collinear vertex leaves the hull
        fp.set_world([[(0, 0), (1, 0), (2, 0), (2, 2), (0, 2)][:4] + [(1, 0)]])
    with pytest.raises(ValueError):
        fp.set_world([_quad(0, 0, 1, 1)], reach=0.0)
    with pytest.raises(ValueError):
        fp.set_world([_quad(0, 0, 1, 1)], cell=math.nan)
    assert fp.world is None
    polys[1] = [(0, 0), (2, 0), (2, 1), (0, 1.5), (1, 0.5)]            # its hull has 4 edges
    fp.set_world(polys)
    w = fp.world
    assert w.M == 3 and w.max_pv == 4 and w.reach == 6.0 and w.cell == 6.0
    assert np.array_equal(fp.world_rows.numpy(), _rows(polys))
    hulls = np.array([convex_hull(np.array(p)) for p in polys])
    assert np.array_equal(fp.world_poly_xy.numpy(), hulls) and (fp.world_poly_nv.numpy() == 4).all()
    assert np.array_equal(fp.world_bbox.numpy(), np.concatenate([hulls.min(1), hulls.max(1)], 1))
    ox, oy, nx, ny, start, items = world_grid(fp.world_bbox.numpy(), 6.0)
    assert (w.origin_x, w.origin_y, w.nx, w.ny) == (ox, oy, nx, ny)
    assert np.array_equal(fp.world_cell_start.numpy(), start) and np.array_equal(fp.world_cell_items.numpy(), items)
    assert fp.stc_shared == 0 and tuple(fp.stc.shape) == (fp.n, 120)
    assert tuple(fp.world_slots.shape) == (fp.n, 10) and tuple(fp.world_reach.shape) == (fp.n,)
    fp.set_world(polys, reach=2.5, cell=1.0)
    assert (fp.world.reach, fp.world.cell) == (2.5, 1.0)
    fp.set_world([])
    assert fp.world.M == 0 and not fp.world.poly_xy


def test_update_static_constraints_and_set_world_none_turn_the_map_off():
    fp, fl = _planner()
    fp.set_world([_quad(10, 10, 1, 2)])
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    assert fp.world is None and fp.stc_shared == 0 and fp.static_polys is not None
    fp.set_world([_quad(10, 10, 1, 2)])
    assert fp.static_polys is None
    fp.set_world(None)
    assert fp.world is None and fp.stc_shared == 1 and not fp.stc.any() and tuple(fp.stc.shape) == (1, 120)
    with pytest.raises(RuntimeError):
        fp.run_world_select()


def test_enable_monitor_defaults_to_the_map():
    fp, fl = _planner()
    polys = [_quad(10, 10, 1, 2), _quad(14, 10, 1, 2)]
    fp.set_world(polys)
    fp.enable_monitor()
    m = fp.monitor
    assert m.poly_shared == 1 and (m.max_poly, m.max_pv) == (2, 4)
    assert m.poly_xy == fp.world_poly_xy.data_ptr() and m.poly_nv == fp.world_poly_nv.data_ptr()
    assert np.array_equal(fp.mon_poly_xy.numpy()[0], fp.world_poly_xy.numpy())
    fp.enable_monitor(polygons=[_quad(0, 0, 1, 1)] * 3)            # polygons given: those
    assert fp.monitor.max_poly == 3
    fp.set_world([])
    fp.enable_monitor()
    assert fp.monitor.poly_xy is None


def test_make_warehouse_routes_keep_their_clearance():
    aisle = 3.0
    wh = t.scenes.make_warehouse(64, 4, seed=3, shelves=400, aisle=aisle)
    shelves = np.array(wh["world_polys"])
    assert len(shelves) == 400
    lo, hi = shelves.min(1), shelves.max(1)
    assert len(wh["task_goals"][0]) == 3 and len(wh["task_paths"][0]) == 3
    for e in range(64):
        chain = [wh["paths"][e]] + wh["task_paths"][e]
        goals = [wh["goal"][e]] + list(wh["task_goals"][e])
        assert np.abs(wh["init"][e, :2] - chain[0][0]).max() <= 0.05
        for k, path in enumerate(chain):
            nodes = np.array(path)
            assert np.allclose(nodes[-1], goals[k][:2])
            if k:
                assert np.allclose(nodes[0], goals[k - 1][:2])
            assert len(nodes) >= 2 and (np.hypot(*np.diff(nodes, axis=0).T) > 0).all()
            for a, b in zip(nodes[:-1], nodes[1:]):
                assert a[0] == b[0] or a[1] == b[1]                     # along an aisle
                s = np.linspace(0.0, 1.0, 200)[:, None]
                p = a + s * (b - a)                                     # samples of the leg
                dx = np.maximum(np.maximum(lo[None, :, 0] - p[:, None, 0], p[:, None, 0] - hi[None, :, 0]), 0)
                dy = np.maximum(np.maximum(lo[None, :, 1] - p[:, None, 1], p[:, None, 1] - hi[None, :, 1]), 0)
                assert np.hypot(dx, dy).min() >= aisle / 2 - 1e-9
    # the same density at any size
    big = t.scenes.make_warehouse(2, 1, seed=3, shelves=40_000, aisle=aisle)
    area = lambda w: np.ptp(np.array(w["world_polys"])[:, :, 0]) * np.ptp(np.array(w["world_polys"])[:, :, 1])
    assert abs(len(big["world_polys"]) / area(big) / (400 / area(wh)) - 1) < 0.1
