"""Obstacle-contact and tracking monitor of the fleet step (ttmpc_fleet_monitor_device) on the CPU:
the oracle's swept clearance against dense sampling with the fleet oracle's independent point
distance, hand-built contact and deviation cases, the ctypes layout of struct ttmpc_fleet_monitor,
the argument checks of the entry point and FleetPlanner.enable_monitor's set-up."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.fleet import COLLIDED, DYN_OBS_SIZE, REACHED, RUNNING, work_mode
from tests import oracle_lib as O
from tests import fleet_monitor_ref as R
from tests.fleet_action_steps_ref import FleetHostK
from tests.fleet_monitor_ref import BUFFERS, MonitorHost

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M = 10_000   # dense samples along a chord


def _star(rng, nv, convex):
    """A simple polygon: nv vertices at sorted angles, radius constant (convex) or random (non-convex)."""
    ang = np.sort(rng.uniform(0.0, 2 * np.pi, nv))
    rad = np.full(nv, 1.0) if convex else rng.uniform(0.3, 1.5, nv)
    return np.stack([rad * np.cos(ang), rad * np.sin(ang)], 1) * rng.uniform(0.5, 2.0) + rng.uniform(-1, 1, 2)


def _dense_poly(xy, p0, p1):
    s = np.linspace(0.0, 1.0, M)
    pts = np.asarray(p0)[None] + s[:, None] * (np.asarray(p1) - np.asarray(p0))[None]
    return min(O.poly_distance(xy, x, y) for x, y in pts)


# ------------------------------------------------------------------ independent geometry
@pytest.mark.parametrize("convex", [True, False])
def test_swept_polygon_distance_matches_dense_sampling(convex):
    rng = np.random.default_rng(1 if convex else 2)
    hits = 0
    for _ in range(40):
        xy = _star(rng, int(rng.integers(3, 9)), convex)
        p0 = rng.uniform(-4, 4, 2)
        p1 = p0 + rng.normal(0.0, 1.5, 2)
        got = R.swept_poly_distance(xy, p0, p1)
        dense = _dense_poly(xy, p0, p1)
        h = np.hypot(*(p1 - p0)) / (M - 1) / 2          # the sampled minimum overshoots by at most this
        assert dense - h - 1e-9 <= got <= dense + 1e-9, (xy.tolist(), p0, p1, got, dense)
        hits += got == 0.0
        # zero-length chord: the point distance, exactly
        assert R.swept_poly_distance(xy, p0, p0) == O.poly_distance(xy, *p0)
    assert 3 <= hits <= 37, hits     # both contact and clear chords were drawn


def test_swept_disc_distance_matches_dense_sampling():
    rng = np.random.default_rng(3)
    s = np.linspace(0.0, 1.0, M)[:, None]
    for _ in range(200):
        p0, c0 = rng.uniform(-3, 3, 2), rng.uniform(-3, 3, 2)
        p1, c1 = p0 + rng.normal(0, 1, 2), c0 + rng.normal(0, 1, 2)
        rel = (p0 - c0)[None] + s * ((p1 - c1) - (p0 - c0))[None]
        dense = np.hypot(rel[:, 0], rel[:, 1]).min()
        h = np.hypot(*((p1 - c1) - (p0 - c0))) / (M - 1) / 2
        got = R.swept_disc_distance(p0, p1, c0, c1)
        assert dense - h - 1e-9 <= got <= dense + 1e-9
    assert R.swept_disc_distance((1.0, 2.0), (1.0, 2.0), (4.0, 6.0), (4.0, 6.0)) == 5.0


# ------------------------------------------------------------------ hand-built cases
SQUARE = [(0.0, 0.0), (1.0, 0.0), (1.0, 1.0), (0.0, 1.0)]


def _fleet(starts, ends, status=RUNNING, ref=None, ref_len=None, idx=0, k=1, dyn_last=None, dyn_cur=None):
    """A FleetHostK whose robots moved from starts to ends in the step that just ran."""
    mc = t.Configurator()
    cfg = mc.to_ttmpc()
    n = len(ends)
    tuning, base = work_mode(mc, "work")
    ref = np.zeros((n, 8, 3)) if ref is None else np.asarray(ref, np.float64)
    ref_len = [ref.shape[1]] * n if ref_len is None else ref_len
    st = np.zeros((n, 3)); st[:, :2] = ends
    fh = FleetHostK(cfg, st, np.zeros((n, 3)), ref, ref_len, np.zeros(cfg.Nstcobs * cfg.nstcobs), tuning, base,
                    mc.low_speed, dyn_cur=dyn_cur, dyn_disp=None if dyn_cur is None else np.zeros_like(dyn_cur),
                    action_steps=k)
    if dyn_last is not None:
        fh.dyn_last[:] = dyn_last
    fh.status[:] = status
    fh.idx_ref[:] = idx
    mh = MonitorHost(np.c_[np.asarray(starts, np.float64), np.zeros(n)])
    return fh, mh


def _polys(polys, max_pv=4, nv=None):
    xy = np.zeros((1, len(polys), max_pv, 2))
    cnt = np.zeros((1, len(polys)), np.int32)
    for j, p in enumerate(polys):
        xy[0, j, :len(p)] = p
        cnt[0, j] = len(p) if nv is None else nv[j]
    return xy, cnt


def test_chord_clipping_a_corner_is_a_contact():
    p0, p1 = (-0.1, 0.9), (0.3, 1.2)       # enters through the left edge, leaves through the top one
    assert O.poly_distance(SQUARE, *p0) > 0.09 and O.poly_distance(SQUARE, *p1) > 0.19
    fh, mh = _fleet([p0], [p1])
    mh.poly_xy, mh.poly_nv = _polys([SQUARE])
    mh.run(fh, step=7)
    assert mh.clearance[0] == 0.0 and mh.contact_steps[0] == 1 and mh.first_contact[0] == 7
    fh2, mh2 = _fleet([p0, p1], [p0, p1])   # standing at either endpoint: clear
    mh2.poly_xy, mh2.poly_nv = mh.poly_xy, mh.poly_nv
    mh2.run(fh2, step=0)
    assert mh2.clearance == pytest.approx([0.1, 0.2]) and not mh2.contact_steps.any()
    assert (mh2.first_contact == -1).all()


def test_thin_wall_crossed_inside_one_step():
    wall = [(1.0, -2.0), (1.02, -2.0), (1.02, 2.0), (1.0, 2.0)]
    fh, mh = _fleet([(0.5, 0.0)], [(1.5, 0.0)])
    mh.poly_xy, mh.poly_nv = _polys([wall])
    mh.run(fh, step=0)
    assert mh.clearance[0] == 0.0 and mh.contact_steps[0] == 1
    assert O.poly_distance(wall, 0.5, 0.0) == pytest.approx(0.5) and O.poly_distance(wall, 1.5, 0.0) == pytest.approx(0.48)


def test_moving_disc_crossing_the_chord_between_samples():
    # the obstacle passes through the robot's path mid-step; at both ends it is 2 m away
    fh, mh = _fleet([(0.0, 0.0)], [(1.0, 0.0)], dyn_last=[[[0.5, 2.0]]], dyn_cur=np.array([[[0.5, -2.0]]]))
    mh.moving_radius = 0.1
    mh.run(fh, step=3)
    assert mh.clearance[0] == pytest.approx(-0.1) and mh.first_contact[0] == 3
    assert np.hypot(0.5, 2.0) - 0.1 > 1.9


def test_parked_robot_hit_by_a_moving_disc():
    fh, mh = _fleet([(0.0, 0.0)], [(0.0, 0.0)], status=REACHED, dyn_last=[[[1.0, 0.0]]],
                    dyn_cur=np.array([[[0.5, 0.0]]]))
    mh.moving_radius, mh.stop_on_contact = 0.6, True
    mh.run(fh, step=2)
    assert mh.clearance[0] == pytest.approx(-0.1) and mh.contact_steps[0] == 1 and mh.first_contact[0] == 2
    assert mh.moved_steps[0] == 0 and fh.status[0] == REACHED      # only a RUNNING robot becomes COLLIDED


def test_unused_slot_is_ignored_and_no_obstacle_is_infinite_clearance():
    fh, mh = _fleet([(0.2, 0.2)], [(0.5, 0.5)])
    mh.poly_xy, mh.poly_nv = _polys([SQUARE, SQUARE], nv=[2, 0])
    mh.run(fh, step=0)
    assert mh.clearance[0] == math.inf and mh.min_clearance[0] == math.inf and mh.contact_steps[0] == 0
    mh.poly_nv[0, 1] = 4
    mh.run(fh, step=1)
    assert mh.clearance[0] == 0.0 and mh.first_contact[0] == 1


def test_deviation_on_a_known_polyline():
    ref = np.zeros((1, 10, 3)); ref[0, :, 0] = np.arange(10.0)   # rows (i, 0)
    cases = [  # (idx_ref, k, ref_len, end position, deviation): the window is rows max(idx-k,0) .. min(idx+5k,L)-1
        (0, 1, 10, (6.0, 1.0), math.hypot(2.0, 1.0)),       # rows 0..4: past the window's far end
        (2, 1, 10, (2.5, 0.3), 0.3),
        (8, 1, 10, (3.0, 0.5), math.hypot(4.0, 0.5)),       # rows 7..9: before the window's near end
        (3, 2, 10, (0.0, 0.0), 1.0),                        # k = 2: rows 1..9
        (0, 1, 1, (3.0, 4.0), 5.0),                         # one row: the point distance
    ]
    for idx, k, L, end, want in cases:
        fh, mh = _fleet([(0.0, 0.0)], [end], ref=ref, ref_len=[L], idx=idx, k=k)
        mh.run(fh, step=0)
        mh.run(fh, step=1)                                  # a second moved step at the same place
        assert mh.deviation_max[0] == pytest.approx(want, abs=1e-15), (idx, k, L)
        assert mh.deviation_sum[0] == pytest.approx(2 * want, abs=1e-15) and mh.moved_steps[0] == 2
    fh, mh = _fleet([(0.0, 0.0)], [(6.0, 1.0)], status=REACHED, ref=ref)
    mh.run(fh, step=0)
    assert mh.moved_steps[0] == 0 and mh.deviation_sum[0] == 0.0 and mh.deviation_max[0] == 0.0


def test_stop_on_contact_only_with_the_flag():
    for stop in (False, True):
        fh, mh = _fleet([(-0.5, 0.5), (-0.5, 3.0)], [(0.5, 0.5), (0.5, 3.0)])
        mh.poly_xy, mh.poly_nv = _polys([SQUARE])
        mh.stop_on_contact = stop
        before = {k: v.copy() for k, v in vars(fh).items() if isinstance(v, np.ndarray)}
        mh.run(fh, step=0)
        assert mh.contact_steps.tolist() == [1, 0] and mh.moved_steps.tolist() == [1, 1]
        assert fh.status.tolist() == ([COLLIDED, RUNNING] if stop else [RUNNING, RUNNING])
        for k, v in before.items():        # the monitor writes nothing else of the fleet
            if k != "status":
                assert np.array_equal(getattr(fh, k), v), k
        assert np.array_equal(mh.prev_xy, fh.state[:, :2])


# ------------------------------------------------------------------ C-ABI
def test_fleet_monitor_struct_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    fields = [f for f, _ in _lib.TtmpcFleetMonitor._fields_]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "ttmpc.h"\nint main(void) {\n'
                   '  printf("%zu %d", sizeof(ttmpc_fleet_monitor), TTMPC_FLEET_COLLIDED);\n'
                   + "".join(f'  printf(" %zu", offsetof(ttmpc_fleet_monitor, {f}));\n' for f in fields)
                   + '  printf("\\n"); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    vals = list(map(int, subprocess.check_output([str(exe)]).split()))
    assert C.sizeof(_lib.TtmpcFleetMonitor) == vals[0]
    assert COLLIDED == vals[1] == 4
    assert [getattr(_lib.TtmpcFleetMonitor, f).offset for f in fields] == vals[2:]
    assert _lib.load().ttmpc_version() == 102


def test_monitor_argument_checks():
    lib = _lib.load()
    fh, mh = _fleet([(0.0, 0.0)] * 4, [(0.1, 0.0)] * 4)
    mh.poly_xy, mh.poly_nv = _polys([SQUARE])
    cfg = fh.cfg
    f = fh.struct()
    before = {name: getattr(mh, name).copy() for name in BUFFERS}
    status = fh.status.copy()

    def call(fleet=f, **kw):
        m = mh.struct()
        for key, v in kw.items():
            setattr(m, key, v)
        return lib.ttmpc_fleet_monitor_device(C.byref(cfg), None if fleet is None else C.byref(fleet),
                                              C.byref(m), None)

    BAD_ARG = -2
    assert lib.ttmpc_fleet_monitor_device(C.byref(cfg), C.byref(f), None, None) == BAD_ARG
    assert "monitor" in lib.ttmpc_last_error().decode()
    bad = [dict(**{name: None}) for name in BUFFERS]
    bad += [dict(poly_nv=None), dict(max_poly=-1), dict(max_pv=2), dict(robot_radius=-0.1),
            dict(moving_radius=-1.0), dict(robot_radius=math.inf), dict(moving_radius=math.nan),
            dict(robot_radius=math.nan)]
    for kw in bad:
        assert call(**kw) == BAD_ARG, kw
        assert "monitor" in lib.ttmpc_last_error().decode()
    # the fleet checks of the step
    for key, v in (("n", -1), ("state", None), ("ref_stride", 0), ("action_steps", 0), ("action_steps", 21)):
        g = fh.struct()
        setattr(g, key, v)
        assert call(fleet=g) == BAD_ARG, key
    assert call(fleet=None) == BAD_ARG
    for name in BUFFERS:
        assert np.array_equal(getattr(mh, name), before[name]), name
    assert np.array_equal(fh.status, status)


# ------------------------------------------------------------------ host side
def test_enable_monitor_defaults_and_buffers():
    mc = t.Configurator()
    fl = t.scenes.make_fleet(6, seed=4)
    fp = t.FleetPlanner(mc, fl["init"], fl["goal"], fl["paths"], mode="work", device="cpu")
    fp.enable_monitor()                                       # no static constraints yet: no polygons
    assert fp.monitor.poly_xy is None and fp.monitor.moving_radius == DYN_OBS_SIZE
    fp.update_static_constraints(fl["static_polys"], per_robot=True)
    fp.enable_monitor(robot_radius=0.3, stop_on_contact=True)
    m = fp.monitor
    assert m.poly_shared == 0 and (m.max_poly, m.max_pv) == (4, 4) and m.stop_on_contact == 1
    assert m.robot_radius == 0.3 and m.moving_radius == DYN_OBS_SIZE
    assert np.array_equal(fp.mon_poly_xy.numpy(), np.asarray(fl["static_polys"], np.float64))
    assert (fp.mon_poly_nv.numpy() == 4).all()
    assert np.array_equal(fp.prev_xy.numpy(), fl["init"][:, :2])
    assert np.isinf(fp.clearance.numpy()).all() and np.isinf(fp.min_clearance.numpy()).all()
    assert (fp.first_contact.numpy() == -1).all()
    for name in ("contact_steps", "deviation_max", "deviation_sum", "moved_steps"):
        assert not getattr(fp, name).numpy().any(), name
    for name in BUFFERS:
        assert getattr(m, name) == getattr(fp, name).data_ptr(), name
    shared = [[(0.0, 0.0), (1.0, 0.0), (0.5, 1.0)]]
    fp.enable_monitor(polygons=shared)
    assert fp.monitor.poly_shared == 1 and (fp.monitor.max_poly, fp.monitor.max_pv) == (1, 3)
    with pytest.raises(ValueError):
        fp.enable_monitor(robot_radius=-1.0)
    with pytest.raises(ValueError):
        fp.enable_monitor(polygons=[shared] * 2, per_robot=True)
