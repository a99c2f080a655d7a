"""Moving obstacles in the DQN's lidar (ttdqn_observe_act_moving_device) and the DQN-boosted step run by
FleetPlanner.enable_dqn, on the GPU.

The moving rings must give exactly what the static path gives for the same rings (centre + offset,
formed in numpy) appended as static solid rings; the planner's DQN step must give exactly what the
hand-composed loop of tools/bench_hybrid.py gives."""
import ctypes as C
import os

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from trajtrack_mpcndqn_rlboost_b200.fleet import DYN_OBS_SIZE
from tests import oracle_lib as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def qnet():
    g = np.load(os.path.join(ROOT, "tests", "golden", "qnet_ray.npz"))
    return t.dqn.QNetWeights(*[g[k] for k in ("w0", "b0", "w1", "b1", "w2", "b2")]), g["internal"]


# ------------------------------------------------------------------ observe + act
def _static_scene(rng, n):
    """Each env: 1-3 padded rotated rectangles and a boundary ring (as tests/test_gpu_parity.py)."""
    rings, agent = [], []
    for _ in range(n):
        boundary = np.array([(0.0, 0.0), (20.0, 0.0), (20.0, 20.0), (0.0, 20.0)]) + rng.normal(0, 0.2, (4, 2))
        obs = []
        for _ in range(rng.integers(1, 4)):
            c = rng.uniform(3, 17, 2); h = rng.uniform(0.4, 2.0, 2); a = rng.uniform(0, np.pi)
            R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
            sq = np.array([(-1, -1), (1, -1), (1, 1), (-1, 1)]) * h
            obs.append(t.geometry.pad_polygon_round(c + sq @ R.T, 0.5))
        rings.append(obs + [boundary])
        agent.append([*rng.uniform(1, 19, 2), rng.uniform(-np.pi, np.pi)])
    return rings, np.array(agent)


def _ellipse(rng, nv=20):
    a, b, phi = rng.uniform(0.3, 2.0), rng.uniform(0.3, 2.0), rng.uniform(0, np.pi)
    s = np.linspace(0, 2 * np.pi, nv, endpoint=False)
    p = np.c_[a * np.cos(s), b * np.sin(s)]
    return p @ np.array([[np.cos(phi), -np.sin(phi)], [np.sin(phi), np.cos(phi)]]).T


# name: (moving obstacles k, vertex slots max_pv, shared templates)
CASES = dict(squares_shared=(2, 4, True), ellipses_per_env=(3, 20, False), mixed_two_passes=(5, 8, False),
             ten_squares_shared=(10, 4, True))


def _moving(rng, n, case):
    k, pv, shared = CASES[case]
    centre = rng.uniform(2, 18, (n, k, 2))
    blocks = 1 if shared else n
    xy = np.zeros((blocks, k, pv, 2))
    nv = np.zeros((blocks, k), np.int32)
    for b in range(blocks):
        for o in range(k):
            if case in ("squares_shared", "ten_squares_shared"):
                shape = t.dqn.rect_shape(DYN_OBS_SIZE if o % 2 == 0 else 0.6)
            elif case == "ellipses_per_env":
                shape = _ellipse(rng) if (b + o) % 7 else np.zeros((2, 2))          # some templates with nv < 3
            else:
                m = int(rng.choice([0, 1, 2, 3, 4, 6, 8]))
                shape = t.dqn.rect_shape(rng.uniform(0.3, 1.5)) if m == 4 else _ellipse(rng, m) if m else np.zeros((0, 2))
            xy[b, o, :len(shape)] = shape
            nv[b, o] = len(shape)
    return centre, xy, nv


def _place_agents(rng, agent, centre, xy, nv):
    """Agents inside a moving ring, on an edge, on a vertex, and with sector 0's centre ray (heading 0)
    collinear with an edge of a square; the rest where _static_scene put them.  Returns the agents and
    the mask of those placed on a ring's boundary."""
    n = len(agent)
    boundary = np.zeros(n, bool)
    for e in range(n):
        b = 0 if len(xy) == 1 else e
        seen = [o for o in range(centre.shape[1]) if nv[b, o] >= 3]
        if not seen:
            continue
        o = seen[e % len(seen)]
        c, r = centre[e, o], xy[b, o, :nv[b, o]]
        kind = e % 6
        if kind == 0:                                   # inside (the centroid of a convex template)
            agent[e, :2] = c + r.mean(axis=0)
        elif kind == 1:                                 # on a vertex: exactly the vertex the kernel forms
            agent[e, :2] = c + r[e % len(r)]
            boundary[e] = True
        elif kind == 2:                                 # on an edge
            v0, v1 = c + r[0], c + r[1]
            agent[e, :2] = v0 + 0.5 * (v1 - v0)
            boundary[e] = True
        elif kind == 3 and nv[b, o] == 4:               # centre ray of sector 0 along the bottom edge
            agent[e, :2] = (c[0] + r[0, 0] - rng.uniform(0.5, 3.0), c[1] + r[0, 1])
            agent[e, 2] = 0.0
    return agent, boundary


def _appended(static_rings, centre, xy, nv):
    rings, solid = [], []
    for e, st in enumerate(static_rings):
        b = 0 if len(xy) == 1 else e
        mv = [centre[e, o] + xy[b, o, :nv[b, o]] for o in range(centre.shape[1]) if nv[b, o] >= 3]
        rings.append(list(st) + mv)
        solid.append([True] * (len(st) - 1) + [False] + [True] * len(mv))
    return rings, solid


def _run(comp, qs, agent, geo, internal, old, moving=None, raw=None):
    import torch
    n = agent.shape[0]
    out = dict(ext=torch.zeros(n, 32, device="cuda"), q=torch.zeros(n, 9, device="cuda"),
               action=torch.full((n,), -1, dtype=torch.int32, device="cuda"),
               seg=torch.zeros(n, 8, dtype=torch.float64, device="cuda"), ray=torch.zeros(n, 8, dtype=torch.float64, device="cuda"))
    old = old.clone()
    if raw is None:
        comp.observe_act_device(agent, *geo, internal, old, out, qs, moving=moving)
    else:                                   # the moving entry point called directly, mv = raw
        dp = lambda x: x.data_ptr()
        rc = comp.lib.ttdqn_observe_act_moving_device(
            C.byref(comp.lay), C.byref(qs), n, dp(agent), *[dp(g) for g in geo], raw, dp(internal), dp(old),
            dp(out["ext"]), dp(out["q"]), dp(out["action"]), dp(out["seg"]), dp(out["ray"]),
            C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, comp.lib.ttdqn_last_error()
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["old_ext"] = old.cpu().numpy()
    return res


def _assert_same(a, b, what):
    for k in ("seg", "ray"):      # fp64 distances: equal as numbers (a zero may come out as -0 on either side)
        assert np.array_equal(a[k], b[k]), f"{k} differs ({what})"
    for k in ("ext", "q", "old_ext", "action"):
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), f"{k} differs ({what})"


def _setup(qnet, rng, n, case):
    import torch
    w, internal_g = qnet
    lay = t.dqn.default_layout(max_poly=16, max_vert=1024)
    static, agent = _static_scene(rng, n)
    centre, xy, nv = _moving(rng, n, case)
    agent, boundary = _place_agents(rng, agent, centre, xy, nv)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    geo = [cuda(a) for a in t.dqn.pack_geometry(lay, static, [[True] * (len(r) - 1) + [False] for r in static])]
    rings, solid = _appended(static, centre, xy, nv)
    app_np = t.dqn.pack_geometry(lay, rings, solid)
    internal = np.resize(internal_g, (n, 14)).astype(np.float32)
    old = rng.uniform(0, 1, (n, 16)).astype(np.float32)
    comp = t.dqn.DqnCompanion(lay, w)
    return dict(lay=lay, w=w, comp=comp, qs=w.device_struct(), agent_np=agent, agent=cuda(agent), geo=geo,
                app_np=app_np, app=[cuda(a) for a in app_np], internal_np=internal, internal=cuda(internal),
                old_np=old, old=cuda(old), moving=(cuda(centre), cuda(xy), cuda(nv)), nv=nv,
                boundary=boundary)


def test_no_moving_rings_equal_the_static_entry_point(qnet):
    """mv = NULL and n_live = 0: the new entry point computes what ttdqn_observe_act_device computes."""
    s = _setup(qnet, np.random.default_rng(11), 512, "squares_shared")
    ref = _run(s["comp"], s["qs"], s["agent"], s["geo"], s["internal"], s["old"])
    for mv in (None, C.byref(_lib.TtdqnMoving(0, 4, 1, 0, None, None, None)),
               C.byref(_lib.TtdqnMoving(0, 32, 0, 0, s["moving"][0].data_ptr(), None, None))):
        got = _run(s["comp"], s["qs"], s["agent"], s["geo"], s["internal"], s["old"], raw=mv)
        _assert_same(got, ref, f"mv {mv}")


@pytest.mark.parametrize("case", list(CASES))
def test_moving_rings_equal_appended_static_rings(qnet, case):
    """2048 random envs: moving rings == the same rings appended as static solid rings, bit for bit, and
    both within the parity tolerances of the CPU oracle on the appended geometry."""
    n = 2048
    s = _setup(qnet, np.random.default_rng(100 + list(CASES).index(case)), n, case)
    got = _run(s["comp"], s["qs"], s["agent"], s["geo"], s["internal"], s["old"], moving=s["moving"])
    want = _run(s["comp"], s["qs"], s["agent"], s["app"], s["internal"], s["old"])
    _assert_same(got, want, case)
    # the cases are there: agents inside a ring (all zeros), on a ring's boundary, several passes
    inside = (got["seg"] == 0).all(axis=1) & (got["ray"] == 0).all(axis=1)
    assert inside.sum() >= n // 12, inside.sum()
    k, pv, _ = CASES[case]
    assert k * pv > 32 or case == "squares_shared"
    if case != "squares_shared":
        assert (s["nv"] < 3).any() or case == "ten_squares_shared"
    # CPU oracle on the appended geometry (tolerances of tests/test_gpu_parity.py).  Not for agents on a
    # ring's boundary: an edge through the sector apex falls inside or outside a sector by the last ulp of
    # the sector's directions, which CUDA's and glibc's sin / cos may round differently (the static path
    # and the oracle differ there by whole metres; the bit-identity above covers those agents).
    ref = O.observe_act(s["lay"], s["w"], s["agent_np"], *s["app_np"], s["internal_np"], s["old_np"].copy())
    keep = ~s["boundary"]
    assert keep.sum() >= n // 2
    got = {k: v[keep] for k, v in got.items()}
    ref = {k: v[keep] for k, v in ref.items()}
    for key in ("seg", "ray"):
        fin = np.isfinite(ref[key])
        assert np.array_equal(fin, np.isfinite(got[key]))
        assert np.abs(got[key][fin] - ref[key][fin]).max() <= 1e-9
    assert np.abs(got["ext"] - ref["ext"]).max() <= 1e-6
    assert np.abs(got["q"] - ref["q"]).max() <= 2e-5
    srt = np.sort(ref["q"], axis=1)
    clear = (srt[:, -1] - srt[:, -2]) > 2e-5
    assert np.array_equal(got["action"][clear], ref["action"][clear])
    assert np.array_equal(got["old_ext"], ref["old_ext"])


def test_collinear_centre_ray_hits_the_edge_start(qnet):
    """Sector 0's centre ray runs along a moving square's bottom edge: the ray distance is the distance
    to the edge's near end, as for a static ring."""
    import torch
    w, internal_g = qnet
    lay = t.dqn.default_layout(max_poly=4, max_vert=16)
    n = 4
    r = DYN_OBS_SIZE
    centre = np.array([[[10.0, 10.0]]] * n)
    agent = np.array([[10.0 - r - d, 10.0 - r, 0.0] for d in (0.5, 1.0, 2.0, 4.0)])   # exact differences
    geo = [torch.from_numpy(a).cuda() for a in t.dqn.pack_geometry(lay, [[]] * n, [[]] * n)]
    moving = (torch.tensor(centre).cuda(), torch.tensor(t.dqn.rect_shape(r)[None, None]).cuda(),
              torch.tensor([[4]], dtype=torch.int32).cuda())
    internal = torch.from_numpy(np.resize(internal_g, (n, 14)).astype(np.float32)).cuda()
    got = _run(t.dqn.DqnCompanion(lay, w), w.device_struct(), torch.tensor(agent).cuda(), geo, internal,
               torch.zeros(n, 16, device="cuda"), moving=moving)
    assert np.array_equal(got["ray"][:, 0], [0.5, 1.0, 2.0, 4.0])


# ------------------------------------------------------------------ FleetPlanner.enable_dqn
def _lidar_rings(fl, n):
    """bench_hybrid's lidar geometry: each env's rectangles padded by 0.5 and a boundary ring."""
    rings, solid = [], []
    for i in range(n):
        r = [t.geometry.pad_polygon_round(np.array(poly), 0.5) for poly in fl["static_polys"][i]]
        x0, y0 = fl["init"][i, 0], fl["init"][i, 1]
        r.append(np.array([(x0 - 30, y0 - 30), (x0 + 30, y0 - 30), (x0 + 30, y0 + 30), (x0 - 30, y0 + 30)]))
        rings.append(r); solid.append([True] * (len(r) - 1) + [False])
    return rings, solid


class HandLoop:
    """tools/bench_hybrid.py's one_step, composed by hand; with rebuild=True the lidar geometry is
    packed on the host every step with the circle_to_rect squares appended at that step's dyn_cur."""

    def __init__(self, fp, w, rings, solid, paths, rebuild=False):
        import torch
        n = fp.n
        self.fp, self.rings, self.solid, self.rebuild = fp, rings, solid, rebuild
        self.lay = t.dqn.default_layout(max_poly=6 + (2 if rebuild else 0), max_vert=192 + (8 if rebuild else 0))
        self.geo = [torch.from_numpy(a).cuda() for a in t.dqn.pack_geometry(self.lay, rings, solid)]
        self.pxy, self.pcnt = paths
        self.comp, self.qs = t.dqn.DqnCompanion(self.lay, w), w.device_struct()
        self.old = torch.zeros(n, 16, dtype=torch.float32, device="cuda")
        self.out = dict(ext=torch.zeros(n, 32, device="cuda"), q=torch.zeros(n, 9, device="cuda"),
                        action=torch.zeros(n, dtype=torch.int32, device="cuda"))
        self.internal = torch.empty(n, 14, dtype=torch.float32, device="cuda")
        self.progress = torch.empty(n, dtype=torch.float64, device="cuda")
        self.rl = torch.empty(n, fp.N, 2, dtype=torch.float64, device="cuda")
        self.agent5 = torch.empty(n, 5, dtype=torch.float64, device="cuda")
        fp.set_hint(self.rl, torch.zeros(n, dtype=torch.int32, device="cuda"))

    def step(self, **kw):
        import torch
        fp = self.fp
        geo = self.geo
        if self.rebuild:
            cur = fp.dyn_cur.cpu().numpy()
            sq = t.dqn.rect_shape(DYN_OBS_SIZE)
            rings = [list(r) + [c + sq for c in cur[e]] for e, r in enumerate(self.rings)]
            solid = [list(s) + [True] * cur.shape[1] for s in self.solid]
            geo = [torch.from_numpy(a).cuda() for a in t.dqn.pack_geometry(self.lay, rings, solid)]
        self.agent5[:, :3] = fp.state; self.agent5[:, 3:] = fp.last_u
        t.dqn.internal_obs_device(self.agent5, self.pxy, self.pcnt, out=self.internal, progress=self.progress)
        self.comp.observe_act_device(fp.state, *geo, self.internal, self.old, self.out, self.qs)
        t.dqn.rl_ref_device(self.agent5, self.out["action"], steps=fp.N, ts=fp.config.ts, ref_speed=1.0, out=self.rl)
        fp.step(**kw)


FLEET = ("p", "u", "y", "cost", "exit_status", "inner", "pred_states", "state", "last_u", "idx_ref", "status",
         "goal", "ref_len", "ref_traj", "dyn_cur", "dyn_last", "use_hint", "sw_state", "hint")


def _drive(qnet, option, moving_shape, steps=40, n=64):
    import torch
    w, _ = qnet
    tasks = option == "tasks"
    fl = t.scenes.make_missions(n, 3, seed=61, max_static=4) if tasks else t.scenes.make_fleet(n, seed=60)
    if tasks:                                       # half the robots start at their first goal: they take task 2
        fl["init"][::2, :2] = fl["goal"][::2, :2] + 0.01
    rings, solid = _lidar_rings(fl, n)
    lay = t.dqn.default_layout(max_poly=6, max_vert=192)
    geo = [torch.from_numpy(a).cuda() for a in t.dqn.pack_geometry(lay, rings, solid)]
    m = max(len(q) for q in fl["paths"] + [q for pl in fl["task_paths"] for q in pl]) if tasks else None
    pxy, pcnt = t.dqn.pack_paths(fl["paths"], max_nodes=m)
    fps, loops = [], []
    for k in range(2):
        fp = t.FleetPlanner(t.Configurator(), fl["init"], fl["goal"], fl["paths"], mode="work",
                            max_inner_iterations=40, max_outer_iterations=3)
        fp.update_static_constraints(fl["static_polys"], per_robot=True)
        fp.set_moving_obstacles(fl["moving_pos"], fl["moving_disp"])
        paths = (torch.tensor(pxy).cuda(), torch.tensor(pcnt).cuda())
        if k == 0:
            fp.enable_hint_switch(fl["static_polys"], per_robot=True)
            fp.enable_dqn(w, geo, paths, moving_shape=moving_shape)
        else:
            loops.append(HandLoop(fp, w, rings, solid, paths, rebuild=moving_shape is not None))
            fp.enable_hint_switch(fl["static_polys"], per_robot=True)
        if tasks:
            fp.set_tasks(fl["task_goals"], fl["task_paths"], dqn_paths=None if k == 0 else paths)
        fps.append(fp)
    a, b = fps
    hand = loops[0]
    kw = dict(warm_start=True, skip_stopped=True) if option in ("warm_skip", "tasks") else {}
    hint_on = 0
    for s in range(steps):
        a.step(**kw)
        hand.step(**kw)
        torch.cuda.synchronize()
        for name in FLEET:
            assert torch.equal(getattr(a, name), getattr(b, name)), f"{name} differs at step {s}"
        assert torch.equal(a.dqn_action, hand.out["action"]), f"action differs at step {s}"
        assert torch.equal(a.dqn_q.view(torch.int32), hand.out["q"].view(torch.int32)), f"q differs at step {s}"
        assert torch.equal(a.dqn_ext.view(torch.int32), hand.out["ext"].view(torch.int32)), f"ext differs at step {s}"
        if tasks:
            assert torch.equal(a.task_next, b.task_next)
            assert all(torch.equal(x, y) for x, y in zip(a.dqn_paths, b.dqn_paths)), f"paths differ at step {s}"
        hint_on += int(a.use_hint.sum())
    assert hint_on > 0
    if tasks:
        assert int(a.task_next.sum()) > 0
    return a


@pytest.mark.parametrize("option", ["switch", "warm_skip", "tasks"])
def test_enable_dqn_blind_equals_the_hand_composed_loop(qnet, option):
    _drive(qnet, option, moving_shape=None)


def test_enable_dqn_rect_equals_a_loop_with_squares_appended_on_the_host(qnet):
    a = _drive(qnet, "switch", moving_shape="rect")
    assert a._dqn.shape_dev is not None and tuple(a._dqn.shape_dev[0].shape) == (1, 2, 4, 2)
