"""The DQN kernels (csrc/ttdqn.cu) at every layout and network shape the C-ABI accepts, on the GPU.

Observation: num_segments 3..16, with and without memory, ray lengths 1000 / 8 / 3 and max_distance
10 / 2.5, against the CPU oracle and the high-precision reference of tests/dqn_exact_ref.py.
Q-network: the tensor-core path (qnet_mma_kernel) and the FMA-pipe path at every input width 6..249
and output count 1..64; their reference is computed from the kernel's own `ext` output plus
`internal`, so it does not depend on the geometry's rounding and can be exact."""
import ctypes as C
import os

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from tests import dqn_exact_ref as R
from tests import oracle_lib as O
from tests.test_dqn_shapes import LAYOUTS, layout
from tests.test_gpu_dqn_moving import _assert_same, _ellipse

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNSUPPORTED = -4


@pytest.fixture
def qnet_path(monkeypatch):
    """qnet_path("fma") forces the FMA-pipe path (TTDQN_QNET=fma), "mma" leaves the dispatcher's choice."""
    def set_path(p):
        monkeypatch.setenv("TTDQN_QNET", p)
    return set_path


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run(lay, w, agent, geo, internal=None, old=None, moving=None):
    """One observe + act call; returns (rc, outputs as numpy).  geo: numpy arrays of pack_geometry."""
    import torch
    n, ns = len(agent), lay.num_segments
    n_ext = (4 if lay.use_memory else 2) * ns
    n_out = w.n_out if w is not None else 1
    out = dict(ext=torch.full((n, n_ext), np.nan, device="cuda"), q=torch.full((n, n_out), np.nan, device="cuda"),
               action=torch.full((n,), -1, dtype=torch.int32, device="cuda"),
               seg=torch.full((n, ns), np.nan, dtype=torch.float64, device="cuda"),
               ray=torch.full((n, ns), np.nan, dtype=torch.float64, device="cuda"))
    old_d = _cuda(old.astype(np.float32)) if lay.use_memory else None
    int_d = _cuda(internal.astype(np.float32)) if internal is not None and lay.n_internal else None
    qs = w.device_struct() if w is not None else None
    comp = t.dqn.DqnCompanion(lay, w)
    dp = lambda x: None if x is None else x.data_ptr()
    agent_d, geo_d = _cuda(agent), [_cuda(a) for a in geo]       # alive until the call has run
    args = [C.byref(lay), C.byref(qs) if qs else None, n, dp(agent_d), *[dp(g) for g in geo_d]]
    outs = [dp(out["ext"]), dp(out["q"] if w else None), dp(out["action"] if w else None), dp(out["seg"]), dp(out["ray"])]
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    if moving is None:
        rc = comp.lib.ttdqn_observe_act_device(*args, dp(int_d), dp(old_d), *outs, st)
    else:
        mdev = [_cuda(a) for a in moving]
        mv = t.dqn.moving_struct(n, *mdev)
        rc = comp.lib.ttdqn_observe_act_moving_device(*args, C.byref(mv), dp(int_d), dp(old_d), *outs, st)
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["old_ext"] = old_d.cpu().numpy() if old_d is not None else None
    res["error"] = comp.lib.ttdqn_last_error().decode() if rc else ""
    return rc, res


def _ok(rc, res):
    assert rc == 0, res["error"]
    return res


def _net_input(lay, res, internal):
    x = res["ext"]
    if lay.n_internal:
        x = np.c_[x, internal.astype(np.float32)]
    return np.ascontiguousarray(x, dtype=np.float32)


def _compare_geometry(lay, got, ref, what):
    for k in ("seg", "ray"):
        fin = np.isfinite(ref[k])
        assert np.array_equal(fin, np.isfinite(got[k])), f"{k} finiteness ({what})"
        assert np.abs(got[k][fin] - ref[k][fin]).max(initial=0.0) <= 1e-9, f"{k} ({what})"
    assert np.abs(got["ext"] - ref["ext"]).max() <= 1e-6, what
    if lay.use_memory:
        assert np.array_equal(got["old_ext"].view(np.uint32), ref["old_ext"].view(np.uint32)), what


# ------------------------------------------------------------------ B1: layout sweep, static rings
@pytest.mark.parametrize("case", LAYOUTS, ids=lambda c: "ns%d_mem%d_L%g_md%g" % c)
def test_layout_sweep_static_rings(case):
    ns, mem, L, md = case
    lay = layout(*case)
    n = 2048
    rng = np.random.default_rng(2000 + 10 * ns + mem)
    scenes, solid, agent = R.shape_scene(rng, n, lay)
    geo = t.dqn.pack_geometry(lay, scenes, solid)
    assert (geo[3] == 0).any() and (geo[3] == lay.max_poly).any()
    internal = rng.uniform(-1, 1, (n, lay.n_internal)).astype(np.float32)
    old = rng.uniform(-1, 1, (n, 2 * ns)).astype(np.float32)
    w = R.random_weights(rng, (4 if mem else 2) * ns + lay.n_internal, 16, 16, 9)
    got = _ok(*run(lay, w, agent, geo, internal, old))
    ref = O.observe_act(lay, w, agent, *geo, internal, old.copy())
    _compare_geometry(lay, got, ref, case)
    if mem:     # the memory rows are the previous observation, passed through unrounded
        assert np.array_equal(got["ext"][:, 2 * ns:].view(np.uint32), old.view(np.uint32))
    # max_distance is the layout's: ext of a finite distance d is 2 / (1 + exp(-2 d / md)) - 1
    fin = np.isfinite(ref["seg"])
    d = ref["seg"][fin].astype(np.float32).astype(np.float64)
    assert np.abs(got["ext"][:, :ns][fin] - (2 / (1 + np.exp(-2 * d / md)) - 1)).max() <= 1e-6
    # 64 environments against the high-precision reference
    scale = max(L, 20.0)
    clear = 0
    for e in range(64):
        sh, rh, m = R.sector_ray_hp(lay, agent[e], scenes[e], solid[e])
        ok = m >= 1e-9 * scale
        clear += int(ok.sum())
        for k, h in (("seg", sh), ("ray", rh)):
            g = got[k][e]
            assert np.array_equal(np.isfinite(g[ok]), np.isfinite(h[ok])), (k, e, g, h)
            f = ok & np.isfinite(h)
            assert np.abs(g[f] - h[f]).max(initial=0.0) <= 1e-12 * scale, (k, e, g, h)
    assert clear >= 0.9 * 64 * ns


# ------------------------------------------------------------------ B2: moving rings, short rays
@pytest.mark.parametrize("ns", [5, 16])
def test_moving_rings_at_short_rays_equal_appended_static_rings(ns):
    lay = layout(ns, 1, 3.0, 2.5)
    n, k, pv = 1024, 4, 8
    rng = np.random.default_rng(300 + ns)
    scenes, solid, agent = R.shape_scene(rng, n, lay)
    lay.max_poly, lay.max_vert = R.SCENE_MAX_POLY + k, R.SCENE_MAX_VERT + k * pv
    centre = np.zeros((n, k, 2)); xy = np.zeros((n, k, pv, 2)); nv = np.zeros((n, k), np.int32)
    for e in range(n):
        for o in range(k):
            if o == 0:                  # a band square of a random sector, as a moving ring
                sq = R.band_square(agent[e], lay, int(rng.integers(0, ns)), rng.uniform(0.1, 0.7))
                centre[e, o] = sq.mean(axis=0)
                shape = sq - centre[e, o]
            else:
                centre[e, o] = agent[e, :2] + rng.uniform(-3.5, 3.5, 2)
                shape = _ellipse(rng, pv) if o % 2 else t.dqn.rect_shape(rng.uniform(0.1, 0.8))
            xy[e, o, :len(shape)] = shape
            nv[e, o] = len(shape)
    static_geo = t.dqn.pack_geometry(lay, scenes, solid)
    app = [list(s) + [centre[e, o] + xy[e, o, :nv[e, o]] for o in range(k)] for e, s in enumerate(scenes)]
    app_solid = [list(s) + [True] * k for s in solid]
    app_geo = t.dqn.pack_geometry(lay, app, app_solid)
    internal = rng.uniform(-1, 1, (n, 14)).astype(np.float32)
    old = rng.uniform(-1, 1, (n, 2 * ns)).astype(np.float32)
    w = R.random_weights(rng, 4 * ns + 14, 16, 16, 9)
    got = _ok(*run(lay, w, agent, static_geo, internal, old, moving=(centre, xy, nv)))
    want = _ok(*run(lay, w, agent, app_geo, internal, old))
    _assert_same(got, want, f"ns {ns}")
    ref = O.observe_act(lay, w, agent, *app_geo, internal, old.copy())
    _compare_geometry(lay, got, ref, f"moving ns {ns}")


# ------------------------------------------------------------------ B3: exact networks
# n_in -> (num_segments, use_memory, n_internal)
SHAPE_LAYOUT = {6: (3, 0, 0), 8: (3, 0, 2), 9: (3, 0, 3), 46: (8, 1, 14), 47: (8, 1, 15), 48: (8, 1, 16),
                78: (8, 1, 46), 248: (16, 1, 184), 249: (16, 1, 185)}


def _shape_layout(n_in):
    ns, mem, ni = SHAPE_LAYOUT[n_in]
    return layout(ns, mem, 1000.0, 10.0, n_internal=ni, max_poly=1, max_vert=4)


def _full_mantissa(rng, shape):
    """fp32 values whose 24-bit significands end in a 1 (the TF32 split's lo part is non-zero)."""
    m = rng.integers(2 ** 22, 2 ** 23, shape) * 2 + 1
    e = rng.integers(-3, 3, shape)
    s = np.where(rng.uniform(size=shape) < 0.25, -1.0, 1.0)
    return (s * np.ldexp(m.astype(np.float64), e - 23)).astype(np.float32)


def _pow2(rng, shape, neg=0.25):
    return (np.where(rng.uniform(size=shape) < neg, -1.0, 1.0) * np.ldexp(1.0, rng.integers(-3, 4, shape))).astype(np.float32)


def _selection_net(rng, n_in, n_out, variant):
    """One non-zero per row, zero biases: every neuron is one exact product.  "pow2": weights +-2^k;
    "mantissa": the first layer's weights have full significands (the inputs are then powers of two)."""
    def sel(rows, cols, full):
        w = np.zeros((rows, cols), np.float32)
        idx = rng.permutation(max(rows, cols))[:rows] % cols
        w[np.arange(rows), idx] = _full_mantissa(rng, rows) if full else _pow2(rng, rows)
        return w
    z = lambda k: np.zeros(k, np.float32)
    return t.dqn.QNetWeights(sel(16, n_in, variant == "mantissa"), z(16), sel(16, 16, False), z(16),
                             sel(n_out, 16, False), z(n_out))


def _exact_forward(w, x):
    """Reference of a selection network: every neuron is one product, exact in fp64 and in fp32."""
    h = x.astype(np.float64)
    for k in range(3):
        a = h @ w.arrays[2 * k].astype(np.float64).T
        y = a.astype(np.float32)
        assert np.array_equal(y.astype(np.float64), a)              # representable: the reference is exact
        h = np.where(y < 0, np.float32(0), y) if k < 2 else y
    return h


def _grid_capacity_n():
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return 2 * (sms * 8 * 4 * 16) + 37       # qnet_mma_kernel: sms x 8 blocks of 4 warps, 16 envs a tile


@pytest.mark.parametrize("path", ["mma", "fma"])
@pytest.mark.parametrize("variant", ["pow2", "mantissa"])
@pytest.mark.parametrize("n_in", [6, 8, 9, 46, 47, 48, 78, 248])
def test_exact_networks(n_in, variant, path, qnet_path):
    qnet_path(path)
    lay = _shape_layout(n_in)
    rng = np.random.default_rng(n_in * 10 + (variant == "mantissa"))
    ns = lay.num_segments
    sizes = [1, 15, 16, 17, 1000]
    for j, n_out in enumerate([1, 2, 9, 15, 16]):
        w = _selection_net(rng, n_in, n_out, variant)
        for n in sizes + ([_grid_capacity_n()] if n_out in (9, 16) and n_in in (46, 248) else []):
            geo = t.dqn.pack_geometry(lay, [[]] * n, [[]] * n)
            agent = np.c_[rng.uniform(0, 20, (n, 2)), rng.uniform(-3, 3, n)]
            gen = _full_mantissa if variant == "pow2" else _pow2
            internal = gen(rng, (n, lay.n_internal))
            old = gen(rng, (n, 2 * ns))
            got = _ok(*run(lay, w, agent, geo, internal, old))
            assert np.all(got["ext"][:, :2 * ns] == 1.0)               # no rings: seg / ray inf, ext 1
            x = _net_input(lay, got, internal)
            if lay.use_memory:
                assert np.array_equal(x[:, 2 * ns:4 * ns].view(np.uint32), old.view(np.uint32))
            q = _exact_forward(w, x)
            assert np.array_equal(got["q"], q), (n_out, n, np.abs(got["q"] - q).max())
            assert np.array_equal(got["action"], R.first_argmax(q)), (n_out, n)


# ------------------------------------------------------------------ B4: random networks
def _random_inputs(rng, lay, n):
    geo = t.dqn.pack_geometry(lay, [[]] * n, [[]] * n)
    agent = np.c_[rng.uniform(0, 20, (n, 2)), rng.uniform(-3, 3, n)]
    internal = rng.uniform(-2, 2, (n, lay.n_internal)).astype(np.float32)
    old = rng.uniform(-1, 1, (n, 2 * lay.num_segments)).astype(np.float32)
    return agent, geo, internal, old


@pytest.mark.parametrize("n_in", [6, 8, 9, 46, 47, 48, 78, 248])
def test_random_16_wide_networks_on_both_paths(n_in, qnet_path):
    """FMA path == the fp64 replica bit for bit; tensor-core path within tc_bound of the correctly
    rounded network, and the same action wherever the correctly rounded top-2 gap exceeds the bound."""
    lay = _shape_layout(n_in)
    rng = np.random.default_rng(700 + n_in)
    n = 512
    worst = 0.0
    for n_out in (1, 2, 9, 15, 16):
        w = R.random_weights(rng, n_in, 16, 16, n_out)
        agent, geo, internal, old = _random_inputs(rng, lay, n)
        qnet_path("fma")
        got = _ok(*run(lay, w, agent, geo, internal, old))
        x = _net_input(lay, got, internal)
        q_fma = R.fma_net(w, x)
        assert np.array_equal(got["q"].view(np.uint32), q_fma.view(np.uint32)), n_out
        assert np.array_equal(got["action"], R.first_argmax(q_fma))
        qnet_path("mma")
        tc = _ok(*run(lay, w, agent, geo, internal, old))
        assert np.array_equal(tc["ext"].view(np.uint32), got["ext"].view(np.uint32))
        q_cr, hidden = R.cr_net(w, x)
        err = np.abs(tc["q"].astype(np.float64) - q_cr)
        unit = R.tc_bound(w, x, hidden, kappa=1.0)
        worst = max(worst, float((err / unit).max()))
        bound = R.KAPPA * unit
        assert np.all(err <= bound), (n_out, float((err / unit).max()))
        if n_out > 1:
            srt = np.sort(q_cr.astype(np.float64), axis=1)
            clear = (srt[:, -1] - srt[:, -2]) > 2 * bound.max(axis=1)
            assert clear.mean() > 0.9
            assert np.array_equal(tc["action"][clear], R.first_argmax(q_cr)[clear])
    print(f"tensor-core error / (2^-24 bound) at n_in {n_in}: max {worst:.3f} (KAPPA {R.KAPPA})")


def test_random_networks_of_other_shapes_on_the_fma_path():
    """Every other shape runs on the FMA path (also 16-16 with n_in = 249): equal to the replica."""
    rng = np.random.default_rng(77)
    n = 300
    shapes = [(46, a, b, c) for a in (1, 31, 32, 33, 64) for b in (1, 31, 32, 33, 64) for c in (1, 17, 64)]
    shapes += [(249, 16, 16, c) for c in (1, 9, 16)] + [(248, 33, 16, 9), (9, 64, 1, 17)]
    for n_in, h1, h2, n_out in shapes:
        lay = _shape_layout(n_in)
        w = R.random_weights(rng, n_in, h1, h2, n_out)
        agent, geo, internal, old = _random_inputs(rng, lay, n)
        got = _ok(*run(lay, w, agent, geo, internal, old))
        q = R.fma_net(w, _net_input(lay, got, internal))
        assert np.array_equal(got["q"].view(np.uint32), q.view(np.uint32)), (n_in, h1, h2, n_out)
        assert np.array_equal(got["action"], R.first_argmax(q)), (n_in, h1, h2, n_out)


# ------------------------------------------------------------------ B5: argmax ties
@pytest.mark.parametrize("path", ["mma", "fma"])
@pytest.mark.parametrize("n_out", [9, 16, 17])
def test_argmax_ties_take_the_first_maximum(n_out, path, qnet_path):
    qnet_path(path)
    rng = np.random.default_rng(n_out)
    lay = _shape_layout(46)
    w = R.random_weights(rng, 46, 16, 16, n_out)
    w2, b2 = w.arrays[4].copy(), w.arrays[5].copy()
    tied = [1, 4, n_out - 1]
    b2[:] = -50.0
    for o in tied:
        w2[o] = np.abs(w2[tied[0]]); b2[o] = 50.0
    w = t.dqn.QNetWeights(*w.arrays[:4], w2, b2)
    agent, geo, internal, old = _random_inputs(rng, lay, 700)
    got = _ok(*run(lay, w, agent, geo, internal, old))
    q = got["q"]
    assert np.all(q[:, tied] == q[:, [tied[0]]])
    assert np.array_equal(got["action"], np.full(len(agent), tied[0]))


# ------------------------------------------------------------------ B6: grid-stride of the observation
def test_observation_grid_stride_loop():
    """16 387 environments: far more than the observation kernel's grid holds at once."""
    lay = layout(8, 1, 8.0, 2.5, max_poly=4, max_vert=32)
    n = 16387
    rng = np.random.default_rng(9)
    sq = lambda c, h: c + np.array([(-h, -h), (h, -h), (h, h), (-h, h)])
    scenes = [[sq(rng.uniform(2, 18, 2), rng.uniform(0.3, 1.5)) for _ in range(2)] for _ in range(n)]
    solid = [[True, True]] * n
    geo = t.dqn.pack_geometry(lay, scenes, solid)
    agent = np.c_[rng.uniform(0, 20, (n, 2)), rng.uniform(-3, 3, n)]
    internal = rng.uniform(-1, 1, (n, 14)).astype(np.float32)
    old = rng.uniform(-1, 1, (n, 16)).astype(np.float32)
    g = np.load(os.path.join(ROOT, "tests", "golden", "qnet_ray.npz"))
    w = t.dqn.QNetWeights(*[g[k] for k in ("w0", "b0", "w1", "b1", "w2", "b2")])
    got = _ok(*run(lay, w, agent, geo, internal, old))
    ref = O.observe_act(lay, w, agent, *geo, internal, old.copy())
    _compare_geometry(lay, got, ref, "grid stride")
    assert np.isfinite(got["seg"]).any(axis=1).mean() > 0.5


# ------------------------------------------------------------------ B7: internal_obs and rl_ref edges
def _paths(rng, m):
    p = [np.array([(3.0, 4.0)]),                                             # one node
         np.array([(0.0, 0.0), (0.0, 0.0), (2.0, 0.0), (2.0, 0.0), (2.0, 2.0)]),  # duplicate nodes
         np.array([(0.0, 0.0), (2.0, 0.0), (2.0, 2.0)]),                     # agent equidistant (below)
         np.cumsum(rng.uniform(-1, 2, (m, 2)), axis=0)]                      # exactly max_nodes nodes
    return p


@pytest.mark.parametrize("corner_samples", [0, 1, 8])
def test_internal_obs_edge_cases(corner_samples):
    import torch
    m = 7
    rng = np.random.default_rng(corner_samples)
    base = _paths(rng, m)
    agents, paths = [], []
    for k, p in enumerate(base):
        for j in range(6):
            a = np.array([*rng.uniform(-1, 4, 2), rng.uniform(-3, 3), rng.uniform(-0.5, 1.5), rng.uniform(-0.5, 0.5)])
            if k == 2:
                a[:2] = (1.0, 1.0) if j % 2 else (3.0, -1.0)   # 1 from both segments / from the corner
            agents.append(a); paths.append(p)
    agents = np.array(agents)
    xy, cnt = t.dqn.pack_paths(paths, max_nodes=m)
    assert cnt.min() == 1 and cnt.max() == m
    for offset in (-1.5, 0.0, 0.7, 100.0):
        for md in (10.0, 3.7):
            obs, prog = t.dqn.internal_obs_device(torch.tensor(agents).cuda(), torch.tensor(xy).cuda(),
                                                  torch.tensor(cnt).cuda(), corner_samples=corner_samples,
                                                  sample_offset=offset, max_distance=md)
            obs, prog = obs.cpu().numpy(), prog.cpu().numpy()
            ref = [O.internal_obs(agents[e], paths[e], corner_samples, offset, md) for e in range(len(agents))]
            assert np.array_equal(prog, np.array([r[1] for r in ref])), (offset, md)
            assert np.abs(obs - np.array([r[0] for r in ref])).max() <= 6e-8, (offset, md)
    # the equidistant agent at (1, 1) projects onto the first segment: progress 1, not 3
    assert prog[13] == 1.0


def test_rl_ref_edge_cases():
    import torch
    rng = np.random.default_rng(3)
    n = 9 * 4
    agents = np.c_[rng.uniform(-5, 5, (n, 2)), rng.uniform(-3, 3, n), rng.uniform(-0.7, 1.7, n), rng.uniform(-0.7, 0.7, n)]
    act = np.arange(n, dtype=np.int32) % 9
    for steps in (1, 2, 20):
        for ref_speed in (-1.0, 0.0, 0.7):
            rl = t.dqn.rl_ref_device(torch.tensor(agents).cuda(), torch.tensor(act).cuda(), steps=steps,
                                     ref_speed=ref_speed).cpu().numpy()
            ref = np.array([O.rl_ref(agents[e], int(act[e]), steps=steps, ref_speed=ref_speed, use_libm=False)
                            for e in range(n)])
            assert np.array_equal(rl, ref), (steps, ref_speed)


# ------------------------------------------------------------------ B8: shared-memory limit
def _fma_smem(n_in, h1, h2, n_out):
    """Shared memory per block of the FMA path (ttmpc.h, ttdqn_observe_act_device)."""
    up = lambda b: (b + 15) // 16 * 16
    return up(4 * (n_in * h1 + h1 + h1 * h2 + h2 + h2 * n_out + n_out)) + 4 * up(1024 + 4 * (n_in + h1 + h2 + n_out + 4))


def test_largest_fma_network_runs_and_the_next_is_refused():
    import torch
    limit = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    n_in, h1, n_out = 46, 256, 64
    h2 = max(h for h in range(1, 257) if _fma_smem(n_in, h1, h, n_out) <= limit)
    assert h2 < 256 and _fma_smem(n_in, h1, h2 + 1, n_out) > limit
    lay = _shape_layout(46)
    rng = np.random.default_rng(8)
    agent, geo, internal, old = _random_inputs(rng, lay, 96)
    w = R.random_weights(rng, n_in, h1, h2, n_out)
    got = _ok(*run(lay, w, agent, geo, internal, old))
    q = R.fma_net(w, _net_input(lay, got, internal))
    assert np.array_equal(got["q"].view(np.uint32), q.view(np.uint32))
    w = R.random_weights(rng, n_in, h1, h2 + 1, n_out)
    rc, res = run(lay, w, agent, geo, internal, old)
    assert rc == UNSUPPORTED
    assert "shared memory" in res["error"] and str(limit) in res["error"], res["error"]
    # nothing ran: every output keeps its fill and the memory rows are untouched
    assert np.isnan(res["ext"]).all() and np.isnan(res["q"]).all() and (res["action"] == -1).all()
    assert np.isnan(res["seg"]).all() and np.array_equal(res["old_ext"], old)
