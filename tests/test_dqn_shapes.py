"""DQN observation and Q-network at non-default layouts and shapes: the parts that need no GPU (layout
checks of the C-ABI and the Python wrappers, self-checks of tests/dqn_exact_ref.py)."""
import ctypes as C
import os

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib
from tests import dqn_exact_ref as R
from tests import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_CONFIG = -1

# (num_segments, use_memory, ray_length, max_distance): the layouts of the GPU sweep
LAYOUTS = [(3, 0, 3.0, 10.0), (3, 1, 1000.0, 2.5), (4, 0, 8.0, 2.5), (4, 1, 3.0, 10.0), (5, 0, 1000.0, 10.0),
           (5, 1, 8.0, 2.5), (7, 0, 3.0, 2.5), (7, 1, 1000.0, 10.0), (8, 0, 8.0, 10.0), (8, 1, 3.0, 2.5),
           (12, 0, 1000.0, 2.5), (12, 1, 8.0, 10.0), (16, 0, 3.0, 10.0), (16, 1, 1000.0, 2.5)]


def layout(ns, mem, L, md, n_internal=14, max_poly=R.SCENE_MAX_POLY, max_vert=R.SCENE_MAX_VERT):
    lay = t.dqn.default_layout(max_poly, max_vert)
    lay.num_segments, lay.use_memory, lay.ray_length, lay.max_distance, lay.n_internal = ns, mem, L, md, n_internal
    return lay


@pytest.mark.parametrize("ns", [0, 1, 2, 17, -3])
def test_degenerate_segment_counts_are_rejected_before_device_work(ns):
    lib = _lib.load()
    lay = t.dqn.default_layout()
    lay.num_segments = ns
    fake = C.c_void_p(16)          # never dereferenced: the layout check comes first
    for n in (0, 4):
        rc = lib.ttdqn_observe_act_device(C.byref(lay), None, n, fake, fake, fake, fake, fake, None, fake,
                                          None, None, None, None, None, None)
        assert rc == BAD_CONFIG, (n, rc)
        assert "num_segments" in lib.ttdqn_last_error().decode()
        mv = _lib.TtdqnMoving(0, 4, 1, 0, None, None, None)
        rc = lib.ttdqn_observe_act_moving_device(C.byref(lay), None, n, fake, fake, fake, fake, fake, C.byref(mv),
                                                 None, fake, None, None, None, None, None, None)
        assert rc == BAD_CONFIG, (n, rc)
        rc = lib.ttdqn_observe_act_host(C.byref(lay), None, n, *[fake] * 12)
        assert rc == BAD_CONFIG, (n, rc)
    with pytest.raises(_lib.TtmpcError, match="num_segments must be in 3..16"):
        t.dqn.DqnCompanion(lay)


@pytest.mark.parametrize("ns", [3, 16])
def test_segment_count_bounds_are_accepted(ns):
    lay = t.dqn.default_layout()
    lay.num_segments = ns
    assert t.dqn.DqnCompanion(lay).n_ext == 4 * ns
    assert _lib.load().ttdqn_observe_act_host(C.byref(lay), None, 0, *[None] * 12) == 0


@pytest.mark.parametrize("ns", [1, 2, 17])
def test_enable_dqn_rejects_degenerate_segment_counts(ns):
    import torch
    fl = t.scenes.make_fleet(4, seed=3)
    fp = t.FleetPlanner(t.Configurator(), fl["init"], fl["goal"], fl["paths"], device="cpu")
    lay = t.dqn.default_layout(max_poly=6, max_vert=64)
    lay.num_segments = ns
    geo = [torch.from_numpy(a) for a in t.dqn.pack_geometry(lay, [[]] * 4, [[]] * 4)]
    pxy, pn = t.dqn.pack_paths(fl["paths"])
    w = R.random_weights(np.random.default_rng(0), 4 * max(ns, 1) + 14, 16, 16, 9)
    with pytest.raises(_lib.TtmpcError, match="num_segments"):
        fp.enable_dqn(w, geo, [torch.from_numpy(pxy), torch.from_numpy(pn)], layout=lay)
    assert fp._dqn is None and fp.hint is None


@pytest.mark.parametrize("case", LAYOUTS, ids=lambda c: "ns%d_mem%d_L%g_md%g" % c)
def test_high_precision_sector_reference_equals_the_oracle(case):
    """tests/dqn_exact_ref.sector_ray_hp against ttdqn_oracle_observe on shape_scene's scenes: the same
    finiteness pattern and 1e-12 of max(L, scene size) wherever the decisions are clear (margin)."""
    ns, mem, L, md = case
    lay = layout(*case)
    rng = np.random.default_rng(1000 + ns * 10 + mem)
    scenes, solid, agent = R.shape_scene(rng, 24, lay)
    scale = max(L, 20.0)
    clear = band = 0
    for e in range(len(agent)):
        so, ro = O.observe(lay, agent[e], scenes[e], solid[e])
        sh, rh, m = R.sector_ray_hp(lay, agent[e], scenes[e], solid[e])
        ok = m >= 1e-9 * scale
        clear += int(ok.sum())
        for a, b in ((so, sh), (ro, rh)):
            assert np.array_equal(np.isfinite(a[ok]), np.isfinite(b[ok])), (e, a, b, m)
            f = ok & np.isfinite(a)
            assert np.abs(a[f] - b[f]).max(initial=0.0) <= 1e-12 * scale, (e, a, b)
        _, rh_all, _ = R.sector_ray_hp(lay, agent[e], scenes[e], solid[e], ray_rule=False)
        band += int((np.isinf(rh) & np.isfinite(rh_all) & ok).sum())
    assert clear >= 0.9 * 24 * ns
    assert band >= 8, band          # the scenes hold rings only the ray-length rule hides


def test_correctly_rounded_network_equals_the_fp64_replica_on_the_trained_weights():
    g = np.load(os.path.join(ROOT, "tests", "golden", "qnet_ray.npz"))
    w = t.dqn.QNetWeights(*[g[k] for k in ("w0", "b0", "w1", "b1", "w2", "b2")])
    rng = np.random.default_rng(5)
    x = np.c_[rng.uniform(-1, 1, (400, 32)), np.resize(g["internal"], (400, 14)) + rng.normal(0, 0.1, (400, 14))]
    x = x.astype(np.float32)
    q_cr, _ = R.cr_net(w, x)
    q_fma = R.fma_net(w, x)
    assert np.array_equal(q_cr.view(np.uint32), q_fma.view(np.uint32))


def test_correct_rounding_of_the_exact_reference():
    """_round_f32 rounds to nearest with ties to even, through the subnormal range."""
    f32 = lambda v: float(np.float32(v))
    assert R._round_f32(2 ** 24 + 1, 0) == 2.0 ** 24                 # tie, even below
    assert R._round_f32(2 ** 24 + 3, 0) == 2.0 ** 24 + 4             # tie, even above
    assert R._round_f32(-(2 ** 25 + 3), 0) == -(2.0 ** 25 + 4)
    assert R._round_f32(1, -150) == 0.0 and R._round_f32(3, -150) == f32(2.0 ** -148)
    assert R._round_f32(3, -151) == f32(2.0 ** -149)
    rng = np.random.default_rng(1)
    for _ in range(2000):           # fp64 values with few enough bits round the same way through numpy
        v = float(rng.normal()) * 2.0 ** int(rng.integers(-60, 60))
        n, d = v.as_integer_ratio()
        e = -(d.bit_length() - 1)
        assert R._round_f32(n, e) == f32(v)
    # the fma replica's ReLU keeps -0.0, as `a < 0 ? 0 : a` does
    y = R.fma_layer(np.array([[1.0]]), np.array([-0.0]), np.array([[-0.0]], np.float32), True)
    assert np.signbit(y[0, 0])
