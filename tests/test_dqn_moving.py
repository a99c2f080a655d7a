"""Moving obstacles in the DQN's lidar and FleetPlanner.enable_dqn: the parts that need no GPU
(struct layout, argument checks, the square template, shape checks of enable_dqn)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_ARG = -2


def test_ttdqn_moving_struct_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    fields = [f for f, _ in _lib.TtdqnMoving._fields_]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "ttmpc.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(ttdqn_moving));\n'
                   + "".join(f'  printf(" %zu", offsetof(ttdqn_moving, {f}));\n' for f in fields)
                   + '  printf("\\n"); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    vals = list(map(int, subprocess.check_output([str(exe)]).split()))
    assert C.sizeof(_lib.TtdqnMoving) == vals[0]
    assert [getattr(_lib.TtdqnMoving, f).offset for f in fields] == vals[1:]
    assert _lib.load().ttmpc_version() == 102


def test_malformed_moving_is_rejected_before_device_work():
    lib = _lib.load()
    lay = t.dqn.default_layout()
    fake = C.c_void_p(16)          # never dereferenced: the checks come first
    good = dict(n_live=2, max_pv=4, shape_shared=1, centre=16, shape_xy=16, shape_nv=16)
    bad = [dict(n_live=-1), dict(max_pv=2), dict(max_pv=33), dict(max_pv=0), dict(max_pv=-4),
           dict(centre=None), dict(shape_xy=None), dict(shape_nv=None), dict(n_live=0, max_pv=2)]
    for n in (0, 4):
        for kw in bad:
            mv = _lib.TtdqnMoving(**{**good, **kw})
            rc = lib.ttdqn_observe_act_moving_device(C.byref(lay), None, n, fake, fake, fake, fake, fake, C.byref(mv),
                                                     None, fake, None, None, None, None, None, None)
            assert rc == BAD_ARG, (n, kw)
            assert "moving" in lib.ttdqn_last_error().decode()
    # well-formed with no environments: nothing to do
    for kw in (dict(), dict(n_live=0, centre=None, shape_xy=None, shape_nv=None), dict(max_pv=3), dict(max_pv=32)):
        mv = _lib.TtdqnMoving(**{**good, **kw})
        assert lib.ttdqn_observe_act_moving_device(C.byref(lay), None, 0, None, None, None, None, None, C.byref(mv),
                                                   None, fake, None, None, None, None, None, None) == 0, kw
    assert lib.ttdqn_observe_act_moving_device(C.byref(lay), None, 0, None, None, None, None, None, None,
                                               None, fake, None, None, None, None, None, None) == 0


def test_rect_shape_is_the_switchers_square():
    """centre + rect_shape(r) gives the circle_to_rect vertices the HintSwitcher's squares have
    (sw_obstacle in csrc/ttmpc_fleet.cu, main.py:91-95), in their order, bit for bit."""
    rng = np.random.default_rng(7)
    for _ in range(200):
        c = rng.uniform(-50, 50, 2)
        r = float(rng.choice([t.fleet.DYN_OBS_SIZE, rng.uniform(0.01, 3.0)]))
        rect = np.array([(c[0] - r, c[1] - r), (c[0] + r, c[1] - r), (c[0] + r, c[1] + r), (c[0] - r, c[1] + r)])
        got = c + t.dqn.rect_shape(r)
        assert got.dtype == np.float64 and got.shape == (4, 2)
        assert np.array_equal(got.view(np.uint64), rect.view(np.uint64))


def _planner_and_inputs(n=4):
    import torch
    fl = t.scenes.make_fleet(n, seed=3)
    fp = t.FleetPlanner(t.Configurator(), fl["init"], fl["goal"], fl["paths"], device="cpu")
    g = np.load(os.path.join(ROOT, "tests", "golden", "qnet_ray.npz"))
    w = t.dqn.QNetWeights(*[g[k] for k in ("w0", "b0", "w1", "b1", "w2", "b2")])
    lay = t.dqn.default_layout(max_poly=6, max_vert=64)
    rings = [[np.array([(0.0, 0.0), (1.0, 0.0), (1.0, 1.0)])]] * n
    geo = [torch.from_numpy(a) for a in t.dqn.pack_geometry(lay, rings, [[True]] * n)]
    pxy, pn = t.dqn.pack_paths(fl["paths"])
    return fp, w, geo, [torch.from_numpy(pxy), torch.from_numpy(pn)]


def test_enable_dqn_rejects_tensors_of_the_wrong_shape():
    fp, w, geo, paths = _planner_and_inputs()
    # well-shaped host tensors pass every shape check and are refused only for not being on the GPU
    with pytest.raises(ValueError, match="contiguous CUDA"):
        fp.enable_dqn(w, geo, paths)
    xy, off, sol, cnt = geo
    cases = [
        ("geometry xy", (xy[:3], off, sol, cnt), paths, {}),
        ("geometry xy", (xy.float(), off, sol, cnt), paths, {}),
        ("geometry xy", (xy[:, :32].contiguous(), off, sol, cnt), paths, dict(layout=t.dqn.default_layout(6, 64))),
        ("geometry off", (xy, off[:, :5].contiguous(), sol, cnt), paths, {}),
        ("geometry off", (xy, off.long(), sol, cnt), paths, {}),
        ("geometry solid", (xy, off, sol.bool(), cnt), paths, {}),
        ("geometry count", (xy, off, sol, cnt[:2]), paths, {}),
        ("geometry count", (xy, off, sol, cnt.double()), paths, {}),
        ("path_xy", geo, (paths[0][:2], paths[1]), {}),
        ("path_xy", geo, (paths[0].float(), paths[1]), {}),
        ("path_xy", geo, (paths[0][:, :1].contiguous(), paths[1]), {}),
        ("path_n", geo, (paths[0], paths[1][:3]), {}),
        ("path_n", geo, (paths[0], paths[1].long()), {}),
        ("geometry = ", geo[:3], paths, {}),
        ("moving_shape", geo, paths, dict(moving_shape=np.zeros((2, 2, 2)))),
        ("moving_shape", geo, paths, dict(moving_shape=np.zeros((2, 33, 2)))),
        ("moving_shape", geo, paths, dict(moving_shape="circle")),
        ("moving_radius", geo, paths, dict(moving_radius=-1.0)),
        ("corner_samples", geo, paths, dict(corner_samples=2)),
    ]
    for name, g, p, kw in cases:
        with pytest.raises(ValueError, match=name):
            fp.enable_dqn(w, g, p, **kw)
    assert fp._dqn is None and fp.hint is None
    with pytest.raises(ValueError, match="Q-network input"):
        fp.enable_dqn(t.dqn.QNetWeights(np.zeros((16, 40)), *w.arrays[1:]), geo, paths)
