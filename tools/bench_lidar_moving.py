#!/usr/bin/env python
"""observe + Q-network (ttdqn_observe_act_*_device) with moving obstacles in the lidar, one GPU.

  python tools/bench_lidar_moving.py [n=16384] [--rounds 5] [--calls 50]

Geometry of tools/bench_qnet.py (three padded rectangles and a boundary ring per env) and three
configurations of the same call:
  static        the static rings alone (ttdqn_observe_act_device)
  moving2       plus 2 moving squares (circle_to_rect of DYN_OBS_SIZE) at random centres, through
                ttdqn_observe_act_moving_device
  appended2     the same 2 squares appended to the static rings (ttdqn_observe_act_device)
Each round times --calls back-to-back calls of every configuration with CUDA events, in the order
static, moving2, appended2; per configuration the median over the rounds is reported.  moving2 and
appended2 are checked to give identical outputs.  The card's name and power limit are read in the
same run.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.fleet import DYN_OBS_SIZE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = None
    return dict(gpu=torch.cuda.get_device_name(), power_limit=pl or None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int, nargs="?", default=16384)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=50)
    a = ap.parse_args()
    n = a.n
    g = np.load(os.path.join(ROOT, "tests", "golden", "qnet_ray.npz"))
    wq = t.dqn.QNetWeights(*[g[k] for k in ("w0", "b0", "w1", "b1", "w2", "b2")])
    lay = t.dqn.default_layout(max_poly=8, max_vert=160)
    rng = np.random.default_rng(0)
    base = [t.geometry.pad_polygon_round(np.array([(3., 3.), (3., 7.), (7., 7.), (7., 3.)]), 0.5),
            t.geometry.pad_polygon_round(np.array([(12., 2.), (12., 9.), (15., 9.), (15., 2.)]), 0.5),
            t.geometry.pad_polygon_round(np.array([(5., 12.), (5., 15.), (16., 15.), (16., 12.)]), 0.5),
            np.array([(0.5, 0.5), (19.5, 0.5), (19.5, 19.5), (0.5, 19.5)])]
    centre = rng.uniform(2, 18, (n, 2, 2))
    sq = t.dqn.rect_shape(DYN_OBS_SIZE)
    cuda = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    static = [cuda(x) for x in t.dqn.pack_geometry(lay, [base] * n, [[True, True, True, False]] * n)]
    appended = [cuda(x) for x in t.dqn.pack_geometry(lay, [base + [c + sq for c in centre[e]] for e in range(n)],
                                                     [[True, True, True, False, True, True]] * n)]
    moving = (cuda(centre), cuda(np.repeat(sq[None, None], 2, 1)), torch.full((1, 2), 4, dtype=torch.int32, device="cuda"))
    agent = cuda(np.c_[rng.uniform(1, 19, (n, 2)), rng.uniform(-3, 3, n)])
    internal = cuda(np.resize(g["internal"], (n, 14)).astype(np.float32))
    comp, qs = t.dqn.DqnCompanion(lay, wq), wq.device_struct()
    configs = dict(static=(static, None), moving2=(static, moving), appended2=(appended, None))
    bufs = {}
    for name in configs:
        bufs[name] = dict(ext=torch.zeros(n, 32, device="cuda"), q=torch.zeros(n, 9, device="cuda"),
                          action=torch.zeros(n, dtype=torch.int32, device="cuda"),
                          seg=torch.zeros(n, 8, dtype=torch.float64, device="cuda"),
                          ray=torch.zeros(n, 8, dtype=torch.float64, device="cuda"),
                          old=torch.zeros(n, 16, dtype=torch.float32, device="cuda"))

    def call(name):
        geo, mv = configs[name]
        b = bufs[name]
        comp.observe_act_device(agent, *geo, internal, b["old"], b, qs, moving=mv)

    for name in configs:                                   # first launches and the memory pool
        for _ in range(3):
            call(name)
    torch.cuda.synchronize()
    for name in configs:                                   # one call from the same memory for the comparison
        bufs[name]["old"].zero_()
        call(name)
    torch.cuda.synchronize()
    same = all(torch.equal(bufs["moving2"][k], bufs["appended2"][k]) for k in ("ext", "q", "action", "seg", "ray", "old"))
    ms = {name: [] for name in configs}
    for _ in range(a.rounds):
        for name in configs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.calls):
                call(name)
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / a.calls)
    out = dict(tool="bench_lidar_moving", **card(), n_envs=n, rounds=a.rounds, calls=a.calls,
               ms_per_call_median={k: float(np.median(v)) for k, v in ms.items()},
               ms_per_call_rounds=ms, moving2_equals_appended2=bool(same),
               inside_a_solid_ring=int((bufs["moving2"]["seg"] == 0).all(dim=1).sum()))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
