"""Occupancy of the bulk solve (-m gpu): batches larger than the resident warps of the unrolled build
run on the rolled build of the solve kernel, which fits 168 registers per thread and 12 scenes per SM
for the default shapes (DESIGN.md section 3.1), launches every CTA size the API picks, and gives the
same results as the unrolled build."""
import dataclasses

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t

pytestmark = pytest.mark.gpu


def test_bulk_batch_runs_12_scenes_per_sm(cfg):
    info = t.BatchSolver(cfg).launch_info(4096)
    assert info["block"] == 64
    assert info["blocks_per_sm"] * info["block"] // 32 == 12
    assert info["grid"] == min(info["sm_count"] * info["blocks_per_sm"], 4096 // 2)


# the default shapes, the sweep shapes of TTMPC_SOLVE_SHAPES, and tables large enough that the API
# packs three scenes per CTA (run-time-dimension kernel)
SHAPES = {
    "default": dict(),
    "N10": dict(N_hor=10),
    "N32": dict(N_hor=32),
    "Nstc4_Ndyn4": dict(Nstcobs=4, Ndynobs=4),
    "Nstc20_Ndyn30": dict(Nstcobs=20, Ndynobs=30),
    "large_tables": dict(N_hor=32, Nother=32, Nstcobs=32, Ndynobs=64, lbfgs_memory=16),
}


@pytest.mark.parametrize("shape", list(SHAPES))
def test_rolled_build_matches_unrolled_build_on_a_bulk_batch(monkeypatch, shape):
    """A batch 300 scenes larger than the unrolled build's resident warps runs on the rolled build.
    Forced onto the unrolled build it gives the same bits in every result field but `evals` (clock
    readings, and evaluation counts that include a tail helper's speculative work)."""
    import torch
    mc = t.Configurator(**SHAPES[shape])
    c = mc.to_ttmpc()
    solver = t.BatchSolver(c)
    monkeypatch.setenv("TTMPC_CODE", "unrolled")
    unrolled_info = solver.launch_info(1 << 20)
    monkeypatch.delenv("TTMPC_CODE")
    n = unrolled_info["grid"] * unrolled_info["block"] // 32 + 300
    rolled_info = solver.launch_info(n)
    assert rolled_info["block"] == unrolled_info["block"]
    assert rolled_info["blocks_per_sm"] >= unrolled_info["blocks_per_sm"]
    p = t.scenes.make_scenes(n, c, seed=97, n_static=min(4, c.Nstcobs), n_dynamic=min(4, c.Ndynobs),
                             blocking_fraction=0.2, mpc=mc)
    dp = torch.from_numpy(p).cuda()

    def solve():
        sol = solver.run_device(dp, solver.alloc_device(n))
        torch.cuda.synchronize()
        return {f.name: getattr(sol, f.name).cpu().numpy() for f in dataclasses.fields(sol)
                if f.name not in ("evals", "solve_time_ms")}

    rolled = solve()
    monkeypatch.setenv("TTMPC_CODE", "unrolled")
    unrolled = solve()
    assert len(rolled) >= 8
    for name, a in rolled.items():
        assert np.array_equal(a, unrolled[name]), name
