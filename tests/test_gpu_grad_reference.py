"""GPU tests (-m gpu): psi and grad psi of the evaluation kernel (BatchSolver.evaluate, i.e.
ttmpc_eval_batch_host) against the complex-step reference edge_scenes.ref_psi_grad and the
long-double edge_scenes.ref_psi, at the cases and within the bounds of tests/test_grad_reference.py
(its Reference docstring states them); and at the solve kernel's own outputs (controls,
multipliers, final penalty) of every specialised solve shape, rolled and unrolled builds.

Every evaluation is also compared bit for bit with O.eval_warp, the kernel's CPU mirror."""
import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from tests import oracle_lib as O
from tests import test_grad_reference as G

pytestmark = pytest.mark.gpu


def kernel_check(case, label, order=1e-11):
    """The kernel's psi and grad psi against the reference and against eval_warp; returns the Reference."""
    cfg, p, u, c, y = case
    ref = G.Reference(cfg, p, u, c, y, order)
    ev = t.BatchSolver(cfg).evaluate(p, u, c, y)
    ref.check(f"{label} kernel", ev["psi"], ev["grad"])
    for i in range(len(p)):
        _, _, ps, gr = O.eval_warp(cfg, u[i], p[i], c[i], y[i])
        assert ps == ev["psi"][i] and np.array_equal(gr, ev["grad"][i]), (label, i)
    return ref


@pytest.mark.parametrize("shape", G.SHAPES, ids=G.shape_id)
def test_kernel_grad_psi_at_every_shape(shape):
    ref = kernel_check(G.shape_case(shape), G.shape_id(shape))
    G.assert_content(ref, ("fleet", "dyn_soft", "penalty_F2", "alm_F1", "terminal", "speed_control"))


@pytest.mark.parametrize("offset", G.OFFSETS, ids=str)
def test_kernel_grad_psi_far_coordinates(offset):
    G.assert_content(kernel_check(G.far_case(offset), f"offset {offset}"))


@pytest.mark.parametrize("shape", [{}, dict(Nother=32, Nstcobs=32, nstcobs=24, Ndynobs=64)], ids=G.shape_id)
@pytest.mark.parametrize("term", G.TERMS)
def test_kernel_grad_psi_one_term_at_a_time(term, shape):
    G.assert_one_term(kernel_check(G.one_term_case(term, shape), f"{term} {G.shape_id(shape)}"), term)


@pytest.mark.parametrize("code", ["small", "unrolled"])
@pytest.mark.parametrize("shape", G.SOLVE_SHAPES + [G.MAX_SHAPE], ids=G.shape_id)
def test_kernel_grad_psi_at_solve_kernel_outputs(monkeypatch, shape, code):
    """The specialised solve kernels (csrc/ttmpc_solve.cu TTMPC_SOLVE_SHAPES) and the run-time one at
    the all-maxima shape: psi and grad psi at what they return.  Bounds as in
    test_grad_reference.test_grad_psi_at_solutions."""
    monkeypatch.setenv("TTMPC_CODE", code)
    c = t.Configurator(**shape).to_ttmpc()
    rng = np.random.default_rng(320)
    p = G.with_weights(G.rich_scenes(c, 16, 320), c, rng)
    sol = t.BatchSolver(c).run(p)
    case = (c, p, sol.solution, sol.penalty, sol.lagrange_multipliers)
    ref = kernel_check(case, f"solve kernel {code} {G.shape_id(shape)}", order=5e-10)
    assert (sol.penalty > 1.0).sum() >= 3
    G.assert_content(ref, ("fleet", "penalty_F2"))
