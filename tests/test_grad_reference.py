"""CPU checks of psi and grad psi -- the WARP-order mirror of the kernel (O.eval_warp) and the
reference-order oracle (O.psi, O.psi_grad) -- against the complex-step reference
edge_scenes.ref_psi_grad and the long-double edge_scenes.ref_psi.

eval_warp is bit-identical to the kernel (tests/test_gpu_edge_scenes.py), and the oracle's reverse
pass is a second hand derivation of the same gradient; the complex step involves no derivation at
all.  The cases: every shape the C-ABI's evaluation and solve kernels are built or tested for
(run-time dimensions, the specialised solve shapes, horizons 1-32, all maxima at once), in-box and
10x out-of-box controls, penalties 0, 0.5 (below the 1 of max(c, 1)), 10 and 250 with non-zero
multipliers, far coordinates, the solver's own solutions, and every term of psi on its own.
tests/test_gpu_grad_reference.py runs the same cases through the kernel."""
import os

import numpy as np
import pytest

import trajtrack_mpcndqn_rlboost_b200 as t
from trajtrack_mpcndqn_rlboost_b200.mpc_config import param_offsets
from tests import edge_scenes as E
from tests import oracle_lib as O
from tests.test_gpu_edge_scenes import SHAPES as EDGE_SHAPES, controls, rich_scenes

EPS = 2.0 ** -53
THREADS = os.cpu_count() or 1
PENALTIES = (0.0, 0.5, 10.0, 250.0)
OFFSETS = [(1e3, -1e3), (1e4, 1e4), (-3e4, 5e4), (1e5, 0.0)]
# csrc/ttmpc_solve.cu TTMPC_SOLVE_SHAPES: the shapes with a specialised solve kernel
SOLVE_SHAPES = [dict(), dict(N_hor=10), dict(N_hor=32), dict(Nstcobs=4, Ndynobs=4), dict(Nstcobs=20, Ndynobs=30)]
MAX_SHAPE = dict(N_hor=32, Nother=32, Nstcobs=32, nstcobs=24, Ndynobs=64)


def _unique(shapes):
    out = []
    for s in shapes:
        if s not in out:
            out.append(s)
    return out


SHAPES = _unique(EDGE_SHAPES + [dict(N_hor=N) for N in (1, 2, 3, 7, 16, 17, 31, 32)] + SOLVE_SHAPES + [MAX_SHAPE])
# psi's term groups (edge_scenes.ref_psi); the one-term cases switch on one of them at a time
TERMS = ("path", "speed_control", "fleet", "dyn_soft", "dyn_hard", "static", "terminal", "acc", "alm_F1")


def shape_id(s):
    return ",".join(f"{k}={v}" for k, v in s.items()) or "default"


def with_weights(p, cfg, rng):
    """Every other block of four scenes gets non-zero control-action and terminal weights (zero in
    the default tuning): the terminal block then runs, and its skip is exercised by the others."""
    o = param_offsets(cfg)
    on = (np.arange(len(p)) // 4) % 2 == 1
    for i in (3, 4, 5, 6):                       # rv, rw, qN, qthetaN
        p[on, o["q"] + i] = rng.uniform(0.5, 5.0, on.sum())
    return p


def mixed_controls(rng, cfg, n):
    """Controls in the box for the first half of the scenes, 10x beyond it for the second."""
    u = controls(rng, cfg, n)
    u[n // 2:] *= 10.0
    return u


def multipliers(rng, cfg, n):
    """Penalties cycled through PENALTIES scene by scene, multipliers y uniform in [-2, 2]."""
    return np.resize(PENALTIES, n).astype(np.float64), rng.uniform(-2.0, 2.0, (n, 2 * cfg.N_hor))


def shape_case(shape, n=16, seed=300):
    """(cfg, p, u, c, y) of rich_scenes content at one shape."""
    c = t.Configurator(**shape).to_ttmpc()
    rng = np.random.default_rng(seed)
    p = with_weights(rich_scenes(c, n, seed), c, rng)
    return (c, p, mixed_controls(rng, c, n)) + multipliers(rng, c, n)


def far_case(offset, n=16, seed=310):
    """The default shape's rich_scenes content moved rigidly by offset (m)."""
    c, p, u, cc, y = shape_case({}, n, seed)
    return c, E.translate(p, c, *offset), u, cc, y


def solution_case(shape, n=16, seed=320):
    """rich_scenes at one shape and the oracle's (WARP-order) solution of each scene: (u, y, penalty)."""
    c = t.Configurator(**shape).to_ttmpc()
    rng = np.random.default_rng(seed)
    p = with_weights(rich_scenes(c, n, seed), c, rng)
    ref = O.solve_batch(c, p, threads=THREADS, warp=True)
    return c, p, ref["u"], ref["pen"], ref["y"]


def smooth_controls(rng, cfg, p):
    """Controls whose accelerations lie inside the constraint box: with y = 0 the ALM term is zero."""
    n, N = len(p), cfg.N_hor
    v = np.clip(p[:, 6:7] + np.cumsum(rng.uniform(-0.1, 0.1, (n, N)), 1), cfg.lin_vel_min, cfg.lin_vel_max)
    w = np.clip(p[:, 7:8] + np.cumsum(rng.uniform(-0.4, 0.4, (n, N)), 1), -cfg.ang_vel_max, cfg.ang_vel_max)
    u = np.empty((n, 2 * N))
    u[:, 0::2], u[:, 1::2] = v, w
    return u


def one_term_case(term, shape, n=16, seed=330):
    """rich_scenes with every weight of the q block and every obstacle block zeroed but those of one
    term.  The fleet term's weight is fixed (1000); dynamic soft and hard terms share the dynamic
    block (qdyn weights the soft one, the penalty c the hard one); static obstacles reach psi only
    through F2_j = S + D_j, so that case keeps Ndynobs zero slots (D_j = 0) and a penalty."""
    c = t.Configurator(**shape).to_ttmpc()
    o = param_offsets(c)
    rng = np.random.default_rng(seed)
    p = rich_scenes(c, n, seed)
    keep = {"path": [7], "speed_control": [1, 3, 4], "terminal": [5, 6], "acc": [8, 9]}.get(term, [])
    q = p[:, o["q"]:o["q"] + 10]
    q[:, [i for i in range(10) if i not in keep]] = 0.0
    for i in keep:
        if not q[:, i].any():
            q[:, i] = rng.uniform(0.5, 5.0, n)
    blocks = {"fleet": ("c", "os"), "dyn_soft": ("od", "qstc"), "dyn_hard": ("od", "qstc"), "static": ("os", "od")}
    for lo, hi in [("c", "os"), ("os", "od"), ("od", "qstc")]:
        if blocks.get(term) != (lo, hi):
            p[:, o[lo]:o[hi]] = 0.0
    if term != "dyn_soft":
        p[:, o["qdyn"]:o["qdyn"] + c.N_hor] = 0.0
    if term in ("dyn_hard", "static"):
        cc, y = rng.choice(PENALTIES[1:], n), np.zeros((n, 2 * c.N_hor))
        u = smooth_controls(rng, c, p)
    elif term == "alm_F1":
        u = mixed_controls(rng, c, n)
        cc, y = rng.choice(PENALTIES[1:], n), rng.uniform(-2.0, 2.0, (n, 2 * c.N_hor))
    else:
        u = mixed_controls(rng, c, n)
        cc, y = np.zeros(n), rng.uniform(-2.0, 2.0, (n, 2 * c.N_hor))
    return c, p, u, cc, y


def max_coordinate(cfg, p, u):
    """R per scene: the largest coordinate of the start and of the rollout."""
    return np.maximum(np.abs(p[:, :2]).max(1), np.abs(E.rollouts(cfg, u, p)).max((1, 2)))


class Reference:
    """ref_psi and ref_psi_grad of one case, and the bounds an fp64 implementation must meet.

    Gradient: |g - g_ref|_k <= (order + 16 eps R) max(1, s_k) + 16 eps c (Z_k / ts + N sum_j |dF2_j/du_k|).
    s_k = sum over the term groups t of psi of |d term_t / d u_k| (ref_psi_grad's groups), R the
    largest coordinate of the scene and its rollout, eps = 2^-53.
    - The fp64 rollout carries a rounding error of up to eps R in each position, which moves each
      term's gradient by a few eps R times its own size; the 16 covers both coordinates, the
      differences with centres and path points, and the adjoint's suffix sums.
    - order is the operation order: 1e-11 (up to 2.2e-12 observed in the one-term cases, where
      products of static-edge factors b - a.x and ellipse terms 1 - A^2/Rx^2 - B^2/Ry^2 are formed
      by cancellation); solutions use more (test_grad_psi_at_solutions).
    - A component's scale is the sum of the term magnitudes, not |g_k|, because at solutions large
      terms cancel (fleet or obstacle pushes against the path and the multipliers): the result is
      small, its rounding is not.
    - The last term: psi holds c e^2 / 2 (e = z - clip(z), z = F1 + y / max(c, 1)) and c |F2|^2 / 2.
      e and F2 are formed with an absolute rounding of a few eps |z| and eps per step, which c
      (up to 2e7 at solutions) multiplies however small e and F2 are.  Z_k sums |z| over the two
      accelerations that control k enters; dF2 is ref_psi_grad's Jacobian of F2.

    psi: |psi - psi_ref| <= (order + 16 eps R) max(1, psi_ref); every term group is non-negative,
    so psi_ref is the sum of their magnitudes.

    The kernel forms each position as x0 + (prefix sum of the steps), one rounding at size R; the
    reference-order oracle adds step after step (x_{k+1} = x_k + step), N roundings at size R.  Its
    bounds take 16 N eps R instead (check(..., roundings=N))."""

    def __init__(self, cfg, p, u, c, y, order=1e-11):
        self.cfg, self.p, self.u, self.c, self.y, self.order = cfg, p, u, c, y, order
        g, self.parts, jac_F2 = E.ref_psi_grad(cfg, u, p, c, y, groups=True)
        self.grad = np.asarray(g, np.float64)
        self.psi = np.asarray(E.ref_psi(cfg, u, p, c, y), np.float64)
        self.scale = np.maximum(1.0, np.asarray(sum(np.abs(v) for v in self.parts.values()), np.float64))
        self.R = max_coordinate(cfg, p, u)
        # c times the absolute rounding of F1 + y / max(c, 1) and of F2, through their Jacobians
        N = cfg.N_hor
        z = np.abs(np.asarray(E.ref_eval(cfg, u, p)[1], np.float64) + y / np.maximum(c, 1.0)[:, None])
        za = np.concatenate([z, np.zeros((len(p), 1))], 1)
        zf = np.empty((len(p), 2 * N))
        zf[:, 0::2] = za[:, 0:N] + np.where(np.arange(N) + 1 < N, za[:, 1:N + 1], 0.0)
        zf[:, 1::2] = za[:, N:2 * N] + np.where(np.arange(N) + 1 < N, za[:, N + 1:2 * N + 1], 0.0)
        dF2 = np.abs(np.asarray(jac_F2, np.float64)).sum(1)
        self.amplified = 16 * EPS * c[:, None] * (zf / cfg.ts + N * dF2)

    def bounds(self, roundings=1):
        rel = self.order + 16 * roundings * EPS * self.R
        return rel[:, None] * self.scale + self.amplified, rel * np.maximum(1.0, np.abs(self.psi))

    def check(self, label, psi, grad, roundings=1):
        """Asserts psi [n] and grad [n, 2N] within the bounds; returns the worst ratios to them."""
        grad_bound, psi_bound = self.bounds(roundings)
        dg = np.abs(np.asarray(grad) - self.grad)
        dp = np.abs(np.asarray(psi) - self.psi)
        rg, rp = float((dg / grad_bound).max()), float((dp / psi_bound).max())
        print(f"{label}: grad max |dg| {dg.max():.3e}, max |dg| / bound {rg:.3f}; "
              f"psi max |dpsi| {dp.max():.3e}, max |dpsi| / bound {rp:.3f}")
        i, k = np.unravel_index(np.argmax(dg / grad_bound), dg.shape)
        assert rg <= 1.0, (label, "grad", int(i), int(k), float(grad[i][k]), float(self.grad[i, k]))
        assert rp <= 1.0, (label, "psi", int(np.argmax(dp / psi_bound)))
        return rg, rp

    def group_grad(self, name):
        return np.asarray(self.parts[name], np.float64)


def oracle_check(case, label, order=1e-11):
    """O.eval_warp and the reference-order oracle against the reference; returns the Reference."""
    cfg, p, u, c, y = case
    ref = Reference(cfg, p, u, c, y, order)
    w = [O.eval_warp(cfg, u[i], p[i], c[i], y[i]) for i in range(len(p))]
    ref.check(f"{label} eval_warp", [e[2] for e in w], [e[3] for e in w])
    ref.check(f"{label} psi_grad", [O.psi(cfg, u[i], p[i], c[i], y[i]) for i in range(len(p))],
              [O.psi_grad(cfg, u[i], p[i], c[i], y[i]) for i in range(len(p))], roundings=cfg.N_hor)
    return ref


def assert_content(ref, groups=("fleet", "dyn_soft", "penalty_F2", "alm_F1", "terminal")):
    """The case exercises what it claims: each named term group moves psi in at least 3 scenes."""
    for name in groups:
        assert (ref.group_grad(name) != 0).any(1).sum() >= 3, name


def assert_one_term(ref, term):
    """Only the term under test moves psi, and it does in at least a quarter of the scenes."""
    own = {"dyn_hard": "penalty_F2", "static": "penalty_F2"}.get(term, term)
    for name in ref.parts:
        live = (ref.group_grad(name) != 0).any(1)
        if name == own:
            assert live.mean() >= 0.25, (term, name)
        else:
            assert not live.any(), (term, name)


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_grad_psi_at_every_shape(shape):
    case = shape_case(shape)
    ref = oracle_check(case, shape_id(shape))
    assert_content(ref, ("fleet", "dyn_soft", "penalty_F2", "alm_F1", "terminal", "speed_control"))


@pytest.mark.parametrize("offset", OFFSETS, ids=str)
def test_grad_psi_far_coordinates(offset):
    ref = oracle_check(far_case(offset), f"offset {offset}")
    assert_content(ref)


@pytest.mark.parametrize("shape", SOLVE_SHAPES + [MAX_SHAPE], ids=shape_id)
def test_grad_psi_at_solutions(shape):
    """At the solver's own outputs: controls, multipliers and final penalty of each scene.  The
    penalty reaches 2e7 there and solutions sit on obstacle edges, where a static product's factors
    b - a.x are small differences of large numbers (relative rounding eps |a| R / |b - a.x|, not
    eps): the operation-order part of the bound is 5e-10 here (1.6e-10 observed, at Nstcobs=20,
    Ndynobs=30 where a solution ends inside a static obstacle at c = 2e7)."""
    case = solution_case(shape)
    ref = oracle_check(case, f"solutions {shape_id(shape)}", order=5e-10)
    assert (case[3] > 1.0).sum() >= 3          # some solves raised the penalty
    assert_content(ref, ("fleet", "penalty_F2"))


@pytest.mark.parametrize("shape", [{}, dict(Nother=32, Nstcobs=32, nstcobs=24, Ndynobs=64)], ids=shape_id)
@pytest.mark.parametrize("term", TERMS)
def test_grad_psi_one_term_at_a_time(term, shape):
    """A wrong small term must not hide under a large one (the fleet term's weight is 1000)."""
    ref = oracle_check(one_term_case(term, shape), f"{term} {shape_id(shape)}")
    assert_one_term(ref, term)


def test_complex_step_matches_central_differences(cfg):
    """The reference itself: ref_psi_grad against fp64 central differences of ref_psi (h = 1e-6,
    truncation error ~h^2 |psi'''|), on the scenes of test_oracle_gradient_finite_differences."""
    p = t.scenes.make_scenes(6, cfg, seed=21, n_static=4, n_dynamic=5, blocking_fraction=0.5)
    rng = np.random.default_rng(1)
    u = rng.uniform(-0.3, 1.2, (6, 40)); u[:, 1::2] = rng.uniform(-0.4, 0.4, (6, 20))
    y, c = rng.normal(0, 1, (6, 40)), np.full(6, 50.0)
    g = np.asarray(E.ref_psi_grad(cfg, u, p, c, y), np.float64)
    gn = np.zeros_like(g)
    for k in range(40):
        e = np.zeros(40); e[k] = 1e-6
        gn[:, k] = np.asarray(E.ref_psi(cfg, u + e, p, c, y) - E.ref_psi(cfg, u - e, p, c, y), np.float64) / 2e-6
    assert np.abs(g - gn).max() <= 1e-6 * max(1.0, np.abs(g).max())
