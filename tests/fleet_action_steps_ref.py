"""CPU restatement of the k-step fleet step (``ttmpc_fleet.action_steps = k > 1``) on top of the
fleet oracle of tests/oracle_lib.py -- TEST INFRASTRUCTURE.

The k-step form is composed from the oracle's one-step entry points, which stay as they are:

* pack: the goal test reads the FIRST control of the previous solution (``InterfaceMpc._last_action
  = actions[0]``), the packed ``v_init, w_init`` are ``last_u`` = the LAST applied control
  (``past_actions[-1]``), and the reference window is ``[idx - k, idx + 5k)``.
* advance: ``run_solver`` computes each of its k taken states from the state the step started in
  and continues from the last one, so the state takes one RK4 step with u[k-1], which is also the
  new ``last_u``; the obstacles move once.
* warm start: the previous solution shifted by k controls, the last control repeated.

``OracleFleetK.step`` is what ``FleetPlanner(action_steps=k).step(...)`` computes, with the solve in
the kernel's WARP order, so the two agree bit for bit.
"""
from __future__ import annotations

import numpy as np

from tests import oracle_lib as O
from tests.fleet_options_ref import CONVERGED, RUNNING, OracleFleet


class FleetHostK(O.FleetHost):
    """FleetHost whose struct carries ``action_steps``."""

    def __init__(self, *args, action_steps=1, **kw):
        super().__init__(*args, **kw)
        self.action_steps = int(action_steps)

    def struct(self):
        f = super().struct()
        f.action_steps = self.action_steps
        return f


def fleet_pack_k(fh: FleetHostK, prev_u, use_libm: bool):
    """Pack of a k-step fleet.  prev_u [n][2N]: the previous step's solutions (zeros before the
    first step).  For k = 1 this is O.fleet_pack."""
    if fh.action_steps == 1:
        return O.fleet_pack(fh, use_libm)
    applied = fh.last_u.copy()
    fh.last_u[:] = np.asarray(prev_u, dtype=np.float64)[:, :2]   # what the goal test reads
    try:
        p = O.fleet_pack(fh, use_libm)
    finally:
        fh.last_u[:] = applied
    p[:, 6:8] = applied                                           # v_init, w_init
    return p


def fleet_advance_k(fh: FleetHostK, u, exit_status, use_libm: bool):
    """Advance of a k-step fleet: the oracle's advance with u[k-1] in place of u[0].  For k = 1
    this is O.fleet_advance."""
    u = np.asarray(u, dtype=np.float64)
    j = 2 * (fh.action_steps - 1)
    uk = np.zeros_like(u)
    uk[:, :u.shape[1] - j] = u[:, j:]
    O.fleet_advance(fh, uk, exit_status, use_libm)


def warm_start_k(status, u, exit_status, k):
    """Initial guesses of a warm-started k-step fleet step: u'[j] = u[min(j + k, N - 1)] for the
    RUNNING robots whose previous solve converged, zeros for the other RUNNING robots, the rows of
    stopped robots unchanged.  For k = 1 this is fleet_options_ref.warm_start."""
    u = np.array(u, dtype=np.float64, copy=True)
    o = np.arange(u.shape[1])
    src = np.minimum(o + 2 * k, u.shape[1] - 2 + (o & 1))
    run = np.asarray(status) == RUNNING
    conv = run & (np.asarray(exit_status) == CONVERGED)
    u[conv] = u[conv][:, src]
    u[run & ~conv] = 0.0
    return u


class OracleFleetK(OracleFleet):
    """The closed loop of FleetPlanner(action_steps=k).step(keep_multipliers=True, warm_start,
    skip_stopped) on an oracle FleetHostK."""

    def step(self, warm=False, skip=False):
        fh, r, k = self.fh, self.res, self.fh.action_steps
        self.p = fleet_pack_k(fh, r["u"], use_libm=False)
        u0 = warm_start_k(fh.status, r["u"], r["exit_status"], k) if warm else np.zeros_like(r["u"])
        idx = np.flatnonzero(fh.status == RUNNING) if skip else np.arange(fh.n)
        self.solved = idx
        if len(idx):
            s = O.solve_batch(self.cfg, self.p[idx], u0=u0[idx], y0=r["y"][idx], threads=self.threads, warp=True)
            for name in self.FIELDS:
                r[name][idx] = s[name]
        fleet_advance_k(fh, r["u"], r["exit_status"], use_libm=False)
