"""CPU restatement of the fleet-step options (TTMPC_FLEET_WARM_START, TTMPC_FLEET_SKIP_STOPPED) on
top of the fleet oracle of tests/oracle_lib.py -- TEST INFRASTRUCTURE.

``warm_start`` is the initial-guess rule the pack kernel applies; ``OracleFleet.step`` is what
``FleetPlanner.step(warm_start=..., skip_stopped=...)`` computes, with the solve in the kernel's
WARP order, so the two agree bit for bit.
"""
from __future__ import annotations

import numpy as np

from tests import oracle_lib as O

RUNNING = 0
CONVERGED = 0


def warm_start(status, u, exit_status):
    """Initial guesses of a warm-started fleet step.  status: fleet status AFTER this step's goal
    test; u [n][2N], exit_status [n]: the previous step's outputs.  Rows of RUNNING robots become
    the previous solution shifted by one step with the last control repeated if that solve
    converged, zeros otherwise; the rows of stopped robots are returned unchanged."""
    u = np.array(u, dtype=np.float64, copy=True)
    run = np.asarray(status) == RUNNING
    conv = run & (np.asarray(exit_status) == CONVERGED)
    shifted = np.concatenate([u[:, 2:], u[:, -2:]], axis=1)
    u[conv] = shifted[conv]
    u[run & ~conv] = 0.0
    return u


class OracleFleet:
    """The closed loop of FleetPlanner.step(keep_multipliers=True, warm_start, skip_stopped) on
    an oracle FleetHost.  Result rows persist between steps like the planner's device buffers."""

    FIELDS = ("u", "y", "cost", "exit_status", "inner", "pred")

    def __init__(self, fh: O.FleetHost, cfg, threads=8):
        n, N = fh.n, cfg.N_hor
        self.fh, self.cfg, self.threads = fh, cfg, threads
        self.res = dict(u=np.zeros((n, 2 * N)), y=np.zeros((n, 2 * N)), cost=np.zeros(n),
                        exit_status=np.zeros(n, np.int32), inner=np.zeros(n, np.int32),
                        pred=np.zeros((n, N, 3)))
        self.p = None
        self.solved = None

    def step(self, warm=False, skip=False):
        fh, r = self.fh, self.res
        self.p = O.fleet_pack(fh, use_libm=False)   # goal test: fh.status is this step's status
        u0 = warm_start(fh.status, r["u"], r["exit_status"]) if warm else np.zeros_like(r["u"])
        idx = np.flatnonzero(fh.status == RUNNING) if skip else np.arange(fh.n)
        self.solved = idx
        if len(idx):
            s = O.solve_batch(self.cfg, self.p[idx], u0=u0[idx], y0=r["y"][idx], threads=self.threads, warp=True)
            for k in self.FIELDS:
                r[k][idx] = s[k]
        O.fleet_advance(fh, r["u"], r["exit_status"], use_libm=False)
