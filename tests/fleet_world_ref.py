"""ctypes binding of the map-selection oracle (oracle/ttfleet_world_oracle.c, its own library
oracle/libttfleet_world_oracle.so), the host copy of struct ttmpc_fleet_world and a restatement of the
grid query rule -- TEST INFRASTRUCTURE.

``WorldHost.select(cfg, state)`` is what ``ttmpc_fleet_world_select_device`` computes for robots at
``state``, by brute force over the whole map (no grid), bit for bit.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess

import numpy as np

from trajtrack_mpcndqn_rlboost_b200._lib import TtmpcConfig, TtmpcFleetWorld
from trajtrack_mpcndqn_rlboost_b200.fleet import world_grid
from tests import oracle_lib as O

WORLD_ORACLE_PATH = os.path.join(O.ROOT, "oracle", "libttfleet_world_oracle.so")
_lib = None


def load():
    """oracle/libttfleet_world_oracle.so (built by ``make``; compiled here when it is missing)."""
    global _lib
    if _lib is None:
        if not os.path.exists(WORLD_ORACLE_PATH):
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", WORLD_ORACLE_PATH,
                                   os.path.join(O.ROOT, "oracle", "ttfleet_world_oracle.c"), "-lm"])
        lib = C.CDLL(WORLD_ORACLE_PATH)
        VP, I, D = C.c_void_p, C.c_int, C.c_double
        lib.ttfleet_oracle_world_distance.argtypes = [VP, I, D, D]
        lib.ttfleet_oracle_world_distance.restype = D
        lib.ttfleet_oracle_world_select.argtypes = [C.POINTER(TtmpcConfig), I, VP, C.POINTER(TtmpcFleetWorld), VP, VP, VP]
        _lib = lib
    return _lib


def distance(xy, px, py):
    """d_o of include/ttmpc.h: 0 inside the ring xy [nv][2] (even-odd rule), else the least edge distance."""
    xy = np.ascontiguousarray(xy, np.float64).reshape(-1, 2)
    return load().ttfleet_oracle_world_distance(xy.ctypes.data, len(xy), float(px), float(py))


class WorldHost:
    """Host copy of a map: poly_xy [M][max_pv][2], poly_nv [M], rows [M][nstcobs], bbox [M][4], reach, and
    the grid of fleet.world_grid (or of the given arrays)."""

    def __init__(self, poly_xy, poly_nv, rows, bbox, reach, cell=None, grid=None):
        self.poly_xy = np.ascontiguousarray(poly_xy, np.float64)
        self.poly_nv = np.ascontiguousarray(poly_nv, np.int32)
        self.rows = np.ascontiguousarray(rows, np.float64)
        self.bbox = np.ascontiguousarray(bbox, np.float64).reshape(-1, 4)
        self.reach = float(reach)
        self.cell = float(reach if cell is None else cell)
        g = world_grid(self.bbox, self.cell) if grid is None else grid
        self.origin_x, self.origin_y, self.nx, self.ny = float(g[0]), float(g[1]), int(g[2]), int(g[3])
        self.cell_start = np.ascontiguousarray(g[4], np.int32)
        self.cell_items = np.ascontiguousarray(g[5], np.int32)

    @classmethod
    def from_hulls(cls, hulls, rows, reach, cell=None):
        """From convex rings [M][nv][2] of one vertex count and their rows [M][nstcobs]."""
        xy = np.asarray(hulls, np.float64)
        bbox = np.concatenate([xy.min(1), xy.max(1)], 1) if len(xy) else np.zeros((0, 4))
        return cls(xy, np.full(len(xy), xy.shape[1], np.int32), rows, bbox, reach, cell)

    @classmethod
    def from_planner(cls, fp):
        w = fp.world
        return cls(fp.world_poly_xy.cpu().numpy(), fp.world_poly_nv.cpu().numpy(), fp.world_rows.cpu().numpy(),
                   fp.world_bbox.cpu().numpy(), w.reach, w.cell,
                   (w.origin_x, w.origin_y, w.nx, w.ny, fp.world_cell_start.cpu().numpy(),
                    fp.world_cell_items.cpu().numpy()))

    @property
    def M(self):
        return len(self.poly_nv)

    def struct(self, ptr=lambda a: a.ctypes.data):
        """The struct over this host copy, or over other arrays of the same names: ptr(array) -> address."""
        w = TtmpcFleetWorld()
        w.M, w.max_pv = self.M, self.poly_xy.shape[1] if self.poly_xy.ndim == 3 else 3
        if self.M:
            w.poly_xy, w.poly_nv, w.rows, w.bbox = (ptr(a) for a in (self.poly_xy, self.poly_nv, self.rows, self.bbox))
            w.cell_start, w.cell_items = ptr(self.cell_start), ptr(self.cell_items)
        w.reach, w.origin_x, w.origin_y, w.cell, w.nx, w.ny = (self.reach, self.origin_x, self.origin_y, self.cell,
                                                               self.nx, self.ny)
        return w

    def select(self, cfg, state):
        """(stc [n][Nstcobs*nstcobs], slot_poly [n][Nstcobs], n_reach [n]) of the oracle."""
        state = np.ascontiguousarray(state, np.float64).reshape(-1, 3)
        n, K = len(state), cfg.Nstcobs
        stc = np.zeros((n, K * cfg.nstcobs))
        slots = np.zeros((n, K), np.int32)
        reach = np.zeros(n, np.int32)
        load().ttfleet_oracle_world_select(C.byref(cfg), n, state.ctypes.data, C.byref(self.struct()),
                                           stc.ctypes.data, slots.ctypes.data, reach.ctypes.data)
        return stc, slots, reach

    # ---------------------------------------------------------------- the grid query rule
    def _axis(self, c, origin, n):
        a = math.floor((c - self.reach - origin) / self.cell) - 1.0
        b = math.floor((c + self.reach - origin) / self.cell) + 1.0
        if not a <= b or b < 0.0 or a > n - 1:
            return 0, -1
        return (0 if a < 0 else int(a)), (n - 1 if b > n - 1 else int(b))

    def query(self, x, y):
        """The polygons the kernel handles for a robot at (x, y): each visited cell's items, a polygon
        only in the lowest visited cell of its box's cell range.  Returns the list in visiting order."""
        qx0, qx1 = self._axis(x, self.origin_x, self.nx)
        qy0, qy1 = self._axis(y, self.origin_y, self.ny)

        def cell(v, origin, n):
            a = math.floor((v - origin) / self.cell)
            return 0 if not a >= 0 else min(int(a), n - 1)
        out = []
        for cy in range(qy0, qy1 + 1):
            for cx in range(qx0, qx1 + 1):
                c = cy * self.nx + cx
                for o in self.cell_items[self.cell_start[c]:self.cell_start[c + 1]].tolist():
                    bb = self.bbox[o]
                    if (cx == max(qx0, cell(bb[0], self.origin_x, self.nx))
                            and cy == max(qy0, cell(bb[1], self.origin_y, self.ny))):
                        out.append(o)
        return out


def python_select(dist, reach, K):
    """Independent selection: the eligible (d, o) sorted with Python's sorted, the first K in map order."""
    eligible = sorted((d, o) for o, d in enumerate(dist) if d <= reach)
    return sorted(o for _, o in eligible[:K]), len(eligible)
