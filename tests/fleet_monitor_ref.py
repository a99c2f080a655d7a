"""ctypes binding of the fleet-monitor oracle (oracle/ttfleet_monitor_oracle.c, its own library
oracle/libttfleet_monitor_oracle.so) and the host copy of struct ttmpc_fleet_monitor -- TEST
INFRASTRUCTURE.

``MonitorHost.run(fh, step)`` is what ``ttmpc_fleet_monitor_device`` computes on the fleet host
``fh`` (tests/fleet_action_steps_ref.FleetHostK); run after the oracle's step it is what
``FleetPlanner.step()`` computes with the monitor enabled, bit for bit.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from trajtrack_mpcndqn_rlboost_b200._lib import TtmpcFleet, TtmpcFleetMonitor
from tests import oracle_lib as O

MONITOR_ORACLE_PATH = os.path.join(O.ROOT, "oracle", "libttfleet_monitor_oracle.so")
BUFFERS = ("prev_xy", "clearance", "min_clearance", "contact_steps", "first_contact", "deviation_max",
           "deviation_sum", "moved_steps")
_lib = None


def load():
    """oracle/libttfleet_monitor_oracle.so (built by ``make``; compiled here when it is missing)."""
    global _lib
    if _lib is None:
        if not os.path.exists(MONITOR_ORACLE_PATH):
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", MONITOR_ORACLE_PATH,
                                   os.path.join(O.ROOT, "oracle", "ttfleet_monitor_oracle.c"), "-lm"])
        lib = C.CDLL(MONITOR_ORACLE_PATH)
        VP, I, D = C.c_void_p, C.c_int, C.c_double
        lib.ttfleet_oracle_seg_distance.argtypes = [D] * 6
        lib.ttfleet_oracle_seg_distance.restype = D
        lib.ttfleet_oracle_swept_poly_distance.argtypes = [VP, I, D, D, D, D]
        lib.ttfleet_oracle_swept_poly_distance.restype = D
        lib.ttfleet_oracle_swept_disc_distance.argtypes = [D] * 8
        lib.ttfleet_oracle_swept_disc_distance.restype = D
        lib.ttfleet_oracle_polyline_distance.argtypes = [VP, I, I, D, D]
        lib.ttfleet_oracle_polyline_distance.restype = D
        lib.ttfleet_oracle_monitor.argtypes = [C.POINTER(TtmpcFleet), C.POINTER(TtmpcFleetMonitor)]
        _lib = lib
    return _lib


def swept_poly_distance(xy, p0, p1):
    """Distance of the chord p0 -> p1 to the polygon ring xy [nv][2]."""
    xy = np.ascontiguousarray(xy, np.float64).reshape(-1, 2)
    return load().ttfleet_oracle_swept_poly_distance(xy.ctypes.data, len(xy), float(p0[0]), float(p0[1]),
                                                     float(p1[0]), float(p1[1]))


def swept_disc_distance(p0, p1, c0, c1):
    """Least distance of a robot moving p0 -> p1 to an obstacle centre moving c0 -> c1 in the same step."""
    return load().ttfleet_oracle_swept_disc_distance(*map(float, (*p0, *p1, *c0, *c1)))


def polyline_distance(ref, lo, hi, px, py):
    """Distance of (px, py) to the polyline through rows lo .. hi-1 of ref [][3]."""
    ref = np.ascontiguousarray(ref, np.float64)
    return load().ttfleet_oracle_polyline_distance(ref.ctypes.data, int(lo), int(hi), float(px), float(py))


class MonitorHost:
    """Host copy of struct ttmpc_fleet_monitor.  poly_xy [n or 1][P][V][2] / poly_nv [n or 1][P] or None."""

    def __init__(self, state, poly_xy=None, poly_nv=None, robot_radius=0.0, moving_radius=1.6,
                 stop_on_contact=False):
        n = len(state)
        self.n = n
        self.poly_xy = None if poly_xy is None else np.ascontiguousarray(poly_xy, np.float64)
        self.poly_nv = None if poly_nv is None else np.ascontiguousarray(poly_nv, np.int32)
        self.robot_radius, self.moving_radius = float(robot_radius), float(moving_radius)
        self.stop_on_contact = bool(stop_on_contact)
        self.prev_xy = np.ascontiguousarray(np.asarray(state, np.float64)[:, :2]).copy()
        self.clearance = np.full(n, np.inf)
        self.min_clearance = np.full(n, np.inf)
        self.contact_steps = np.zeros(n, np.int32)
        self.first_contact = np.full(n, -1, np.int32)
        self.deviation_max = np.zeros(n)
        self.deviation_sum = np.zeros(n)
        self.moved_steps = np.zeros(n, np.int32)

    def struct(self, step=0, ptr=lambda a: a.ctypes.data):
        """The struct over this host copy, or over other arrays of the same names: ptr(array) -> address."""
        m = TtmpcFleetMonitor()
        if self.poly_xy is not None:
            m.poly_xy, m.poly_nv = ptr(self.poly_xy), ptr(self.poly_nv)
            m.max_poly, m.max_pv = self.poly_xy.shape[1], self.poly_xy.shape[2]
            m.poly_shared = 1 if self.poly_xy.shape[0] == 1 else 0
        m.robot_radius, m.moving_radius = self.robot_radius, self.moving_radius
        m.stop_on_contact = 1 if self.stop_on_contact else 0
        m.step = int(step)
        for name in BUFFERS:
            setattr(m, name, ptr(getattr(self, name)))
        return m

    def run(self, fh, step):
        """The monitor of the step that just ran on fh (FleetHostK): updates these buffers and, with
        stop_on_contact, fh.status."""
        load().ttfleet_oracle_monitor(C.byref(fh.struct()), C.byref(self.struct(step)))
