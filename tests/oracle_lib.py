"""ctypes binding of the CPU oracle (oracle/libttmpc_oracle.so) -- TEST INFRASTRUCTURE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
leg may import this module.  The product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from trajtrack_mpcndqn_rlboost_b200._lib import TtmpcConfig, TtmpcResult, TtdqnLayout, TtdqnQnet, TtmpcFleet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_PATH = os.path.join(ROOT, "oracle", "libttmpc_oracle.so")


class OracleStatus(C.Structure):
    _fields_ = [("exit_status", C.c_int), ("outer_iters", C.c_int), ("inner_iters", C.c_int),
                ("last_fpr", C.c_double), ("delta_y_norm", C.c_double), ("f2_norm", C.c_double),
                ("penalty", C.c_double), ("cost", C.c_double),
                ("n_cost_evals", C.c_longlong), ("n_grad_evals", C.c_longlong)]


_lib = None


def build():
    src = [os.path.join(ROOT, "oracle", f) for f in ("ttmpc_oracle.c", "ttdqn_oracle.c", "ttfleet_oracle.c")]
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", ORACLE_PATH,
                           *src, "-lm", "-lpthread"])


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_PATH):
            build()
        lib = C.CDLL(ORACLE_PATH)
        VP, I, D = C.c_void_p, C.c_int, C.c_double
        CFG = C.POINTER(TtmpcConfig)
        lib.ttmpc_oracle_eval.argtypes = [CFG, VP, VP, VP, VP, VP]
        lib.ttmpc_oracle_psi.argtypes = [CFG, VP, VP, D, VP]
        lib.ttmpc_oracle_psi.restype = D
        lib.ttmpc_oracle_psi_grad.argtypes = [CFG, VP, VP, D, VP, VP]
        lib.ttmpc_oracle_solve.argtypes = [CFG, VP, VP, VP, D, C.POINTER(OracleStatus)]
        lib.ttmpc_oracle_solve_batch.argtypes = [CFG, I, VP, I, I, VP, C.POINTER(TtmpcResult), I]
        lib.ttmpc_oracle_rollout.argtypes = [CFG, VP, VP, VP]
        lib.ttmpc_oracle_solve_batch_mode.argtypes = [CFG, I, VP, I, I, VP, C.POINTER(TtmpcResult), I, I]
        lib.ttmpc_oracle_eval_warp.argtypes = [CFG, VP, VP, D, VP, VP, VP, VP, VP]
        lib.ttmpc_oracle_sincos.argtypes = [D, C.POINTER(D), C.POINTER(D)]
        lib.ttmpc_oracle_panoc_mock.argtypes = [I, VP, D, I, I, C.POINTER(C.c_int), C.POINTER(D), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
        lib.ttmpc_oracle_panoc_mock.restype = I
        lib.ttmpc_oracle_lbfgs_kat.argtypes = [I, I, I, VP, VP, VP, C.POINTER(D), C.POINTER(D), I]
        lib.ttmpc_oracle_lbfgs_kat.restype = I
        lib.ttmpc_oracle_lipschitz_mock.argtypes = [VP]
        lib.ttmpc_oracle_lipschitz_mock.restype = D
        lib.ttdqn_oracle_observe_act.argtypes = [C.POINTER(TtdqnLayout), C.POINTER(TtdqnQnet), I] + [VP] * 12
        lib.ttdqn_oracle_observe.argtypes = [C.POINTER(TtdqnLayout), VP, VP, VP, VP, I, VP, VP]
        lib.ttdqn_oracle_project.argtypes = [VP, I, D, D]
        lib.ttdqn_oracle_project.restype = D
        lib.ttdqn_oracle_internal_obs.argtypes = [I, D, D, VP, VP, I, VP, VP]
        lib.ttdqn_oracle_rl_ref.argtypes = [I, D, D, VP, I, VP, I]
        lib.ttfleet_oracle_pack.argtypes = [CFG, C.POINTER(TtmpcFleet), VP, I]
        lib.ttfleet_oracle_advance.argtypes = [CFG, C.POINTER(TtmpcFleet), VP, VP, I]
        lib.ttfleet_oracle_poly_contains.argtypes = [VP, I, D, D]
        lib.ttfleet_oracle_poly_distance.argtypes = [VP, I, D, D]
        lib.ttfleet_oracle_poly_distance.restype = D
        _lib = lib
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data


def evaluate(cfg, u, p):
    lib = load()
    N = cfg.N_hor
    u = np.ascontiguousarray(u, np.float64); p = np.ascontiguousarray(p, np.float64)
    f = np.zeros(1); F1 = np.zeros(2 * N); F2 = np.zeros(max(cfg.Ndynobs, 1))
    lib.ttmpc_oracle_eval(C.byref(cfg), _p(u), _p(p), _p(f), _p(F1), _p(F2))
    return float(f[0]), F1, F2[:cfg.Ndynobs]


def psi(cfg, u, p, c, y=None):
    lib = load()
    u = np.ascontiguousarray(u, np.float64); p = np.ascontiguousarray(p, np.float64)
    y = None if y is None else np.ascontiguousarray(y, np.float64)
    return lib.ttmpc_oracle_psi(C.byref(cfg), _p(u), _p(p), float(c), _p(y))


def psi_grad(cfg, u, p, c, y=None):
    lib = load()
    u = np.ascontiguousarray(u, np.float64); p = np.ascontiguousarray(p, np.float64)
    y = None if y is None else np.ascontiguousarray(y, np.float64)
    g = np.zeros(2 * cfg.N_hor)
    lib.ttmpc_oracle_psi_grad(C.byref(cfg), _p(u), _p(p), float(c), _p(y), _p(g))
    return g


def eval_warp(cfg, u, p, c=0.0, y=None):
    """f, F2, psi, grad psi with the GPU's operation order (bit-exact mirror)."""
    lib = load()
    u = np.ascontiguousarray(u, np.float64); p = np.ascontiguousarray(p, np.float64)
    y = None if y is None else np.ascontiguousarray(y, np.float64)
    f = np.zeros(1); ps = np.zeros(1); F2 = np.zeros(max(cfg.Ndynobs, 1)); g = np.zeros(2 * cfg.N_hor)
    lib.ttmpc_oracle_eval_warp(C.byref(cfg), _p(u), _p(p), float(c), _p(y), _p(f), _p(F2), _p(ps), _p(g))
    return float(f[0]), F2[:cfg.Ndynobs], float(ps[0]), g


def rollout(cfg, u, p):
    """States after each of the N steps of one scene (unicycle RK4 from p's start, libm order): [N, 3]."""
    lib = load()
    u = np.ascontiguousarray(u, np.float64); p = np.ascontiguousarray(p, np.float64)
    st = np.zeros((cfg.N_hor, 3))
    lib.ttmpc_oracle_rollout(C.byref(cfg), _p(u), _p(p), _p(st))
    return st


def sincos(x):
    lib = load()
    s = C.c_double(); c = C.c_double()
    lib.ttmpc_oracle_sincos(float(x), C.byref(s), C.byref(c))
    return s.value, c.value


def lbfgs_kat(mem, gs, xs, q, cbfgs=False):
    """update_hessian(g_i, x_i) for every row, then apply_hessian(q) of the restated L-BFGS."""
    lib = load()
    gs = np.ascontiguousarray(gs, np.float64); xs = np.ascontiguousarray(xs, np.float64)
    q = np.array(q, np.float64)
    a = C.c_double(0.0); r = C.c_double(0.0)
    code = lib.ttmpc_oracle_lbfgs_kat(gs.shape[1], int(mem), gs.shape[0], _p(gs), _p(xs), _p(q), C.byref(a), C.byref(r), int(cbfgs))
    return dict(direction=q, alpha0=a.value, rho0=r.value, accepted=code // 100, active=code % 100)


def lipschitz_mock(u3):
    u = np.array(u3, np.float64)
    return load().ttmpc_oracle_lipschitz_mock(_p(u))


def panoc_mock(which, u0, tolerance, lbfgs_memory, max_iter):
    """The restated PANOC engine on one of the two unit-test problems of optimization_engine's mocks.rs."""
    lib = load()
    u = np.array(u0, np.float64)
    it = C.c_int(0); fpr = C.c_double(0.0); nc = C.c_longlong(0); ng = C.c_longlong(0)
    st = lib.ttmpc_oracle_panoc_mock(int(which), _p(u), float(tolerance), int(lbfgs_memory), int(max_iter),
                                     C.byref(it), C.byref(fpr), C.byref(nc), C.byref(ng))
    return dict(u=u, exit_status=st, iterations=it.value, norm_fpr=fpr.value, cost_evals=nc.value, grad_evals=ng.value)


def solve_batch(cfg, p, u0=None, y0=None, c0=None, threads=1, warp=False):
    """Same outputs as BatchSolver.run (dict of numpy arrays).
    warp=True uses the GPU's operation order (bit-exact mirror of the kernel)."""
    lib = load()
    p = np.ascontiguousarray(p, np.float64)
    n, N = p.shape[0], cfg.N_hor
    u = np.zeros((n, 2 * N)) if u0 is None else np.array(u0, np.float64, order="C").reshape(n, 2 * N)
    y = np.zeros((n, 2 * N)) if y0 is None else np.array(y0, np.float64, order="C").reshape(n, 2 * N)
    c0a = None if c0 is None else np.ascontiguousarray(np.broadcast_to(np.asarray(c0, np.float64), (n,)))
    out = dict(cost=np.zeros(n), exit_status=np.zeros(n, np.int32), outer=np.zeros(n, np.int32),
               inner=np.zeros(n, np.int32), fpr=np.zeros(n), f1=np.zeros(n), f2=np.zeros(n),
               pen=np.zeros(n), pred=np.zeros((n, N, 3)), evals=np.zeros((n, 4), np.int64))
    res = TtmpcResult(u=_p(u), cost=_p(out["cost"]), exit_status=_p(out["exit_status"]),
                      outer_iters=_p(out["outer"]), inner_iters=_p(out["inner"]), last_fpr=_p(out["fpr"]),
                      f1_infeas=_p(out["f1"]), f2_norm=_p(out["f2"]), penalty=_p(out["pen"]), y=_p(y),
                      pred_states=_p(out["pred"]), evals=_p(out["evals"]))
    lib.ttmpc_oracle_solve_batch_mode(C.byref(cfg), n, _p(p), int(u0 is not None), int(y0 is not None),
                                      _p(c0a), C.byref(res), int(threads), int(warp))
    out["u"] = u; out["y"] = y
    return out


def observe_act(lay, weights, agent, xy, off, sol, cnt, internal=None, old_ext=None):
    lib = load()
    n = len(agent)
    ns = lay.num_segments
    n_ext = (4 if lay.use_memory else 2) * ns
    agent = np.ascontiguousarray(agent, np.float64)
    internal = np.zeros((n, lay.n_internal), np.float32) if internal is None else \
        np.ascontiguousarray(internal, np.float32)
    old_ext = np.zeros((n, 2 * ns), np.float32) if old_ext is None else old_ext
    ext = np.zeros((n, n_ext), np.float32)
    q = np.zeros((n, weights.n_out), np.float32)
    act = np.zeros(n, np.int32)
    seg = np.zeros((n, ns)); ray = np.zeros((n, ns))
    qs = weights.host_struct()
    lib.ttdqn_oracle_observe_act(C.byref(lay), C.byref(qs), n, _p(agent), _p(xy), _p(off), _p(sol),
                                 _p(cnt), _p(internal), _p(old_ext), _p(ext), _p(q), _p(act), _p(seg),
                                 _p(ray))
    return dict(ext=ext, q=q, action=act, seg=seg, ray=ray, old_ext=old_ext)


class FleetHost:
    """Host-side fleet state (numpy) for the fleet-step oracle; same members as struct ttmpc_fleet."""

    def __init__(self, cfg, state, goal, ref_traj, ref_len, stc, tuning, base_speed, low_speed,
                 stc_weight=1e3, dyn_weight=1e3, dyn_cur=None, dyn_disp=None, dyn_size=1.6, other=None):
        f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        self.cfg = cfg
        self.state, self.goal = f64(state).copy(), f64(goal)
        self.n = len(self.state)
        self.last_u = np.zeros((self.n, 2))
        self.idx_ref = np.zeros(self.n, dtype=np.int32)
        self.status = np.zeros(self.n, dtype=np.int32)
        self.ref_traj, self.ref_len = f64(ref_traj), np.ascontiguousarray(ref_len, dtype=np.int32)
        self.stc = f64(stc)
        self.stc_shared = 1 if self.stc.ndim == 1 else 0  # one row block for every robot, or [n][...]
        self.tuning, self.base_speed, self.low_speed = list(tuning), float(base_speed), float(low_speed)
        self.stc_weight, self.dyn_weight, self.dyn_size = float(stc_weight), float(dyn_weight), float(dyn_size)
        self.other = None if other is None else f64(other)
        self.dyn_cur = None if dyn_cur is None else f64(dyn_cur).copy()
        self.dyn_last = None if dyn_cur is None else f64(dyn_cur).copy()
        self.dyn_disp = None if dyn_disp is None else f64(dyn_disp)
        self.hint = None
        self.use_hint = None
        self.sw_state = None     # HintSwitcher: set sw_state [n][2] int32, sw_poly_xy [n|1][P][V][2], sw_poly_nv [n|1][P]
        self.sw_poly_xy = self.sw_poly_nv = None
        self.sw_params = (10.0, 2.0, 10)

    def struct(self):
        f = TtmpcFleet()
        f.n, f.ref_stride = self.n, self.ref_traj.shape[1]
        f.state, f.goal, f.last_u = _p(self.state), _p(self.goal), _p(self.last_u)
        f.idx_ref, f.status = _p(self.idx_ref), _p(self.status)
        f.ref_traj, f.ref_len, f.stc = _p(self.ref_traj), _p(self.ref_len), _p(self.stc)
        f.stc_shared, f.action_steps = self.stc_shared, 1
        f.n_dyn_live = 0 if self.dyn_cur is None else self.dyn_cur.shape[1]
        f.other, f.dyn = _p(self.other), None
        f.dyn_cur, f.dyn_last, f.dyn_disp = _p(self.dyn_cur), _p(self.dyn_last), _p(self.dyn_disp)
        f.dyn_size = self.dyn_size
        for i, v in enumerate(self.tuning):
            f.tuning[i] = float(v)
        f.base_speed, f.low_speed = self.base_speed, self.low_speed
        f.stc_weight, f.dyn_weight = self.stc_weight, self.dyn_weight
        if self.hint is not None:
            self.hint = np.ascontiguousarray(self.hint, dtype=np.float64)
            self.use_hint = np.ascontiguousarray(self.use_hint, dtype=np.int32)
            f.hint, f.use_hint = _p(self.hint), _p(self.use_hint)
        if self.sw_state is not None:
            self.sw_state = np.ascontiguousarray(self.sw_state, dtype=np.int32)
            self.sw_poly_xy = np.ascontiguousarray(self.sw_poly_xy, dtype=np.float64)
            self.sw_poly_nv = np.ascontiguousarray(self.sw_poly_nv, dtype=np.int32)
            f.sw_state, f.sw_poly_xy, f.sw_poly_nv = _p(self.sw_state), _p(self.sw_poly_xy), _p(self.sw_poly_nv)
            f.sw_max_poly, f.sw_max_pv = self.sw_poly_xy.shape[1], self.sw_poly_xy.shape[2]
            f.sw_poly_shared = 1 if self.sw_poly_xy.shape[0] == 1 and self.n != 1 else (1 if self.sw_poly_xy.shape[0] == 1 else 0)
            f.sw_switch_distance, f.sw_detach_distance, f.sw_detach_steps = self.sw_params
            f.sw_dyn_radius = 1.6
        return f


def fleet_pack(fh: FleetHost, use_libm: bool):
    lib = load()
    n_p = 2 * fh.cfg.ns + fh.cfg.nu + fh.cfg.nq + fh.cfg.ns * fh.cfg.N_hor + fh.cfg.N_hor + \
        fh.cfg.ns * fh.cfg.N_hor * fh.cfg.Nother + fh.cfg.Nstcobs * fh.cfg.nstcobs + \
        fh.cfg.Ndynobs * fh.cfg.ndynobs * fh.cfg.N_hor + 2 * fh.cfg.N_hor
    p = np.zeros((fh.n, n_p))
    f = fh.struct()
    lib.ttfleet_oracle_pack(C.byref(fh.cfg), C.byref(f), _p(p), 1 if use_libm else 0)
    return p


def fleet_advance(fh: FleetHost, u, exit_status, use_libm: bool):
    lib = load()
    u = np.ascontiguousarray(u, dtype=np.float64)
    es = None if exit_status is None else np.ascontiguousarray(exit_status, dtype=np.int32)
    f = fh.struct()
    lib.ttfleet_oracle_advance(C.byref(fh.cfg), C.byref(f), _p(u), _p(es), 1 if use_libm else 0)


def internal_obs(agent5, path, corner_samples=3, offset=0.0, max_distance=10.0):
    lib = load()
    a = np.ascontiguousarray(agent5, np.float64); xy = np.ascontiguousarray(path, np.float64).reshape(-1, 2)
    obs = np.zeros(5 + 3 * corner_samples, np.float32); prog = np.zeros(1)
    lib.ttdqn_oracle_internal_obs(corner_samples, offset, max_distance, _p(a), _p(xy), len(xy), _p(obs), _p(prog))
    return obs, float(prog[0])


def rl_ref(agent5, action, steps=20, ts=0.2, ref_speed=1.0, use_libm=True):
    lib = load()
    a = np.ascontiguousarray(agent5, np.float64)
    out = np.zeros((steps, 2))
    lib.ttdqn_oracle_rl_ref(steps, ts, ref_speed, _p(a), int(action), _p(out), 1 if use_libm else 0)
    return out


def poly_contains(xy, px, py):
    xy = np.ascontiguousarray(xy, np.float64)
    return bool(load().ttfleet_oracle_poly_contains(_p(xy), len(xy), float(px), float(py)))


def poly_distance(xy, px, py):
    xy = np.ascontiguousarray(xy, np.float64)
    return float(load().ttfleet_oracle_poly_distance(_p(xy), len(xy), float(px), float(py)))


def observe(lay, agent, rings, solid):
    """Sector / ray distances of ONE environment (ttdqn_oracle_observe): rings = list of [nv,2] arrays."""
    from trajtrack_mpcndqn_rlboost_b200.dqn import pack_geometry
    xy, off, sol, cnt = pack_geometry(lay, [rings], [solid])
    agent = np.ascontiguousarray(agent, np.float64)
    seg = np.zeros(lay.num_segments); ray = np.zeros(lay.num_segments)
    load().ttdqn_oracle_observe(C.byref(lay), _p(agent), _p(xy[0]), _p(off[0]), _p(sol[0]), int(cnt[0]), _p(seg), _p(ray))
    return seg, ray
