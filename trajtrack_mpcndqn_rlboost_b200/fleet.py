"""Batched, device-resident counterpart of ``InterfaceMpc`` for a fleet of independent robots.

One ``FleetPlanner.step()`` does, for every robot at once and without leaving the GPU, what the
reference's control loop does per robot per step (src/main.py:155-172, decision_mode 1):

    original_ref_traj, _ = traj_gen.get_local_ref_traj()     # interface_mpc.py:72-79
    traj_gen.update_dynamic_constraints(pred)                 # main.py:80-89 est_dyn_obs_positions
    action, pred_states, cost = traj_gen.get_action(ref)      # interface_mpc.py:80-92

through ``ttmpc_fleet_step_device`` (pack -> solve -> advance, include/ttmpc.h).  With
``FleetPlanner.enable_monitor`` every step is followed by ``ttmpc_fleet_monitor_device``, which
records per robot on the device how close it came to its obstacles over the step (swept clearance,
contacts) and how far it was from its reference path.  With ``FleetPlanner.set_world`` the robots
share one static map of any size, and every step starts with ``ttmpc_fleet_world_select_device``,
which writes each robot's nearest map polygons into its static slots.  The first global
reference trajectories are sampled on the host with the same
``TrajectoryGenerator.get_global_ref_traj`` the single-robot mirror uses.  Tasks queued with
``FleetPlanner.set_tasks`` are taken on the device (``ttmpc_fleet_step_tasks_device``) and their
trajectories are sampled there, from the state in which a robot takes the task; they agree with
the host sampler to within a few ulps, not bit for bit (the device uses ``sqrt(fma(dx, dx, dy*dy))``
and its own 1-ulp atan2 where Python uses ``math.hypot`` and ``math.atan2``).
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from .geometry import convex_hull, polygon_halfspace_representation
from .mpc_config import Configurator
from .planner import TrajectoryGenerator

RUNNING, REACHED, FAILED, BAD_TASK, COLLIDED = 0, 1, 2, 3, 4
GOAL_REACH = 0.08  # a robot that stops at a goal is within its 5 cm box: at most 0.0708 m away
DYN_OBS_SIZE = 0.8 + 0.8  # main.py:32


def world_grid(bbox: np.ndarray, cell: float):
    """The uniform grid of ``ttmpc_fleet_world`` (include/ttmpc.h) over boxes bbox [M][4] (xmin, ymin,
    xmax, ymax): origin at the boxes' least corner, ``nx x ny`` cells of size cell, and polygon o
    listed, ascending within a cell, in every cell its box overlaps.  Returns (origin_x, origin_y, nx,
    ny, cell_start [nx*ny+1] int32, cell_items int32)."""
    bbox = np.asarray(bbox, np.float64).reshape(-1, 4)
    M = len(bbox)
    if M == 0:
        return 0.0, 0.0, 1, 1, np.zeros(2, np.int32), np.zeros(0, np.int32)
    ox, oy = float(bbox[:, 0].min()), float(bbox[:, 1].min())
    nx = int(np.floor((bbox[:, 2].max() - ox) / cell)) + 1
    ny = int(np.floor((bbox[:, 3].max() - oy) / cell)) + 1
    if nx * ny >= 2 ** 31 - 1:
        raise ValueError(f"world_grid: {nx} x {ny} cells of {cell} m do not fit the grid's int32 offsets")

    def cells(v, o, n):  # floor((v - origin) / cell) in IEEE double, as the kernel computes it
        return np.clip(np.floor((v - o) / cell), 0, n - 1).astype(np.int64)
    bx0, bx1 = cells(bbox[:, 0], ox, nx), cells(bbox[:, 2], ox, nx)
    by0, by1 = cells(bbox[:, 1], oy, ny), cells(bbox[:, 3], oy, ny)
    wx = bx1 - bx0 + 1
    cnt = wx * (by1 - by0 + 1)
    o = np.repeat(np.arange(M), cnt)
    k = np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    c = (by0[o] + k // wx[o]) * nx + bx0[o] + k % wx[o]
    order = np.lexsort((o, c))
    start = np.zeros(nx * ny + 1, np.int64)
    start[1:] = np.cumsum(np.bincount(c, minlength=nx * ny))
    if start[-1] >= 2 ** 31:
        raise ValueError("world_grid: more cell entries than int32 offsets hold")
    return ox, oy, nx, ny, start.astype(np.int32), o[order].astype(np.int32)


def work_mode(config: Configurator, mode: str = "work"):
    """(tuning_params, base_speed) of TrajectoryGenerator.set_work_mode (trajectory_generator.py:117-139)."""
    c = config
    if mode == "aligning":
        tuning = [0.0] * 10
        tuning[2] = 100
        return tuning, c.lin_vel_max * c.medium_speed
    tuning = [c.qpos, c.qvel, c.qtheta, c.lin_vel_penalty, c.ang_vel_penalty,
              c.qpN, c.qthetaN, c.qrpd, c.lin_acc_penalty, c.ang_acc_penalty]
    speed = {"safe": c.low_speed, "work": c.high_speed, "super": c.full_speed}
    if mode not in speed:
        raise ModuleNotFoundError(f"There is no mode called {mode}.")
    return tuning, c.lin_vel_max * speed[mode]


class FleetPlanner:
    """n robots, each with its own start, goal, reference path and (optionally) obstacles."""

    def __init__(self, config: Configurator, init_states: np.ndarray, goal_states: np.ndarray,
                 ref_paths: Sequence[Sequence], mode: str = "work", device: str = "cuda",
                 stc_weights: float = 1e3, dyn_weights: float = 1e3, action_steps: int = 1,
                 **solver_overrides):
        """action_steps: controls of each solution a robot applies before its next solve
        (``config.action_steps``; pass it to mirror a configuration).  1..N_hor, checked by the
        first ``step()``; values other than 1 work only through ``step()``."""
        import torch
        self.torch = torch
        self.config = config
        self.cfg = config.to_ttmpc(**solver_overrides)
        self.lib = _lib.load()
        self.n = n = len(ref_paths)
        self.N = config.N_hor
        self.np = self.lib.ttmpc_num_params(C.byref(self.cfg))
        self.action_steps = int(action_steps)
        self.tuning, self.base_speed = work_mode(config, mode)
        init_states = np.asarray(init_states, dtype=np.float64).reshape(n, 3)
        goal_states = np.asarray(goal_states, dtype=np.float64).reshape(n, 3)
        trajs = [TrajectoryGenerator.get_global_ref_traj(config.ts, path, init_states[i], self.base_speed)
                 for i, path in enumerate(ref_paths)]
        self.ref_stride = max(1, max(len(t) for t in trajs))
        ref = np.zeros((n, self.ref_stride, 3))
        for i, t in enumerate(trajs):
            ref[i, :len(t)] = t
        f64 = dict(dtype=torch.float64, device=device)
        i32 = dict(dtype=torch.int32, device=device)
        self.state = torch.tensor(init_states, **f64)
        self.goal = torch.tensor(goal_states, **f64)
        self.last_u = torch.zeros(n, 2, **f64)
        self.idx_ref = torch.zeros(n, **i32)
        self.status = torch.zeros(n, **i32)
        self.ref_traj = torch.tensor(ref, **f64)
        self.ref_len = torch.tensor([len(t) for t in trajs], **i32)
        self.stc = torch.zeros(1, config.Nstcobs * config.nstcobs, **f64)
        self.stc_shared = 1
        self.other = None
        self.dyn_cur = self.dyn_last = self.dyn_disp = None
        self.n_dyn_live = 0
        self.stc_weight, self.dyn_weight = float(stc_weights), float(dyn_weights)
        self.p = torch.empty(n, self.np, **f64)
        self.u = torch.zeros(n, 2 * self.N, **f64)
        self.y = torch.zeros(n, 2 * self.N, **f64)
        self.cost = torch.zeros(n, **f64)
        self.exit_status = torch.zeros(n, **i32)
        self.inner = torch.zeros(n, **i32)
        self.pred_states = torch.zeros(n, self.N, 3, **f64)
        self.hint = None       # [n][N][2] DQN hint positions (rl_ref) and the per-robot switch
        self.use_hint = None
        self.tasks = None      # _lib.TtmpcFleetTasks of the queued tasks (set_tasks), None: no queue
        self.task_next = None  # [n] int32: queued tasks taken so far
        self.static_polys = None  # (polygons, per_robot) of the last update_static_constraints
        self.monitor = None    # _lib.TtmpcFleetMonitor (enable_monitor), None: no monitor
        self.world = None      # _lib.TtmpcFleetWorld of the shared map (set_world), None: no map
        self.dqn_paths = None  # (path_xy, path_n) the task step keeps current (set_tasks / enable_dqn)
        self._dqn = None       # the DQN side of the step (enable_dqn), None: off
        self.steps = 0

    # ------------------------------------------------------------------ obstacles
    def update_static_constraints(self, obstacle_list, per_robot: bool = False):
        """obstacle_list: polygons shared by every robot, or (per_robot=True) one list per robot.
        Same row layout as InterfaceMpc.update_static_constraints (interface_mpc.py:62-65).  Turns a
        map of ``set_world`` off."""
        cfg = self.config
        self.world = None

        def rows(polys):
            r = [0.0] * cfg.Nstcobs * cfg.nstcobs
            for i, poly in enumerate(polys):
                b, a0, a1 = polygon_halfspace_representation(np.array(poly))
                r[i * cfg.nstcobs:(i + 1) * cfg.nstcobs] = (b + a0 + a1)
            return r
        data = [rows(pl) for pl in obstacle_list] if per_robot else [rows(obstacle_list)]
        self.stc = self.torch.tensor(np.array(data, dtype=np.float64), device=self.state.device)
        self.stc_shared = 0 if per_robot else 1
        self.static_polys = (obstacle_list, per_robot)

    def set_world(self, polygons, reach: Optional[float] = None, cell: Optional[float] = None):
        """Share one static map of any size among the robots: before every ``step()``, on the step's
        stream, ``ttmpc_fleet_world_select_device`` (include/ttmpc.h, ``ttmpc_fleet_world``) writes
        into each robot's Nstcobs static slots the map polygons nearest to it (distance <= reach,
        ranked by (distance, map index), written in map-index order).  A map of at most Nstcobs
        polygons, all within reach, gives every robot exactly what
        ``update_static_constraints(polygons)`` gives.

        polygons: convex obstacles as vertex lists, already processed (inflated) as
        ``update_static_constraints`` takes them.  Each is replaced by its convex hull, which must
        have nstcobs / 3 edges (what ``update_static_constraints`` needs to be well defined).
        reach defaults to N_hor * ts * max(|lin_vel_min|, lin_vel_max), the farthest a feasible
        rollout gets; cell, the grid's cell size, defaults to reach.  None turns the map off (as
        ``update_static_constraints`` does) and leaves no static obstacles.

        Per robot, on the device, overwritten by every step: ``stc`` [n][Nstcobs*nstcobs] (the rows
        the step packs), ``world_slots`` [n][Nstcobs] (map index per slot, -1: empty) and
        ``world_reach`` [n] (polygons within reach; more than Nstcobs: one of them got no slot)."""
        t = self.torch
        cfg = self.config
        dev = self.state.device
        K, ns = cfg.Nstcobs, cfg.nstcobs
        if polygons is None:
            self.world = None
            self.stc = t.zeros(1, K * ns, dtype=t.float64, device=dev)
            self.stc_shared = 1
            self.static_polys = None
            return
        if reach is None:
            reach = cfg.N_hor * cfg.ts * max(abs(cfg.lin_vel_min), cfg.lin_vel_max)
        reach = float(reach)
        cell = reach if cell is None else float(cell)
        if not (np.isfinite(reach) and reach > 0.0 and np.isfinite(cell) and cell > 0.0):
            raise ValueError("set_world: reach and cell must be finite and > 0")
        ne = ns // 3
        M = len(polygons)
        xy = np.zeros((M, ne, 2))
        rows = np.zeros((M, ns))
        for o, poly in enumerate(polygons):
            pts = np.asarray(poly, np.float64).reshape(-1, 2)
            if not np.isfinite(pts).all():
                raise ValueError(f"set_world: polygon {o} has a non-finite vertex")
            hull = convex_hull(pts)
            b, a0, a1 = polygon_halfspace_representation(np.array(poly))
            if len(hull) != ne or len(b) != ne:
                raise ValueError(f"set_world: polygon {o} has a hull of {len(hull)} edges, nstcobs = {ns} needs {ne}")
            xy[o] = hull
            rows[o] = b + a0 + a1
        bbox = np.concatenate([xy.min(axis=1), xy.max(axis=1)], axis=1) if M else np.zeros((0, 4))
        ox, oy, nx, ny, start, items = world_grid(bbox, cell)
        f64 = dict(dtype=t.float64, device=dev)
        self.world_poly_xy, self.world_rows, self.world_bbox = (t.tensor(a, **f64) for a in (xy, rows, bbox))
        self.world_poly_nv = t.full((M,), ne, dtype=t.int32, device=dev)
        self.world_cell_start = t.tensor(start, device=dev)
        self.world_cell_items = t.tensor(items, device=dev)
        w = _lib.TtmpcFleetWorld()
        w.M, w.max_pv = M, ne
        if M:
            w.poly_xy, w.poly_nv = self.world_poly_xy.data_ptr(), self.world_poly_nv.data_ptr()
            w.rows, w.bbox = self.world_rows.data_ptr(), self.world_bbox.data_ptr()
            w.cell_start, w.cell_items = self.world_cell_start.data_ptr(), self.world_cell_items.data_ptr()
        w.reach, w.origin_x, w.origin_y, w.cell, w.nx, w.ny = reach, ox, oy, cell, nx, ny
        self.stc = t.zeros(self.n, K * ns, **f64)
        self.stc_shared = 0
        self.world_slots = t.full((self.n, K), -1, dtype=t.int32, device=dev)
        self.world_reach = t.zeros(self.n, dtype=t.int32, device=dev)
        self.static_polys = None
        self.world = w

    def run_world_select(self, stream=None):
        """Write each robot's nearest map polygons into ``stc`` from its current state.  ``step()``
        calls this itself first.  Needs ``set_world``."""
        if self.world is None:
            raise RuntimeError("run_world_select: call set_world first")
        st = stream if stream is not None else self.torch.cuda.current_stream().cuda_stream
        _lib.check(self.lib.ttmpc_fleet_world_select_device(C.byref(self.cfg), C.byref(self._fleet_struct()),
                                                            C.byref(self.world), self.stc.data_ptr(),
                                                            self.world_slots.data_ptr(), self.world_reach.data_ptr(),
                                                            st), "ttmpc_fleet_world_select_device")

    def set_moving_obstacles(self, positions: np.ndarray, displacement_per_step: np.ndarray):
        """positions, displacement_per_step: [n][k][2].  Every step the planner sees
        est_dyn_obs_positions(last, current) (main.py:80-89) and the obstacles then move on."""
        t = self.torch
        pos = np.asarray(positions, dtype=np.float64).reshape(self.n, -1, 2)
        self.n_dyn_live = pos.shape[1]
        dev = self.state.device
        self.dyn_cur = t.tensor(pos, device=dev)
        self.dyn_last = t.tensor(pos, device=dev)
        self.dyn_disp = t.tensor(np.asarray(displacement_per_step, dtype=np.float64).reshape(self.n, -1, 2), device=dev)

    def set_hint(self, rl_ref, use_hint):
        """Hybrid mode (main.py:194-201): rl_ref [n][N][2] float64 CUDA tensor (dqn.rl_ref_device),
        use_hint [n] int32 -- where non-zero the hint replaces the reference positions."""
        self.hint, self.use_hint = rl_ref, use_hint

    def enable_hint_switch(self, polygons, per_robot: bool = False, max_switch_distance: float = 10.0,
                           min_detach_distance: float = 2.0, min_detach_steps: int = 10):
        """Let the pack kernel decide per step whether the DQN hint is used, as
        ``HintSwitcher(10, 2, 10).switch(...)`` does in main.py:129,200 (main_pre.py:27-52).
        polygons: the processed (inflated) static obstacle polygons, shared or one list per robot;
        moving obstacles enter as circle_to_rect squares of radius DYN_OBS_SIZE."""
        t = self.torch
        xy, nv = self._polygon_rings(polygons, per_robot)
        dev = self.state.device
        self.sw_poly_xy, self.sw_poly_nv = t.tensor(xy, device=dev), t.tensor(nv, device=dev)
        self.sw_shape = (xy.shape[1], xy.shape[2], 0 if per_robot else 1)
        self.sw_params = (float(max_switch_distance), float(min_detach_distance), int(min_detach_steps))
        self.sw_state = t.zeros(self.n, 2, dtype=t.int32, device=dev)
        if self.use_hint is None:
            self.use_hint = t.zeros(self.n, dtype=t.int32, device=dev)

    @staticmethod
    def _polygon_rings(polygons, per_robot: bool):
        """Vertex rings of polygons (shared, or one list per robot) in the layout the kernels read:
        xy [n or 1][max_poly][max_pv][2] float64, nv [n or 1][max_poly] int32 (0: unused slot)."""
        lists = polygons if per_robot else [polygons]
        max_poly = max(1, max(len(pl) for pl in lists))
        max_pv = max(3, max((len(poly) for pl in lists for poly in pl), default=3))
        xy = np.zeros((len(lists), max_poly, max_pv, 2))
        nv = np.zeros((len(lists), max_poly), np.int32)
        for i, pl in enumerate(lists):
            for j, poly in enumerate(pl):
                a = np.asarray(poly, np.float64).reshape(-1, 2)
                xy[i, j, :len(a)] = a
                nv[i, j] = len(a)
        return xy, nv

    # ------------------------------------------------------------------ monitor
    def enable_monitor(self, polygons=None, per_robot: Optional[bool] = None, robot_radius: float = 0.0,
                       moving_radius: float = DYN_OBS_SIZE, stop_on_contact: bool = False):
        """Run the obstacle-contact and tracking monitor (``ttmpc_fleet_monitor_device``, include/ttmpc.h)
        after every ``step()``, on the step's stream.

        polygons: static obstacles as vertex rings, shared or (per_robot=True) one list per robot;
        default: the map of ``set_world`` (its hulls, shared) when one is set, else the polygons last
        given to ``update_static_constraints``, with their per_robot flag.  The monitor measures every
        robot against every polygon it is given: with a map that is O(M) per robot and step.
        The robot is a disc of robot_radius, a moving obstacle a disc of moving_radius.  The defaults
        monitor the region the MPC's constraints exclude: the robot centre against the polygons the
        MPC sees, and the DYN_OBS_SIZE discs the pack writes for moving obstacles.

        Per robot, on the device (reset here; ``prev_xy`` starts at the current state):
        ``clearance`` (the last step's swept clearance, +inf before the first), ``min_clearance``,
        ``contact_steps`` (steps with clearance <= 0), ``first_contact`` (index of the first such
        ``step()`` call, counted from the planner's construction; -1: none), and over the steps in
        which the robot moved ``deviation_max``, ``deviation_sum`` and ``moved_steps``.
        stop_on_contact=True: a RUNNING robot in contact stops with status ``COLLIDED``."""
        t = self.torch
        use_map = polygons is None and self.world is not None
        if polygons is None and self.static_polys is not None:
            polygons, stored = self.static_polys
            per_robot = stored if per_robot is None else per_robot
        per_robot = bool(per_robot)
        if not (np.isfinite(robot_radius) and robot_radius >= 0.0 and np.isfinite(moving_radius) and moving_radius >= 0.0):
            raise ValueError("enable_monitor: radii must be finite and >= 0")
        if per_robot and polygons is not None and len(polygons) != self.n:
            raise ValueError(f"enable_monitor: {len(polygons)} polygon lists for {self.n} robots")
        dev = self.state.device
        m = _lib.TtmpcFleetMonitor()
        self.mon_poly_xy = self.mon_poly_nv = None
        if use_map and self.world.M > 0:     # the map's own tensors, kept alive here
            self.mon_poly_xy, self.mon_poly_nv = self.world_poly_xy[None], self.world_poly_nv[None]
            m.poly_xy, m.poly_nv = self.mon_poly_xy.data_ptr(), self.mon_poly_nv.data_ptr()
            m.max_poly, m.max_pv, m.poly_shared = self.world.M, self.world.max_pv, 1
        elif polygons is not None:
            xy, nv = self._polygon_rings(polygons, per_robot)
            self.mon_poly_xy, self.mon_poly_nv = t.tensor(xy, device=dev), t.tensor(nv, device=dev)
            m.poly_xy, m.poly_nv = self.mon_poly_xy.data_ptr(), self.mon_poly_nv.data_ptr()
            m.max_poly, m.max_pv, m.poly_shared = xy.shape[1], xy.shape[2], 0 if per_robot else 1
        m.robot_radius, m.moving_radius = float(robot_radius), float(moving_radius)
        m.stop_on_contact = 1 if stop_on_contact else 0
        f64 = dict(dtype=t.float64, device=dev)
        i32 = dict(dtype=t.int32, device=dev)
        self.prev_xy = self.state[:, :2].clone()
        self.clearance = t.full((self.n,), float("inf"), **f64)
        self.min_clearance = t.full((self.n,), float("inf"), **f64)
        self.contact_steps = t.zeros(self.n, **i32)
        self.first_contact = t.full((self.n,), -1, **i32)
        self.deviation_max = t.zeros(self.n, **f64)
        self.deviation_sum = t.zeros(self.n, **f64)
        self.moved_steps = t.zeros(self.n, **i32)
        for name in ("prev_xy", "clearance", "min_clearance", "contact_steps", "first_contact", "deviation_max",
                     "deviation_sum", "moved_steps"):
            setattr(m, name, getattr(self, name).data_ptr())
        self.monitor = m

    def run_monitor(self, stream=None):
        """Run the monitor on the last ``step()``.  ``step()`` calls this itself unless it is called
        with monitor=False.  Needs ``enable_monitor``."""
        if self.monitor is None:
            raise RuntimeError("run_monitor: call enable_monitor first")
        st = stream if stream is not None else self.torch.cuda.current_stream().cuda_stream
        self.monitor.step = self.steps - 1
        _lib.check(self.lib.ttmpc_fleet_monitor_device(C.byref(self.cfg), C.byref(self._fleet_struct()),
                                                       C.byref(self.monitor), st), "ttmpc_fleet_monitor_device")

    # ------------------------------------------------------------------ tasks
    def ref_rows_bound(self, start_xy, path) -> int:
        """An upper bound of the rows ``get_global_ref_traj`` gives for ``path`` from any start within
        GOAL_REACH of ``start_xy``: every row but the last advances the walker by base_speed*ts of
        arc length, so rows <= length / (base_speed*ts) + 1 (+1 for rounding)."""
        nodes = np.asarray(path, dtype=np.float64).reshape(-1, 2)
        if len(nodes) == 0:
            return 1
        length = float(np.hypot(*(nodes[0] - np.asarray(start_xy, dtype=np.float64)[:2]))) + GOAL_REACH
        length += float(np.hypot(*np.diff(nodes, axis=0).T).sum()) if len(nodes) > 1 else 0.0
        return int(length / (self.base_speed * self.config.ts)) + 2

    def set_tasks(self, goals: Sequence[Sequence], paths: Sequence[Sequence], dqn_paths=None):
        """Replace every robot's task queue.  goals[e]: the goals [3] of robot e's tasks, paths[e]: one
        polyline (list of (x, y) nodes) per task.  A robot that has reached its goal takes its next
        task inside the step, on the device: ``InterfaceMpc.initialization(state, goal, path, mode)``
        (include/ttmpc.h, ``ttmpc_fleet_tasks``); ``task_next`` counts the tasks taken, and
        ``REACHED`` then means that the last task is done.  A task that cannot be driven stops its
        robot with status ``BAD_TASK``.

        ``ref_stride`` grows, keeping the rows, to cover every queued task from a start within
        GOAL_REACH of the goal before it.  dqn_paths=(path_xy [n][m][2] float64, path_n [n] int32),
        the CUDA tensors the hybrid loop passes to ``dqn.internal_obs_device``: the step writes each
        robot's current path there when it takes a task (m must hold the longest task path).  With
        the DQN enabled (``enable_dqn``) and dqn_paths not given, its path tensors are the ones kept."""
        t = self.torch
        n = self.n
        if dqn_paths is None and self._dqn is not None:
            dqn_paths = self._dqn.paths
        if len(goals) != n or len(paths) != n or any(len(g) != len(p) for g, p in zip(goals, paths)):
            raise ValueError("set_tasks: one list of goals and one of paths per robot, of equal lengths")
        T = max(len(g) for g in goals)
        M = max([1] + [len(q) for pl in paths for q in pl])
        if dqn_paths is not None:
            if dqn_paths[0].shape[1] < M:
                raise ValueError(f"set_tasks: dqn path buffer holds {dqn_paths[0].shape[1]} nodes, tasks need {M}")
            M = int(dqn_paths[0].shape[1])
        dev = self.state.device
        if T == 0:
            self.tasks, self.task_next = None, t.zeros(n, dtype=t.int32, device=dev)
            return
        goal = np.zeros((n, T, 3))
        xy = np.zeros((n, T, M, 2))
        pn = np.zeros((n, T), np.int32)
        stride = self.ref_stride
        prev = self.goal.cpu().numpy()
        for e in range(n):
            start = prev[e, :2]
            for k, (g, q) in enumerate(zip(goals[e], paths[e])):
                goal[e, k] = np.asarray(g, dtype=np.float64).reshape(3)
                a = np.asarray(q, dtype=np.float64).reshape(-1, 2)
                xy[e, k, :len(a)] = a
                pn[e, k] = len(a)
                stride = max(stride, self.ref_rows_bound(start, a))
                start = goal[e, k, :2]
        if stride > self.ref_stride:
            ref = t.zeros(n, stride, 3, dtype=t.float64, device=dev)
            ref[:, :self.ref_stride] = self.ref_traj
            self.ref_traj, self.ref_stride = ref, stride
        self.task_count = t.tensor([len(g) for g in goals], dtype=t.int32, device=dev)
        self.task_next = t.zeros(n, dtype=t.int32, device=dev)
        self.task_goal = t.tensor(goal, dtype=t.float64, device=dev)
        self.task_path = t.tensor(xy, dtype=t.float64, device=dev)
        self.task_path_n = t.tensor(pn, dtype=t.int32, device=dev)
        tk = _lib.TtmpcFleetTasks()
        tk.max_tasks, tk.max_nodes = T, M
        tk.count, tk.next = self.task_count.data_ptr(), self.task_next.data_ptr()
        tk.goal, tk.path_xy, tk.path_n = self.task_goal.data_ptr(), self.task_path.data_ptr(), self.task_path_n.data_ptr()
        if dqn_paths is not None:
            tk.path_out, tk.path_out_n = dqn_paths[0].data_ptr(), dqn_paths[1].data_ptr()
        self.dqn_paths = dqn_paths
        self.tasks = tk if int(self.task_count.sum()) > 0 else None

    # ------------------------------------------------------------------ DQN
    def enable_dqn(self, weights, geometry, paths, layout=None, moving_shape="rect",
                   moving_radius: float = DYN_OBS_SIZE, ref_speed: float = 1.0, corner_samples: int = 3,
                   sample_offset: float = 0.0):
        """Run the DQN side of the hybrid loop (main.py:174-193) at the start of every ``step()``, on
        the step's stream: ``agent5`` <- (state, last_u); the internal observation
        (``dqn.internal_obs_device``); lidar observation + Q-network + argmax
        (``DqnCompanion.observe_act_device``, with ``use_memory`` on the layout's memory rows); the
        rl_ref rollout of the chosen action into ``self.hint``.  The fleet step follows as before.

        weights: ``dqn.QNetWeights``.  geometry: the CUDA tensors of ``dqn.pack_geometry``
        (xy [n][max_vert][2] float64, off [n][max_poly+1], solid [n][max_poly], count [n] int32);
        layout defaults to ``dqn.default_layout`` with those max_poly / max_vert.  paths: the CUDA
        tensors of ``dqn.pack_paths`` (path_xy [n][m][2] float64, path_n [n] int32); task queues keep
        them current (``set_tasks``).

        moving_shape: how the lidar sees the moving obstacles of ``set_moving_obstacles``, as solid
        rings at the positions this step's pack treats as current (``dyn_cur``): ``"rect"`` the
        ``circle_to_rect`` square of moving_radius the HintSwitcher uses, a ``[k][nv][2]`` array of
        vertex offsets (one template per moving obstacle, 3 <= nv <= 32), or None (not seen: the
        static geometry alone).

        Results, overwritten by every step: ``dqn_action`` [n] int32, ``dqn_q`` [n][n_out],
        ``dqn_ext`` [n][n_ext] float32 and ``hint`` [n][N][2].  Whether a robot follows the hint is
        decided as without the DQN: ``use_hint`` (zeros unless set), or the switcher of
        ``enable_hint_switch``."""
        from types import SimpleNamespace

        from . import dqn
        t = self.torch
        n, dev = self.n, self.state.device

        def want(x, name, dtype, shape):
            if not isinstance(x, t.Tensor) or x.dtype != dtype or tuple(x.shape) != tuple(shape):
                got = (tuple(x.shape), x.dtype) if isinstance(x, t.Tensor) else type(x).__name__
                raise ValueError(f"enable_dqn: {name} must be a {dtype} tensor {tuple(shape)}, got {got}")

        if len(geometry) != 4 or len(paths) != 2:
            raise ValueError("enable_dqn: geometry = (xy, off, solid, count), paths = (path_xy, path_n)")
        xy, off, sol, cnt = geometry
        path_xy, path_n = paths
        if layout is None:
            if not (isinstance(xy, t.Tensor) and xy.dim() == 3 and isinstance(sol, t.Tensor) and sol.dim() == 2):
                raise ValueError("enable_dqn: geometry xy must be [n][max_vert][2] and solid [n][max_poly]")
            layout = dqn.default_layout(max_poly=sol.shape[1], max_vert=xy.shape[1])
        comp = dqn.DqnCompanion(layout, weights)       # rejects a bad layout before anything is set
        want(xy, "geometry xy", t.float64, (n, layout.max_vert, 2))
        want(off, "geometry off", t.int32, (n, layout.max_poly + 1))
        want(sol, "geometry solid", t.int32, (n, layout.max_poly))
        want(cnt, "geometry count", t.int32, (n,))
        if not (isinstance(path_xy, t.Tensor) and path_xy.dim() == 3 and path_xy.shape[1] >= 2):
            raise ValueError("enable_dqn: path_xy must be [n][m >= 2][2]")
        want(path_xy, "path_xy", t.float64, (n, path_xy.shape[1], 2))
        want(path_n, "path_n", t.int32, (n,))
        if 5 + 3 * int(corner_samples) != layout.n_internal or corner_samples < 0:
            raise ValueError(f"enable_dqn: 5 + 3 * corner_samples must equal the layout's n_internal {layout.n_internal}")
        ns = layout.num_segments
        n_ext = (4 if layout.use_memory else 2) * ns
        if weights.n_in != n_ext + layout.n_internal:
            raise ValueError(f"enable_dqn: Q-network input {weights.n_in} != {n_ext} + {layout.n_internal}")
        shape = None
        if isinstance(moving_shape, str):
            if moving_shape != "rect":
                raise ValueError(f"enable_dqn: moving_shape must be 'rect', a [k][nv][2] array or None, got {moving_shape!r}")
            if not (np.isfinite(moving_radius) and moving_radius >= 0.0):
                raise ValueError("enable_dqn: moving_radius must be finite and >= 0")
            shape = dqn.rect_shape(moving_radius)[None]
        elif moving_shape is not None:
            shape = np.asarray(moving_shape, dtype=np.float64)
            if shape.ndim != 3 or shape.shape[2] != 2 or not 3 <= shape.shape[1] <= 32:
                raise ValueError(f"enable_dqn: moving_shape must be [k][3..32][2], got {shape.shape}")
        if not all(x.is_cuda and x.is_contiguous() for x in (xy, off, sol, cnt, path_xy, path_n)):
            raise ValueError("enable_dqn: geometry and path tensors must be contiguous CUDA tensors")
        if self.tasks is not None and (self.dqn_paths is None or self.dqn_paths[0] is not path_xy):
            if self.tasks.max_nodes != path_xy.shape[1]:
                raise ValueError(f"enable_dqn: path_xy holds {path_xy.shape[1]} nodes, the queued tasks "
                                 f"{self.tasks.max_nodes}: call set_tasks after enable_dqn")
            self.tasks.path_out, self.tasks.path_out_n = path_xy.data_ptr(), path_n.data_ptr()
            self.dqn_paths = (path_xy, path_n)
        f32 = dict(dtype=t.float32, device=dev)
        w = [t.from_numpy(a).to(dev) for a in weights.arrays]
        d = SimpleNamespace(
            lay=layout, geometry=(xy, off, sol, cnt), paths=(path_xy, path_n), shape=shape, shape_dev=None,
            ref_speed=float(ref_speed), corner_samples=int(corner_samples), sample_offset=float(sample_offset),
            comp=comp, w=w,
            qnet=_lib.TtdqnQnet(weights.n_in, weights.n_h1, weights.n_h2, weights.n_out, *[a.data_ptr() for a in w]),
            agent5=t.zeros(n, 5, dtype=t.float64, device=dev), internal=t.zeros(n, layout.n_internal, **f32),
            progress=t.zeros(n, dtype=t.float64, device=dev),
            old_ext=t.zeros(n, 2 * ns, **f32) if layout.use_memory else None)
        self.dqn_ext = t.zeros(n, n_ext, **f32)
        self.dqn_q = t.zeros(n, weights.n_out, **f32)
        self.dqn_action = t.zeros(n, dtype=t.int32, device=dev)
        self.hint = t.zeros(n, self.N, 2, dtype=t.float64, device=dev)
        if self.use_hint is None:
            self.use_hint = t.zeros(n, dtype=t.int32, device=dev)
        self._dqn = d

    def _moving_shapes(self):
        """(shape_xy [1][k][nv][2], shape_nv [1][k]) device tensors of the lidar's moving rings for the
        current k = n_dyn_live, or None when the lidar does not see moving obstacles."""
        d = self._dqn
        if d.shape is None or self.dyn_cur is None or self.n_dyn_live == 0:
            return None
        k = self.n_dyn_live
        if d.shape_dev is None or d.shape_dev[0].shape[1] != k:
            xy = d.shape
            if len(xy) == 1:
                xy = np.repeat(xy, k, axis=0)
            if len(xy) != k:
                raise ValueError(f"enable_dqn: {len(xy)} moving shapes for {k} moving obstacles")
            dev = self.state.device
            d.shape_dev = (self.torch.tensor(xy[None], device=dev),
                           self.torch.full((1, k), xy.shape[1], dtype=self.torch.int32, device=dev))
        return d.shape_dev

    def _dqn_step(self, st, stream):
        import contextlib

        from . import dqn
        d, t = self._dqn, self.torch
        xy, off, sol, cnt = d.geometry
        with contextlib.nullcontext() if stream is None else t.cuda.stream(t.cuda.ExternalStream(stream)):
            d.agent5[:, :3] = self.state                                 # env.set_agent_state (main.py:175-176)
            d.agent5[:, 3:] = self.last_u
        dqn.internal_obs_device(d.agent5, *d.paths, corner_samples=d.corner_samples, sample_offset=d.sample_offset,
                                max_distance=d.lay.max_distance, out=d.internal, progress=d.progress, stream=st)
        shapes = self._moving_shapes()
        d.comp.observe_act_device(self.state, xy, off, sol, cnt, d.internal, d.old_ext,
                                  dict(ext=self.dqn_ext, q=self.dqn_q, action=self.dqn_action), d.qnet, stream=st,
                                  moving=None if shapes is None else (self.dyn_cur, *shapes))
        dqn.rl_ref_device(d.agent5, self.dqn_action, steps=self.N, ts=self.config.ts, ref_speed=d.ref_speed,
                          out=self.hint, stream=st)

    # ------------------------------------------------------------------ the step
    def _fleet_struct(self) -> _lib.TtmpcFleet:
        f = _lib.TtmpcFleet()
        f.n, f.ref_stride = self.n, self.ref_stride
        f.state, f.goal, f.last_u = self.state.data_ptr(), self.goal.data_ptr(), self.last_u.data_ptr()
        f.idx_ref, f.status = self.idx_ref.data_ptr(), self.status.data_ptr()
        f.ref_traj, f.ref_len = self.ref_traj.data_ptr(), self.ref_len.data_ptr()
        f.stc, f.stc_shared = self.stc.data_ptr(), self.stc_shared
        f.n_dyn_live, f.action_steps = self.n_dyn_live, self.action_steps
        f.other = self.other.data_ptr() if self.other is not None else None
        f.dyn = None
        if self.dyn_cur is not None:
            f.dyn_cur, f.dyn_last, f.dyn_disp = self.dyn_cur.data_ptr(), self.dyn_last.data_ptr(), self.dyn_disp.data_ptr()
        f.dyn_size = DYN_OBS_SIZE
        for i, v in enumerate(self.tuning):
            f.tuning[i] = float(v)
        f.base_speed, f.low_speed = float(self.base_speed), float(self.config.low_speed)
        f.stc_weight, f.dyn_weight = self.stc_weight, self.dyn_weight
        if self.hint is not None and self.use_hint is not None:
            f.hint, f.use_hint = self.hint.data_ptr(), self.use_hint.data_ptr()
        if getattr(self, "sw_state", None) is not None:
            f.sw_state = self.sw_state.data_ptr()
            f.sw_poly_xy, f.sw_poly_nv = self.sw_poly_xy.data_ptr(), self.sw_poly_nv.data_ptr()
            f.sw_max_poly, f.sw_max_pv, f.sw_poly_shared = self.sw_shape
            f.sw_switch_distance, f.sw_detach_distance, f.sw_detach_steps = self.sw_params
            f.sw_dyn_radius = DYN_OBS_SIZE
        return f

    def _result_struct(self) -> _lib.TtmpcResult:
        r = _lib.TtmpcResult()
        r.u, r.cost, r.exit_status = self.u.data_ptr(), self.cost.data_ptr(), self.exit_status.data_ptr()
        r.inner_iters, r.y, r.pred_states = self.inner.data_ptr(), self.y.data_ptr(), self.pred_states.data_ptr()
        return r

    def step(self, keep_multipliers: bool = True, warm_start: bool = False, skip_stopped: bool = False,
             stream=None, monitor: bool = True):
        """One control step of every robot, asynchronous on the current torch stream.

        keep_multipliers=True (default) is what the reference's control loop does: the PyO3 ``Solver``
        object of a robot owns its AlmCache, so the Lagrange multipliers one ``run()`` ends with are
        the ones the next ``run()`` starts from (``self.y`` lives on the device between steps and is
        passed in / out of the solve).  False starts every step from y = 0 (a fresh solver object).

        warm_start=True starts the solve of every running robot from its previous solution shifted
        by one step (the last control repeated) when that solve converged, and from zeros otherwise
        (``TTMPC_FLEET_WARM_START``; ``run_step(..., initial_guess)`` in the reference).  ``self.u``
        and ``self.exit_status`` start as zeros, so a warm first step equals a cold one.
        skip_stopped=True solves only the robots that are still RUNNING; the result rows of the
        others keep what their last solve wrote (``TTMPC_FLEET_SKIP_STOPPED``).  Both default to off.

        With ``action_steps = k > 1`` the step does what ``InterfaceMpc`` does with
        ``config.action_steps = k`` (include/ttmpc.h, ``action_steps``): the state takes one RK4
        step with u[k-1] from the state the step started in (``run_solver`` computes each taken
        state from there) and ``last_u`` becomes u[k-1]; the goal test of the next step reads u[0]
        of this solution.  A warm start shifts by k.  Moving obstacles still move once per step.

        With tasks queued (``set_tasks``) a robot that reaches its goal takes its next task in the
        same step and is packed and solved on it; with warm_start it then starts from zeros.

        ``pred_states`` is the rollout of u* from the state the step STARTED in (p.s), i.e. one step
        earlier than ``TrajectoryGenerator.run_step``'s list, which re-applies u from the post-step
        state (trajectory_generator.py:296-301; ``planner.TrajectoryGenerator`` reproduces that list
        on the host).

        With the monitor enabled (``enable_monitor``) the step ends with it, on the same stream;
        monitor=False leaves it to a ``run_monitor()`` call before the next step (a benchmark that
        times the step alone does that).

        With the DQN enabled (``enable_dqn``) the step starts with the DQN side of the hybrid loop,
        which writes ``hint``, on the same stream.  With a map (``set_world``) the map selection
        runs before both."""
        st = stream if stream is not None else self.torch.cuda.current_stream().cuda_stream
        if self.world is not None:
            self.run_world_select(st)
        if self._dqn is not None:
            self._dqn_step(st, stream)
        f, r = self._fleet_struct(), self._result_struct()
        f.options = (_lib.FLEET_WARM_START if warm_start else 0) | (_lib.FLEET_SKIP_STOPPED if skip_stopped else 0)
        if self.tasks is not None:
            _lib.check(self.lib.ttmpc_fleet_step_tasks_device(C.byref(self.cfg), C.byref(f), C.byref(self.tasks),
                                                              self.p.data_ptr(), 1 if keep_multipliers else 0,
                                                              C.byref(r), st), "ttmpc_fleet_step_tasks_device")
        else:
            _lib.check(self.lib.ttmpc_fleet_step_device(C.byref(self.cfg), C.byref(f), self.p.data_ptr(),
                                                        1 if keep_multipliers else 0, C.byref(r), st),
                       "ttmpc_fleet_step_device")
        self.steps += 1
        if self.monitor is not None and monitor:
            self.run_monitor(st)

    def pack(self, stream=None):
        """The pack kernel alone (action_steps = 1 only: raises TtmpcError otherwise)."""
        st = stream if stream is not None else self.torch.cuda.current_stream().cuda_stream
        f = self._fleet_struct()
        _lib.check(self.lib.ttmpc_fleet_pack_device(C.byref(self.cfg), C.byref(f), self.p.data_ptr(), st), "fleet pack")

    def advance(self, stream=None):
        """The advance kernel alone (action_steps = 1 only: raises TtmpcError otherwise)."""
        st = stream if stream is not None else self.torch.cuda.current_stream().cuda_stream
        f = self._fleet_struct()
        _lib.check(self.lib.ttmpc_fleet_advance_device(C.byref(self.cfg), C.byref(f), self.u.data_ptr(),
                                                       self.exit_status.data_ptr(), st), "fleet advance")
