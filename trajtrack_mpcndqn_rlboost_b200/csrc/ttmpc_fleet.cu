// ttmpc_fleet.cu -- the caller side of the solve, batched on the device: one control step of
// n independent robots as the reference's InterfaceMpc.get_action / TrajectoryGenerator.run_step
// perform it (src/interface_mpc.py:72-92, src/mpc_traj_tracker/trajectory_generator.py:203-294).
// See include/ttmpc.h ("Fleet step") for the contract; oracle/ttfleet_oracle.c is the CPU
// restatement these kernels match bit for bit (use_libm = 0).
//
// The kernels are copy / scalar work: pack writes the n x np parameter block once, coalesced
// (HBM-bound, 21 KB per robot), advance touches 5 doubles per robot, the monitor (run after the
// step, include/ttmpc.h: ttmpc_fleet_monitor) reads a robot's polygons, obstacles and reference rows,
// the map selection (run before the step, ttmpc_fleet_world) the map polygons near a robot.
#include <cuda_runtime.h>

#include "ttmpc_device.cuh"
#include "ttmpc_launch.cuh"

namespace ttmpc {

__device__ __forceinline__ double hyp2(double dx, double dy) { return sqrt(fma(dx, dx, dy * dy)); }

// shapely Polygon.contains(Point) (strictly inside, even-odd rule) / Polygon.distance(Point)
__device__ __forceinline__ bool poly_contains(const double *xy, int nv, double px, double py) {
  bool in = false;
  for (int i = 0, j = nv - 1; i < nv; j = i++) {
    const double xi = xy[2 * i], yi = xy[2 * i + 1], xj = xy[2 * j], yj = xy[2 * j + 1];
    if (((yi > py) != (yj > py)) && (px < (xj - xi) * (py - yi) / (yj - yi) + xi)) in = !in;
  }
  return in;
}
// distance of (px, py) to the segment from (ax, ay) to (bx, by)
__device__ __forceinline__ double seg_distance(double ax, double ay, double bx, double by, double px, double py) {
  const double dx = bx - ax, dy = by - ay;
  const double len2 = dx * dx + dy * dy;
  double t = 0.0;
  if (len2 > 0.0) { t = ((px - ax) * dx + (py - ay) * dy) / len2; t = t < 0.0 ? 0.0 : (t > 1.0 ? 1.0 : t); }
  const double qx = ax + t * dx - px, qy = ay + t * dy - py;
  return sqrt(qx * qx + qy * qy);
}
__device__ __forceinline__ double poly_distance(const double *xy, int nv, double px, double py) {
  if (poly_contains(xy, nv, px, py)) return 0.0;
  double best = INFINITY;
  for (int i = 0, j = nv - 1; i < nv; j = i++) {
    const double d = seg_distance(xy[2 * j], xy[2 * j + 1], xy[2 * i], xy[2 * i + 1], px, py);
    if (d < best) best = d;
  }
  return best;
}
constexpr int SW_MAX_OBS = 64;  // obstacles per robot the parallel switch path handles (more: serial path)
// obstacle o of robot e in the list "static polygons + circle_to_rect(moving obstacle)"; rect: 8 doubles scratch
__device__ __forceinline__ const double *sw_obstacle(const ttmpc_fleet &f, int e, int o, int n_stc, double *rect, int *nv) {
  if (o < n_stc) {
    const double *pxy = f.sw_poly_xy + (f.sw_poly_shared ? 0 : (size_t)e * f.sw_max_poly * f.sw_max_pv * 2);
    const int *pnv = f.sw_poly_nv + (f.sw_poly_shared ? 0 : (size_t)e * f.sw_max_poly);
    *nv = pnv[o];
    return pxy + (size_t)o * f.sw_max_pv * 2;
  }
  const double *c = f.dyn_cur + ((size_t)e * f.n_dyn_live + (o - n_stc)) * 2, rr = f.sw_dyn_radius;  // main.py:91-95
  rect[0] = c[0] - rr; rect[1] = c[1] - rr; rect[2] = c[0] + rr; rect[3] = c[1] - rr;
  rect[4] = c[0] + rr; rect[5] = c[1] + rr; rect[6] = c[0] - rr; rect[7] = c[1] + rr;
  *nv = 4;
  return rect;
}
// the state machine of HintSwitcher.switch on precomputed predicates: dist[o] (distance of the
// robot to obstacle o, < 0: unused slot) and in[k * n_obs + o] (reference point k inside obstacle o)
__device__ int hint_switch_sm(const ttmpc_fleet &f, int e, int N, int n_obs, const double *dist,
                              const unsigned char *in) {
  int *st = f.sw_state + 2 * e;
  bool cnt_flag = false;
  for (int k = 0; k < N; k++)
    for (int o = 0; o < n_obs; o++) {
      if (dist[o] < 0.0) continue;
      if (in[k * n_obs + o]) {
        if (dist[o] < f.sw_switch_distance && !st[0]) { st[0] = 1; return 1; }
      } else if (dist[o] > f.sw_detach_distance && st[0]) {
        if (st[1] > f.sw_detach_steps) { st[0] = 0; st[1] = 0; }
        else if (!cnt_flag) { st[1] += 1; cnt_flag = true; }
      }
    }
  return st[0];
}
// HintSwitcher.switch (main_pre.py:35-52) of robot e, on the ORIGINAL local reference (serial form)
__device__ int hint_switch(const ttmpc_fleet &f, int e, int N, const double *ref, int L, int idx) {
  int *st = f.sw_state + 2 * e;  // switch_on, detach_cnt
  const double px = f.state[3 * e], py = f.state[3 * e + 1];
  const int n_stc = f.sw_poly_xy ? f.sw_max_poly : 0, n_dyn = f.dyn_cur ? f.n_dyn_live : 0;
  const double *pxy = f.sw_poly_xy ? f.sw_poly_xy + (f.sw_poly_shared ? 0 : (size_t)e * f.sw_max_poly * f.sw_max_pv * 2) : nullptr;
  const int *pnv = f.sw_poly_nv ? f.sw_poly_nv + (f.sw_poly_shared ? 0 : (size_t)e * f.sw_max_poly) : nullptr;
  bool cnt_flag = false;
  for (int k = 0; k < N; k++) {
    int r = idx + k; if (r > L - 1) r = L - 1;
    const double ox = ref[3 * r], oy = ref[3 * r + 1];
    for (int o = 0; o < n_stc + n_dyn; o++) {
      double rect[8];
      const double *xy; int nv;
      if (o < n_stc) { nv = pnv[o]; xy = pxy + (size_t)o * f.sw_max_pv * 2; if (nv < 3) continue; }
      else {  // circle_to_rect (main.py:91-95)
        const double *c = f.dyn_cur + ((size_t)e * f.n_dyn_live + (o - n_stc)) * 2, rr = f.sw_dyn_radius;
        rect[0] = c[0] - rr; rect[1] = c[1] - rr; rect[2] = c[0] + rr; rect[3] = c[1] - rr;
        rect[4] = c[0] + rr; rect[5] = c[1] + rr; rect[6] = c[0] - rr; rect[7] = c[1] + rr;
        xy = rect; nv = 4;
      }
      const double dist = poly_distance(xy, nv, px, py);
      if (poly_contains(xy, nv, ox, oy)) {
        if (dist < f.sw_switch_distance && !st[0]) { st[0] = 1; return 1; }
      } else if (dist > f.sw_detach_distance && st[0]) {
        if (st[1] > f.sw_detach_steps) { st[0] = 0; st[1] = 0; }
        else if (!cnt_flag) { st[1] += 1; cnt_flag = true; }
      }
    }
  }
  return st[0];
}

// get_global_ref_traj (trajectory_generator.py:160-201) of a queued task from (px, py): rows
// (x, y, heading) into out (nullptr: count only).  Returns the row count, or -1 for a task that
// cannot be driven: no node, a walk that would index past the last node (the reference raises),
// no row, or more than cap rows.  Python's operation order; oracle: ttfleet_oracle_global_ref_traj.
__device__ int global_ref_walk(const double *path, int n_nodes, double px, double py, double ts, double speed,
                               int cap, double *out) {
  if (n_nodes < 1) return -1;
  double tx = path[0], ty = path[1], ux = 0.0, uy = 0.0, gap = 0.0;
  int k = 0, rows = 0;
  bool alive = true;
  while (alive) {
    for (;;) {
      gap = hyp2(tx - px, ty - py);
      if (gap < 1e-9) {
        k += 1;
        if (k > n_nodes - 1) return -1;
        tx = path[2 * k]; ty = path[2 * k + 1];
        break;
      }
      ux = (tx - px) / gap; uy = (ty - py) / gap;
      const double eta = gap / speed;
      if (eta > ts) { px = px + ux * speed * ts; py = py + uy * speed * ts; break; }
      px = px + ux * speed * eta; py = py + uy * speed * eta;
      k += 1;
      if (k > n_nodes - 1) { alive = false; break; }
      tx = path[2 * k]; ty = path[2 * k + 1];
    }
    if (!(gap < 1e-9)) {
      if (rows >= cap) return -1;  // also bounds the walk
      if (out) { out[3 * rows] = px; out[3 * rows + 1] = py; out[3 * rows + 2] = tt_atan2(uy, ux); }
      rows++;
    }
  }
  return rows > 0 ? rows : -1;
}

// get_local_ref_traj (trajectory_generator.py:214-219): first minimum in the window [idx-k, idx+5k)
__device__ __forceinline__ int local_ref_idx(const double *ref, int L, int idx, int k, double x, double y) {
  int lo = idx - 1 * k; if (lo < 0) lo = 0;
  int hi = idx + 5 * k; if (hi > L) hi = L;
  double best = INFINITY; int arg = lo;
  for (int i = lo; i < hi; i++) {
    const double dist = hyp2(x - ref[3 * i], y - ref[3 * i + 1]);
    if (dist < best) { best = dist; arg = i; }
  }
  return arg;
}

// One CTA per robot.  Thread 0 does the scalar decisions (closest reference point, goal test,
// speed reference); all threads then write the packed vector, element o of the row by thread
// o mod blockDim (coalesced 8-byte stores).  prev_u holds the previous step's solutions.  With
// action_steps = k > 1 the goal test reads their first control (InterfaceMpc._last_action =
// actions[0]) while p packs last_u = u[k-1] (past_actions[-1]); with k = 1 both are last_u.  With
// warm_exit (warm start of the fleet step) the CTA of a robot that is RUNNING after the goal test
// also rewrites its row of prev_u, the initial guess of this step's solve: the previous solution
// shifted by k steps (last control repeated) if that solve converged, zeros otherwise.
// tk.count != nullptr (ttmpc_fleet_step_tasks_device): after the goal test thread 0 lets a REACHED
// robot take its next queued task (include/ttmpc.h, ttmpc_fleet_tasks): it samples the task's
// reference trajectory into the robot's ref_traj rows, sets goal, ref_len, idx_ref, last_u and
// status, and repeats the search and the goal test on the new task.  The other threads read the
// new rows and last_u from global memory and the new ref_len from s_len, all behind the barrier.
__global__ void __launch_bounds__(128) fleet_pack_kernel(const ttmpc_fleet f, const FleetDims d,
                                                         double *__restrict__ p_all, double *prev_u,
                                                         const int *__restrict__ warm_exit,
                                                         const ttmpc_fleet_tasks tk) {
  const int e = blockIdx.x;
  if (e >= f.n) return;
  __shared__ int s_idx, s_hint, s_sw, s_run, s_len, s_new;
  __shared__ double s_speed;
  __shared__ double s_dist[SW_MAX_OBS];
  __shared__ unsigned char s_in[32 * SW_MAX_OBS];
  const double *st = f.state + 3 * e, *goal = f.goal + 3 * e, *lu = f.last_u + 2 * e;
  const double *ref = f.ref_traj + (size_t)e * f.ref_stride * 3;
  const int N = d.N;
  if (threadIdx.x == 0) {
    int idx = f.idx_ref[e], L = f.ref_len[e];
    const double x = st[0], y = st[1];
    const bool was_running = f.status[e] == TTMPC_FLEET_RUNNING;
    // check_termination_condition (:158-164): np.allclose(atol=0.05, rtol=0) and |v| < 0.05.
    // Runs before the warm-start rewrite of the same prev_u row (behind a __syncthreads).
    if (f.status[e] == TTMPC_FLEET_RUNNING) {
      idx = local_ref_idx(ref, L, idx, f.action_steps, x, y);
      f.idx_ref[e] = idx;
      const bool close = fabs(x - goal[0]) <= 0.05 && fabs(y - goal[1]) <= 0.05;
      const double v0 = f.action_steps > 1 ? prev_u[(size_t)e * 2 * N] : lu[0];
      if (close && fabs(v0) < 0.05) f.status[e] = TTMPC_FLEET_REACHED;
    }
    bool took = false;
    if (tk.count) {
      int next = tk.next[e];
      const int count = min(tk.count[e], tk.max_tasks);
      while (f.status[e] == TTMPC_FLEET_REACHED && next < count) {  // InterfaceMpc.initialization
        const size_t t = (size_t)e * tk.max_tasks + next;
        const double *path = tk.path_xy + t * tk.max_nodes * 2;
        const int pn = tk.path_n[t];
        next += 1;
        const int rows = pn <= tk.max_nodes ? global_ref_walk(path, pn, x, y, d.ts, f.base_speed, f.ref_stride, nullptr) : -1;
        if (rows < 0) { f.status[e] = TTMPC_FLEET_BAD_TASK; break; }
        global_ref_walk(path, pn, x, y, d.ts, f.base_speed, f.ref_stride, const_cast<double *>(ref));
        L = rows;
        const_cast<int *>(f.ref_len)[e] = rows;
        double *g = const_cast<double *>(goal);
        g[0] = tk.goal[3 * t]; g[1] = tk.goal[3 * t + 1]; g[2] = tk.goal[3 * t + 2];
        f.last_u[2 * e] = 0.0; f.last_u[2 * e + 1] = 0.0;
        if (tk.path_out) {
          for (int i = 0; i < 2 * pn; i++) tk.path_out[(size_t)e * tk.max_nodes * 2 + i] = path[i];
          tk.path_out_n[e] = pn;
        }
        f.status[e] = TTMPC_FLEET_RUNNING;
        took = true;
        idx = local_ref_idx(ref, L, 0, f.action_steps, x, y);
        f.idx_ref[e] = idx;
        // _last_action is kept: with k > 1 the first control of the previous solution, with k = 1
        // the last applied control, which passed |v| < 0.05 when the robot stopped
        const bool close = fabs(x - g[0]) <= 0.05 && fabs(y - g[1]) <= 0.05;
        const double v0 = f.action_steps > 1 ? prev_u[(size_t)e * 2 * N] : 0.0;
        if (close && fabs(v0) < 0.05) f.status[e] = TTMPC_FLEET_REACHED;
      }
      tk.next[e] = next;
    }
    s_run = f.status[e] == TTMPC_FLEET_RUNNING;
    s_idx = idx;
    s_len = L;
    s_new = took;
    s_sw = (f.sw_state && f.hint && f.use_hint && (took ? s_run : was_running)) ? 1 : 0;
    // speed reference (:248-255)
    const double dist = hyp2(x - goal[0], y - goal[1]);
    double v = f.base_speed;
    if (!(dist >= f.base_speed * N * d.ts)) {
      v = dist / N / d.ts;
      if (!(v > f.low_speed)) v = f.low_speed;
    }
    s_speed = v;
  }
  __syncthreads();
  const int idx = s_idx, L = s_len;
  // hybrid mode: main.py:200 evaluates HintSwitcher.switch before get_action's goal test.  The
  // geometric predicates are independent: one obstacle distance / one (point, obstacle)
  // containment per thread, then thread 0 walks the state machine over them.
  if (s_sw) {
    const int n_stc = f.sw_poly_xy ? f.sw_max_poly : 0, n_obs = n_stc + (f.dyn_cur ? f.n_dyn_live : 0);
    if (n_obs <= SW_MAX_OBS) {
      double rect[8]; int nv;
      for (int o = threadIdx.x; o < n_obs; o += blockDim.x) {
        const double *xy = sw_obstacle(f, e, o, n_stc, rect, &nv);
        s_dist[o] = nv < 3 ? -1.0 : poly_distance(xy, nv, st[0], st[1]);
      }
      for (int q = threadIdx.x; q < N * n_obs; q += blockDim.x) {
        const int k = q / n_obs, o = q - k * n_obs;
        const double *xy = sw_obstacle(f, e, o, n_stc, rect, &nv);
        int r = idx + k; if (r > L - 1) r = L - 1;
        s_in[q] = (nv >= 3 && poly_contains(xy, nv, ref[3 * r], ref[3 * r + 1])) ? 1 : 0;
      }
      __syncthreads();
      if (threadIdx.x == 0) f.use_hint[e] = hint_switch_sm(f, e, N, n_obs, s_dist, s_in);
    } else if (threadIdx.x == 0) {
      f.use_hint[e] = hint_switch(f, e, N, ref, L, idx);
    }
  }
  if (threadIdx.x == 0) s_hint = (f.hint && f.use_hint && f.use_hint[e]) ? 1 : 0;
  __syncthreads();
  if (warm_exit && s_run) {  // in place: every element is read before any is written
    double *u = prev_u + (size_t)e * 2 * N;
    const int o = threadIdx.x, nz = 2 * N;  // nz <= 64 < blockDim
    double v = 0.0;
    if (o < nz && warm_exit[e] == TTMPC_CONVERGED && !s_new) {  // u'[j] = u[min(j + k, N - 1)]
      const int src = o + 2 * f.action_steps, last = nz - 2 + (o & 1);
      v = u[src < last ? src : last];
    }
    __syncthreads();
    if (o < nz) u[o] = v;
  }
  double *p = p_all + (size_t)e * d.np;
  const int o_refs = 18, o_speed = o_refs + 3 * N, o_other = o_speed + N, o_stc = o_other + d.n_other,
            o_dyn = o_stc + d.n_stc, o_ws = o_dyn + d.n_dyn, o_wd = o_ws + N;
  const double *stc = f.stc + (f.stc_shared ? 0 : (size_t)e * d.n_stc);
  const bool hinted = s_hint != 0;  // hybrid mode: DQN hint positions
  const double *hint = f.hint + (size_t)e * N * 2;
  for (int o = threadIdx.x; o < d.np; o += blockDim.x) {
    double v;
    if (o < 3) v = st[o];
    else if (o < 6) {
      int r = idx + N - 1; if (r > L - 1) r = L - 1;
      v = (hinted && o < 5) ? hint[2 * (N - 1) + (o - 3)] : ref[3 * r + (o - 3)];
    }
    else if (o < 8) v = lu[o - 6];
    else if (o < o_refs) v = f.tuning[o - 8];
    else if (o < o_speed) {
      const int k = (o - o_refs) / 3, c = (o - o_refs) - 3 * k;
      int r = idx + k; if (r > L - 1) r = L - 1;
      v = (hinted && c < 2) ? hint[2 * k + c] : ref[3 * r + c];
    }
    else if (o < o_other) v = s_speed;
    else if (o < o_stc) v = f.other ? f.other[(size_t)e * d.n_other + (o - o_other)] : 0.0;
    else if (o < o_dyn) v = stc[o - o_stc];
    else if (o < o_ws) {
      const int q = o - o_dyn;
      if (f.dyn) v = f.dyn[(size_t)e * d.n_dyn + q];
      else {
        v = 0.0;
        const int j = q / (6 * N);
        if (f.dyn_cur && j < f.n_dyn_live) {  // est_dyn_obs_positions (main.py:80-89)
          const int i = (q - j * 6 * N) / 6, c = q - j * 6 * N - 6 * i;
          const double *cur = f.dyn_cur + ((size_t)e * f.n_dyn_live + j) * 2;
          const double *last = f.dyn_last + ((size_t)e * f.n_dyn_live + j) * 2;
          if (c < 2) v = cur[c] + (cur[c] - last[c]) * (double)(i + 1);
          else if (c < 4) v = f.dyn_size;
          else v = c == 4 ? 0.0 : 1.0;
        }
      }
    }
    else if (o < o_wd) v = f.stc_weight;
    else v = f.dyn_weight;
    p[o] = v;
  }
}

// One thread per robot: obstacles move (once per control step), RUNNING robots take their step.
// With action_steps = k, run_solver (trajectory_generator.py:291-294) computes each of its k taken
// states from the state the step started in, with u[i], and continues from the last one: the new
// state is one RK4 step with u[k-1], which is also the new last action (past_actions[-1]).
__global__ void __launch_bounds__(128) fleet_advance_kernel(const ttmpc_fleet f, const FleetDims d,
                                                            const double *__restrict__ u_all,
                                                            const int *__restrict__ exit_status) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= f.n) return;
  if (f.dyn_cur) {
    for (int j = 0; j < f.n_dyn_live; j++) {
      double *c = f.dyn_cur + ((size_t)e * f.n_dyn_live + j) * 2;
      double *l = f.dyn_last + ((size_t)e * f.n_dyn_live + j) * 2;
      const double *dd = f.dyn_disp + ((size_t)e * f.n_dyn_live + j) * 2;
      l[0] = c[0]; l[1] = c[1];
      c[0] = c[0] + dd[0]; c[1] = c[1] + dd[1];
    }
  }
  if (f.status[e] != TTMPC_FLEET_RUNNING) return;
  if (exit_status && exit_status[e] == TTMPC_NOT_FINITE) { f.status[e] = TTMPC_FLEET_FAILED; return; }
  const double *u = u_all + (size_t)e * 2 * d.N;
  double *st = f.state + 3 * e;
  const int j = 2 * (f.action_steps - 1);
  const double v = u[j], w = u[j + 1], ts = d.ts;
  // unicycle_model, RK4 branch, in numpy's operation order (motion_model.py:166-174)
  double s, c;
  tt_sincos(st[2], &s, &c);
  const double k1x = ts * (v * c), k1y = ts * (v * s), k1t = ts * w;
  tt_sincos(st[2] + 0.5 * k1t, &s, &c);
  const double k2x = ts * (v * c), k2y = ts * (v * s), k2t = ts * w;
  tt_sincos(st[2] + 0.5 * k2t, &s, &c);
  const double k3x = ts * (v * c), k3y = ts * (v * s), k3t = ts * w;
  tt_sincos(st[2] + k3t, &s, &c);
  const double k4x = ts * (v * c), k4y = ts * (v * s), k4t = ts * w;
  const double sixth = 1.0 / 6.0;
  st[0] = st[0] + sixth * (((k1x + 2.0 * k2x) + 2.0 * k3x) + k4x);
  st[1] = st[1] + sixth * (((k1y + 2.0 * k2y) + 2.0 * k3y) + k4y);
  st[2] = st[2] + sixth * (((k1t + 2.0 * k2t) + 2.0 * k3t) + k4t);
  f.last_u[2 * e] = v; f.last_u[2 * e + 1] = w;
}

// Distance of the chord (x0, y0) -> (x1, y1) to a polygon ring: 0 if an endpoint is inside or the
// chord properly crosses an edge, else the least endpoint-to-edge and vertex-to-chord distance (the
// distance of two segments that do not cross).  A chord that touches an edge without crossing it
// gets its distance from the touching endpoint or vertex.  Zero length: poly_distance.
__device__ double swept_poly_distance(const double *xy, int nv, double x0, double y0, double x1, double y1) {
  if (poly_contains(xy, nv, x0, y0) || poly_contains(xy, nv, x1, y1)) return 0.0;
  const bool moved = x0 != x1 || y0 != y1;
  const double cx = x1 - x0, cy = y1 - y0;
  double best = INFINITY;
  for (int i = 0, j = nv - 1; i < nv; j = i++) {
    const double ax = xy[2 * j], ay = xy[2 * j + 1], bx = xy[2 * i], by = xy[2 * i + 1];
    double d = seg_distance(ax, ay, bx, by, x0, y0);
    if (moved) {
      const double ex = bx - ax, ey = by - ay;  // orientations of the chord ends to the edge, and back
      const double o0 = ex * (y0 - ay) - ey * (x0 - ax), o1 = ex * (y1 - ay) - ey * (x1 - ax);
      const double oa = cx * (ay - y0) - cy * (ax - x0), ob = cx * (by - y0) - cy * (bx - x0);
      if (((o0 > 0.0 && o1 < 0.0) || (o0 < 0.0 && o1 > 0.0)) && ((oa > 0.0 && ob < 0.0) || (oa < 0.0 && ob > 0.0)))
        return 0.0;
      const double d1 = seg_distance(ax, ay, bx, by, x1, y1), dv = seg_distance(x0, y0, x1, y1, ax, ay);
      if (d1 < d) d = d1;
      if (dv < d) d = dv;
    }
    if (d < best) best = d;
  }
  return best;
}

// One thread per robot: the obstacle-contact and tracking monitor of the step that just ran
// (include/ttmpc.h, ttmpc_fleet_monitor).  oracle/ttfleet_monitor_oracle.c restates it.
__global__ void __launch_bounds__(128) fleet_monitor_kernel(const ttmpc_fleet f, const ttmpc_fleet_monitor m) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= f.n) return;
  double *pv = m.prev_xy + 2 * e;
  const double x0 = pv[0], y0 = pv[1], x1 = f.state[3 * e], y1 = f.state[3 * e + 1];
  double c = INFINITY;
  if (m.poly_xy) {
    const double *pxy = m.poly_xy + (m.poly_shared ? 0 : (size_t)e * m.max_poly * m.max_pv * 2);
    const int *pnv = m.poly_nv + (m.poly_shared ? 0 : (size_t)e * m.max_poly);
    for (int o = 0; o < m.max_poly; o++) {
      const int nv = min(pnv[o], m.max_pv);
      if (nv < 3) continue;
      const double d = swept_poly_distance(pxy + (size_t)o * m.max_pv * 2, nv, x0, y0, x1, y1) - m.robot_radius;
      if (d < c) c = d;
    }
  }
  if (f.dyn_cur) {  // robot relative to the obstacle: prev - last -> state - cur, linear in time
    const double r = m.moving_radius + m.robot_radius;
    for (int j = 0; j < f.n_dyn_live; j++) {
      const double *cur = f.dyn_cur + ((size_t)e * f.n_dyn_live + j) * 2;
      const double *last = f.dyn_last + ((size_t)e * f.n_dyn_live + j) * 2;
      const double d = seg_distance(x0 - last[0], y0 - last[1], x1 - cur[0], y1 - cur[1], 0.0, 0.0) - r;
      if (d < c) c = d;
    }
  }
  m.clearance[e] = c;
  if (c < m.min_clearance[e]) m.min_clearance[e] = c;
  const bool contact = c <= 0.0;
  if (contact) {
    m.contact_steps[e] += 1;
    if (m.first_contact[e] < 0) m.first_contact[e] = m.step;
  }
  if (f.status[e] == TTMPC_FLEET_RUNNING) {
    const int k = f.action_steps, L = f.ref_len[e], idx = f.idx_ref[e];
    const double *ref = f.ref_traj + (size_t)e * f.ref_stride * 3;
    int lo = idx - k; if (lo < 0) lo = 0;
    int hi = idx + 5 * k; if (hi > L) hi = L;
    double dev = seg_distance(ref[3 * lo], ref[3 * lo + 1], ref[3 * lo], ref[3 * lo + 1], x1, y1);
    if (hi - lo >= 2) {
      dev = INFINITY;
      for (int i = lo + 1; i < hi; i++) {
        const double d = seg_distance(ref[3 * i - 3], ref[3 * i - 2], ref[3 * i], ref[3 * i + 1], x1, y1);
        if (d < dev) dev = d;
      }
    }
    if (dev > m.deviation_max[e]) m.deviation_max[e] = dev;
    m.deviation_sum[e] = m.deviation_sum[e] + dev;
    m.moved_steps[e] += 1;
    if (m.stop_on_contact && contact) f.status[e] = TTMPC_FLEET_COLLIDED;
  }
  pv[0] = x1; pv[1] = y1;
}

cudaError_t launch_fleet_monitor(const ttmpc_fleet &f, const ttmpc_fleet_monitor &m, cudaStream_t st) {
  fleet_monitor_kernel<<<(f.n + 127) / 128, 128, 0, st>>>(f, m);
  return cudaGetLastError();
}

// ---- shared obstacle map: each robot's nearest map polygons into its static slots
constexpr int WS_WARPS = 4;     // robots (one warp each) per CTA of fleet_world_select_kernel
constexpr int WS_CAP = 128;     // candidates a warp buffers; >= K + 32 for every K <= 32 (Nstcobs)
constexpr int WS_MAX_K = 32;

// grid cell of coordinate v, clamped to 0..n-1 (NaN: 0)
__device__ __forceinline__ int world_cell(double v, double origin, double cell, int n) {
  const double a = floor((v - origin) / cell);
  return a >= 0.0 ? (a <= n - 1 ? (int)a : n - 1) : 0;
}
// cells x..y of one axis that the query c +- R visits, widened by one against rounding and
// clamped to the grid; x > y: none (also for a NaN or infinite coordinate)
__device__ __forceinline__ int2 world_axis(double c, double R, double origin, double cell, int n) {
  const double a = floor((c - R - origin) / cell) - 1.0, b = floor((c + R - origin) / cell) + 1.0;
  if (!(a <= b) || b < 0.0 || a > n - 1) return make_int2(0, -1);
  return make_int2(a < 0.0 ? 0 : (int)a, b > n - 1 ? n - 1 : (int)b);
}
// Keep the K smallest keys (d, o) of the warp's buffer [0, c): each lane ranks its entries against
// all c (keys are unique: one entry per polygon), the winners land at their rank.  Returns min(c, K).
__device__ __forceinline__ int world_keep_best(double *bd, int *bo, double *td, int *to, int c, int K, int lane) {
  if (lane < K) { td[lane] = INFINITY; to[lane] = -1; }
  __syncwarp();
  for (int i = lane; i < c; i += 32) {
    const double di = bd[i];
    const int oi = bo[i];
    int r = 0;
    for (int j = 0; j < c; j++) r += (bd[j] < di || (bd[j] == di && bo[j] < oi)) ? 1 : 0;
    if (r < K) { td[r] = di; to[r] = oi; }
  }
  __syncwarp();
  const int k = min(c, K);
  if (lane < k) { bd[lane] = td[lane]; bo[lane] = to[lane]; }
  __syncwarp();
  return k;
}

// One warp per robot (include/ttmpc.h, ttmpc_fleet_world).  The lanes walk the items of the visited
// cells one row of cells at a time (a row's items are contiguous in cell_items), each lane finds its
// item's cell, takes the polygon only in its lowest visited cell and computes its distance; eligible
// (d, o) go to the warp's shared buffer by ballot.  A full buffer is cut to its best K, so any
// candidate count stays exact.  At the end the best K are ordered by map index and the rows written
// with consecutive lanes on consecutive doubles.  oracle/ttfleet_world_oracle.c is the brute-force
// restatement over all M polygons.
__global__ void __launch_bounds__(32 * WS_WARPS) fleet_world_select_kernel(
    const double *__restrict__ state, int n, const ttmpc_fleet_world w, int K, int ns,
    double *__restrict__ stc_out, int *__restrict__ slot_poly, int *__restrict__ n_reach) {
  __shared__ double s_d[WS_WARPS][WS_CAP], s_td[WS_WARPS][WS_MAX_K];
  __shared__ int s_o[WS_WARPS][WS_CAP], s_to[WS_WARPS][WS_MAX_K];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * WS_WARPS + warp;
  if (e >= n) return;  // the whole warp
  double *bd = s_d[warp], *td = s_td[warp];
  int *bo = s_o[warp], *to = s_to[warp];
  const double x = state[3 * e], y = state[3 * e + 1], R = w.reach;
  int c = 0, total = 0;
  if (w.M > 0) {
    const int2 qx = world_axis(x, R, w.origin_x, w.cell, w.nx), qy = world_axis(y, R, w.origin_y, w.cell, w.ny);
    const int qx0 = qx.x, qx1 = qx.y, qy0 = qy.x, qy1 = qy.y;
    const int n_items = max(w.cell_start[w.nx * w.ny], 0);
    for (int cy = qy0; cy <= qy1; cy++) {
      const int *cs = w.cell_start + (size_t)cy * w.nx;
      const int lo = min(max(cs[qx0], 0), n_items), hi = min(max(cs[qx1 + 1], 0), n_items);
      int cx = qx0;
      for (int base = lo; base < hi; base += 32) {
        const int i = base + lane;
        double d = 0.0;
        int o = -1;
        bool take = false;
        if (i < hi) {
          while (cx < qx1 && i >= cs[cx + 1]) cx++;
          o = w.cell_items[i];
          if (o >= 0 && o < w.M) {
            const double *bb = w.bbox + 4 * (size_t)o;
            const int nv = min(w.poly_nv[o], w.max_pv);
            if (nv >= 3 && cx == max(qx0, world_cell(bb[0], w.origin_x, w.cell, w.nx)) &&
                cy == max(qy0, world_cell(bb[1], w.origin_y, w.cell, w.ny))) {
              d = poly_distance(w.poly_xy + (size_t)o * w.max_pv * 2, nv, x, y);
              take = d <= R;
            }
          }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, take);
        if (!bal) continue;
        const int cnt = __popc(bal);
        total += cnt;
        if (c + cnt > WS_CAP) c = world_keep_best(bd, bo, td, to, c, K, lane);
        if (take) {
          const int pos = c + __popc(bal & ((1u << lane) - 1u));
          bd[pos] = d; bo[pos] = o;
        }
        c += cnt;
        __syncwarp();
      }
    }
  }
  const int k = world_keep_best(bd, bo, td, to, c, K, lane);
  if (lane < K) to[lane] = -1;
  __syncwarp();
  if (lane < k) {  // slot = rank by map index among the taken
    const int oi = bo[lane];
    int s = 0;
    for (int j = 0; j < k; j++) s += bo[j] < oi ? 1 : 0;
    to[s] = oi;
  }
  __syncwarp();
  const int nrow = K * ns;
  double *out = stc_out + (size_t)e * nrow;
  for (int q = lane; q < nrow; q += 32) {
    const int s = q / ns, o = to[s];
    out[q] = (o >= 0 && o < w.M) ? w.rows[(size_t)o * ns + (q - s * ns)] : 0.0;
  }
  if (slot_poly && lane < K) slot_poly[(size_t)e * K + lane] = to[lane];
  if (n_reach && lane == 0) n_reach[e] = total;
}

cudaError_t launch_fleet_world_select(const ttmpc_fleet &f, const ttmpc_fleet_world &w, int K, int ns,
                                      double *stc_out, int *slot_poly, int *n_reach, cudaStream_t st) {
  fleet_world_select_kernel<<<(f.n + WS_WARPS - 1) / WS_WARPS, 32 * WS_WARPS, 0, st>>>(
      f.state, f.n, w, K, ns, stc_out, slot_poly, n_reach);
  return cudaGetLastError();
}

cudaError_t launch_fleet_pack(const ttmpc_fleet &f, const FleetDims &d, double *p, double *prev_u,
                              const int *warm_exit, const ttmpc_fleet_tasks *tasks, cudaStream_t st) {
  ttmpc_fleet_tasks tk = {};
  if (tasks && tasks->max_tasks > 0) tk = *tasks;
  fleet_pack_kernel<<<f.n, 128, 0, st>>>(f, d, p, prev_u, warm_exit, tk);
  return cudaGetLastError();
}
cudaError_t launch_fleet_advance(const ttmpc_fleet &f, const FleetDims &d, const double *u,
                                 const int *exit_status, cudaStream_t st) {
  fleet_advance_kernel<<<(f.n + 127) / 128, 128, 0, st>>>(f, d, u, exit_status);
  return cudaGetLastError();
}

}  // namespace ttmpc
