/*
 * ttfleet_tasks_oracle.c -- CPU ORACLE (test infrastructure, NOT product code) of the task queues of
 * the fleet step (ttmpc_fleet_step_tasks_device): the reference's get_global_ref_traj sampler and
 * the kernels' tt_atan2, restated in plain C.  Built as its own library,
 * oracle/libttfleet_tasks_oracle.so; tests/fleet_tasks_ref.py binds it.
 *
 * use_libm = 1: hypot / atan2 from libm, as the reference's math module does.
 * use_libm = 0: the device's arithmetic -- sqrt(fma(dx,dx,dy*dy)) and tt_atan2 -- which the CUDA
 *               path reproduces bit for bit (compiled with -ffp-contract=off like the kernels'
 *               -fmad=false).
 */
#include <math.h>

double ttmpc_oracle_atan2(double y, double x);
int ttfleet_oracle_global_ref_traj(const double *path, int n_nodes, double x, double y, double ts,
                                   double speed, int cap, double *out, int use_libm);

static double hyp(double dx, double dy, int use_libm) {
  return use_libm ? hypot(dx, dy) : sqrt(fma(dx, dx, dy * dy));
}

/* tt_atan2 of csrc/ttmpc_device.cuh: fdlibm's atan2 with Horner in fma and the rounding error of
 * y/x corrected through 1 / (1 + t^2).  Same operations in the same order as the kernels.       */
static double tt_atan_ratio(double ay, double ax) {
  const double t = ay / ax;
  if (!(t <= 0x1p60)) return 1.57079632679489655800e+00;
  if (t < 0x1p-27) return t;
  const double e = fma(-t, ax, ay) / ax / fma(t, t, 1.0);
  double r, hi, lo;
  int id;
  if (t < 0.4375) { id = -1; r = t; hi = lo = 0.0; }
  else if (t < 0.6875) { id = 0; r = (2.0 * t - 1.0) / (2.0 + t); hi = 4.63647609000806093515e-01; lo = 2.26987774529616870924e-17; }
  else if (t < 1.1875) { id = 1; r = (t - 1.0) / (t + 1.0); hi = 7.85398163397448278999e-01; lo = 3.06161699786838301793e-17; }
  else if (t < 2.4375) { id = 2; r = (t - 1.5) / fma(1.5, t, 1.0); hi = 9.82793723247329054082e-01; lo = 1.39033110312309984516e-17; }
  else { id = 3; r = -1.0 / t; hi = 1.57079632679489655800e+00; lo = 6.12323399573676603587e-17; }
  const double z = r * r, w = z * z;
  double s1 = fma(w, 1.62858201153657823623e-02, 4.97687799461593236017e-02);
  s1 = fma(w, s1, 6.66107313738753120669e-02);
  s1 = fma(w, s1, 9.09088713343650656196e-02);
  s1 = fma(w, s1, 1.42857142725034663711e-01);
  s1 = fma(w, s1, 3.33333333333329318027e-01);
  double s2 = fma(w, -3.65315727442169155270e-02, -5.83357013379057348645e-02);
  s2 = fma(w, s2, -7.69187620504482999495e-02);
  s2 = fma(w, s2, -1.11111104054623557880e-01);
  s2 = fma(w, s2, -1.99999999998764832476e-01);
  const double s = fma(z, s1, w * s2);
  if (id < 0) return r - fma(r, s, -e);
  return hi - ((fma(r, s, -lo) - r) - e);
}
double ttmpc_oracle_atan2(double y, double x) {
  const double pi = 3.1415926535897931160e+00, pi_lo = 1.2246467991473531772e-16;
  if (x != x || y != y) return x + y;
  const double ax = fabs(x), ay = fabs(y);
  const int xneg = signbit(x) != 0;
  double z;
  if (ay == 0.0) z = xneg ? pi : 0.0;
  else if (ax == INFINITY) {
    if (ay == INFINITY) z = xneg ? 2.35619449019234483700e+00 : 7.85398163397448278999e-01;
    else z = xneg ? pi : 0.0;
  }
  else if (ax == 0.0 || ay == INFINITY) z = 1.57079632679489655800e+00;
  else {
    z = tt_atan_ratio(ay, ax);
    if (xneg) z = pi - (z - pi_lo);
  }
  return copysign(z, y);
}

/* TrajectoryGenerator.get_global_ref_traj (trajectory_generator.py:160-201; planner.py restates it)
 * from (x, y) along the polyline path [n_nodes][2], as the fleet pack kernel samples a queued task:
 * rows (x, y, heading) into out [cap][3] (NULL: count only).  Returns the row count, or -1 for a
 * task that cannot be driven: no node, a walk that would index past the last node (the reference
 * raises IndexError), no row, or more than cap rows.
 * use_libm = 1: hypot / atan2 from libm, as the reference's math module; 0: the device's
 * sqrt(fma(dx,dx,dy*dy)) and tt_atan2 (ttmpc_oracle_atan2), bit for bit with the kernel. */
int ttfleet_oracle_global_ref_traj(const double *path, int n_nodes, double x, double y, double ts,
                                   double speed, int cap, double *out, int use_libm) {
  if (n_nodes < 1) return -1;
  double px = x, py = y, tx = path[0], ty = path[1], ux = 0.0, uy = 0.0, gap = 0.0;
  int k = 0, rows = 0, alive = 1;
  while (alive) {
    for (;;) {
      gap = hyp(tx - px, ty - py, use_libm);
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
      if (k > n_nodes - 1) { alive = 0; break; }
      tx = path[2 * k]; ty = path[2 * k + 1];
    }
    if (!(gap < 1e-9)) {
      if (rows >= cap) return -1;
      if (out) {
        out[3 * rows] = px; out[3 * rows + 1] = py;
        out[3 * rows + 2] = use_libm ? atan2(uy, ux) : ttmpc_oracle_atan2(uy, ux);
      }
      rows++;
    }
  }
  return rows > 0 ? rows : -1;
}
