/*
 * ttfleet_monitor_oracle.c -- CPU ORACLE (test infrastructure, NOT product code) of the fleet
 * monitor (ttmpc_fleet_monitor_device): swept clearance against static polygons and moving discs,
 * contact counters and tracking deviation, restated in plain C.  Built as its own library,
 * oracle/libttfleet_monitor_oracle.so; tests/fleet_monitor_ref.py binds it.
 *
 * Compiled with -ffp-contract=off like the kernels' -fmad=false: the CUDA path reproduces every
 * output bit for bit.
 */
#include <math.h>
#include <stddef.h>

#include "../include/ttmpc.h"

double ttfleet_oracle_seg_distance(double ax, double ay, double bx, double by, double px, double py);
double ttfleet_oracle_swept_poly_distance(const double *xy, int nv, double x0, double y0, double x1, double y1);
double ttfleet_oracle_swept_disc_distance(double x0, double y0, double x1, double y1, double lx, double ly,
                                          double cx, double cy);
double ttfleet_oracle_polyline_distance(const double *ref, int lo, int hi, double px, double py);
void ttfleet_oracle_monitor(const ttmpc_fleet *f, const ttmpc_fleet_monitor *m);

/* shapely Polygon.contains(Point): strictly inside, even-odd rule (as ttfleet_oracle.c) */
static int poly_contains(const double *xy, int nv, double px, double py) {
  int in = 0;
  for (int i = 0, j = nv - 1; i < nv; j = i++) {
    const double xi = xy[2 * i], yi = xy[2 * i + 1], xj = xy[2 * j], yj = xy[2 * j + 1];
    if (((yi > py) != (yj > py)) && (px < (xj - xi) * (py - yi) / (yj - yi) + xi)) in = !in;
  }
  return in;
}

/* distance of (px, py) to the segment (ax, ay) -> (bx, by) */
double ttfleet_oracle_seg_distance(double ax, double ay, double bx, double by, double px, double py) {
  const double dx = bx - ax, dy = by - ay;
  const double len2 = dx * dx + dy * dy;
  double t = 0.0;
  if (len2 > 0.0) { t = ((px - ax) * dx + (py - ay) * dy) / len2; t = t < 0.0 ? 0.0 : (t > 1.0 ? 1.0 : t); }
  const double qx = ax + t * dx - px, qy = ay + t * dy - py;
  return sqrt(qx * qx + qy * qy);
}

/* distance of the chord (x0, y0) -> (x1, y1) to a polygon ring: 0 if an endpoint is inside or the
 * chord properly crosses an edge, else the least endpoint-to-edge and vertex-to-chord distance */
double ttfleet_oracle_swept_poly_distance(const double *xy, int nv, double x0, double y0, double x1, double y1) {
  if (poly_contains(xy, nv, x0, y0) || poly_contains(xy, nv, x1, y1)) return 0.0;
  const int moved = x0 != x1 || y0 != y1;
  const double cx = x1 - x0, cy = y1 - y0;
  double best = INFINITY;
  for (int i = 0, j = nv - 1; i < nv; j = i++) {
    const double ax = xy[2 * j], ay = xy[2 * j + 1], bx = xy[2 * i], by = xy[2 * i + 1];
    double d = ttfleet_oracle_seg_distance(ax, ay, bx, by, x0, y0);
    if (moved) {
      const double ex = bx - ax, ey = by - ay;
      const double o0 = ex * (y0 - ay) - ey * (x0 - ax), o1 = ex * (y1 - ay) - ey * (x1 - ax);
      const double oa = cx * (ay - y0) - cy * (ax - x0), ob = cx * (by - y0) - cy * (bx - x0);
      if (((o0 > 0.0 && o1 < 0.0) || (o0 < 0.0 && o1 > 0.0)) && ((oa > 0.0 && ob < 0.0) || (oa < 0.0 && ob > 0.0)))
        return 0.0;
      const double d1 = ttfleet_oracle_seg_distance(ax, ay, bx, by, x1, y1);
      const double dv = ttfleet_oracle_seg_distance(x0, y0, x1, y1, ax, ay);
      if (d1 < d) d = d1;
      if (dv < d) d = dv;
    }
    if (d < best) best = d;
  }
  return best;
}

/* least distance between a robot moving (x0, y0) -> (x1, y1) and an obstacle centre moving
 * (lx, ly) -> (cx, cy) over the same step, both linear in time */
double ttfleet_oracle_swept_disc_distance(double x0, double y0, double x1, double y1, double lx, double ly,
                                          double cx, double cy) {
  return ttfleet_oracle_seg_distance(x0 - lx, y0 - ly, x1 - cx, y1 - cy, 0.0, 0.0);
}

/* distance of (px, py) to the polyline through rows lo .. hi-1 of ref [][3]; one row (or none):
 * the point distance to row lo */
double ttfleet_oracle_polyline_distance(const double *ref, int lo, int hi, double px, double py) {
  double dev = ttfleet_oracle_seg_distance(ref[3 * lo], ref[3 * lo + 1], ref[3 * lo], ref[3 * lo + 1], px, py);
  if (hi - lo >= 2) {
    dev = INFINITY;
    for (int i = lo + 1; i < hi; i++) {
      const double d = ttfleet_oracle_seg_distance(ref[3 * i - 3], ref[3 * i - 2], ref[3 * i], ref[3 * i + 1], px, py);
      if (d < dev) dev = d;
    }
  }
  return dev;
}

/* fleet_monitor_kernel, robot by robot (include/ttmpc.h, ttmpc_fleet_monitor) */
void ttfleet_oracle_monitor(const ttmpc_fleet *f, const ttmpc_fleet_monitor *m) {
  for (int e = 0; e < f->n; e++) {
    double *pv = m->prev_xy + 2 * e;
    const double x0 = pv[0], y0 = pv[1], x1 = f->state[3 * e], y1 = f->state[3 * e + 1];
    double c = INFINITY;
    if (m->poly_xy) {
      const double *pxy = m->poly_xy + (m->poly_shared ? 0 : (size_t)e * m->max_poly * m->max_pv * 2);
      const int *pnv = m->poly_nv + (m->poly_shared ? 0 : (size_t)e * m->max_poly);
      for (int o = 0; o < m->max_poly; o++) {
        const int nv = pnv[o] < m->max_pv ? pnv[o] : m->max_pv;
        if (nv < 3) continue;
        const double d = ttfleet_oracle_swept_poly_distance(pxy + (size_t)o * m->max_pv * 2, nv, x0, y0, x1, y1) -
                         m->robot_radius;
        if (d < c) c = d;
      }
    }
    if (f->dyn_cur) {
      const double r = m->moving_radius + m->robot_radius;
      for (int j = 0; j < f->n_dyn_live; j++) {
        const double *cur = f->dyn_cur + ((size_t)e * f->n_dyn_live + j) * 2;
        const double *last = f->dyn_last + ((size_t)e * f->n_dyn_live + j) * 2;
        const double d = ttfleet_oracle_swept_disc_distance(x0, y0, x1, y1, last[0], last[1], cur[0], cur[1]) - r;
        if (d < c) c = d;
      }
    }
    m->clearance[e] = c;
    if (c < m->min_clearance[e]) m->min_clearance[e] = c;
    const int contact = c <= 0.0;
    if (contact) {
      m->contact_steps[e] += 1;
      if (m->first_contact[e] < 0) m->first_contact[e] = m->step;
    }
    if (f->status[e] == TTMPC_FLEET_RUNNING) {
      const int k = f->action_steps, L = f->ref_len[e], idx = f->idx_ref[e];
      int lo = idx - k; if (lo < 0) lo = 0;
      int hi = idx + 5 * k; if (hi > L) hi = L;
      const double dev = ttfleet_oracle_polyline_distance(f->ref_traj + (size_t)e * f->ref_stride * 3, lo, hi, x1, y1);
      if (dev > m->deviation_max[e]) m->deviation_max[e] = dev;
      m->deviation_sum[e] = m->deviation_sum[e] + dev;
      m->moved_steps[e] += 1;
      if (m->stop_on_contact && contact) f->status[e] = TTMPC_FLEET_COLLIDED;
    }
    pv[0] = x1; pv[1] = y1;
  }
}
