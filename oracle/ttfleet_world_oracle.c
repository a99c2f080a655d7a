/*
 * ttfleet_world_oracle.c -- CPU ORACLE (test infrastructure, NOT product code) of the map selection
 * (ttmpc_fleet_world_select_device): each robot's nearest map polygons by brute force over all M,
 * with no grid.  Built as its own library, oracle/libttfleet_world_oracle.so; tests/fleet_world_ref.py
 * binds it.
 *
 * Compiled with -ffp-contract=off like the kernels' -fmad=false: the distance is the same sequence
 * of IEEE operations, so the CUDA path reproduces every output bit for bit.
 */
#include <math.h>
#include <stddef.h>
#include <stdlib.h>

#include "../include/ttmpc.h"

double ttfleet_oracle_world_distance(const double *xy, int nv, double px, double py);
void ttfleet_oracle_world_select(const ttmpc_config *cfg, int n, const double *state, const ttmpc_fleet_world *w,
                                 double *stc_out, int *slot_poly, int *n_reach);

/* shapely Polygon.contains(Point) / Polygon.distance(Point), as poly_distance in ttmpc_fleet.cu */
double ttfleet_oracle_world_distance(const double *xy, int nv, double px, double py) {
  int in = 0;
  for (int i = 0, j = nv - 1; i < nv; j = i++) {
    const double xi = xy[2 * i], yi = xy[2 * i + 1], xj = xy[2 * j], yj = xy[2 * j + 1];
    if (((yi > py) != (yj > py)) && (px < (xj - xi) * (py - yi) / (yj - yi) + xi)) in = !in;
  }
  if (in) return 0.0;
  double best = INFINITY;
  for (int i = 0, j = nv - 1; i < nv; j = i++) {
    const double ax = xy[2 * j], ay = xy[2 * j + 1], dx = xy[2 * i] - ax, dy = xy[2 * i + 1] - ay;
    const double len2 = dx * dx + dy * dy;
    double t = 0.0;
    if (len2 > 0.0) { t = ((px - ax) * dx + (py - ay) * dy) / len2; t = t < 0.0 ? 0.0 : (t > 1.0 ? 1.0 : t); }
    const double qx = ax + t * dx - px, qy = ay + t * dy - py;
    const double d = sqrt(qx * qx + qy * qy);
    if (d < best) best = d;
  }
  return best;
}

typedef struct { double d; int o; } key;
static int by_key(const void *a, const void *b) {
  const key *x = a, *y = b;
  if (x->d != y->d) return x->d < y->d ? -1 : 1;
  return (x->o > y->o) - (x->o < y->o);
}
static int by_index(const void *a, const void *b) { return (*(const int *)a > *(const int *)b) - (*(const int *)a < *(const int *)b); }

/* every robot of state [n][3]: all M distances, the eligible ones sorted by (d, o), the first
 * Nstcobs written in map-index order (include/ttmpc.h, ttmpc_fleet_world) */
void ttfleet_oracle_world_select(const ttmpc_config *cfg, int n, const double *state, const ttmpc_fleet_world *w,
                                 double *stc_out, int *slot_poly, int *n_reach) {
  const int K = cfg->Nstcobs, ns = cfg->nstcobs;
  key *keys = malloc(sizeof(key) * (size_t)(w->M > 0 ? w->M : 1));
  int slots[32];
  for (int e = 0; e < n; e++) {
    const double x = state[3 * e], y = state[3 * e + 1];
    int c = 0;
    for (int o = 0; o < w->M; o++) {
      int nv = w->poly_nv[o];
      if (nv > w->max_pv) nv = w->max_pv;
      if (nv < 3) continue;
      const double d = ttfleet_oracle_world_distance(w->poly_xy + (size_t)o * w->max_pv * 2, nv, x, y);
      if (d <= w->reach) { keys[c].d = d; keys[c].o = o; c++; }
    }
    qsort(keys, (size_t)c, sizeof(key), by_key);
    const int k = c < K ? c : K;
    for (int s = 0; s < k; s++) slots[s] = keys[s].o;
    qsort(slots, (size_t)k, sizeof(int), by_index);
    for (int s = 0; s < K; s++) {
      double *out = stc_out + ((size_t)e * K + s) * ns;
      for (int r = 0; r < ns; r++) out[r] = s < k ? w->rows[(size_t)slots[s] * ns + r] : 0.0;
      if (slot_poly) slot_poly[(size_t)e * K + s] = s < k ? slots[s] : -1;
    }
    if (n_reach) n_reach[e] = c;
  }
  free(keys);
}
