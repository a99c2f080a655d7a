// ttdqn.cu -- DQN companion kernel: sector+ray ("lidar") observation against the
// obstacle set, Q-network inference and argmax, one environment per warp, so
// the DQN-boosted action selection stays on the device next to the NMPC solve.
//
// Reference behaviour:
//   SectorAndRayObservation.external_obs
//     /root/reference/src/pkg_dqn/environment/components/ext_obsv_sector_and_ray.py:33-83
//   normalize_distance           src/pkg_dqn/environment/components/utils.py:10-15
//   model.predict(obsv, deterministic=True)   src/main.py:148
//     (SB3 1.6.2 DQN MultiInputPolicy: concat(external, internal) -> 46-16-16-9 ReLU MLP -> argmax)
//
// Geometry: for sector triangle T with apex at the agent A, and a closed ring G,
// the closest point of T^G to A lies on G's boundary whenever A is outside G, so
// the sector distance is min over edges e of dist(A, e clipped to T); the ray
// distance is the first hit along the centre ray of length L, counted only for rings that meet T
// (the reference intersects the ray with a ring only when the sector intersection is non-empty: a
// ring crossing the ray between L cos(pi / ns), where the ray leaves T, and L is not seen unless
// another part of it reaches into T).  A inside a solid ring gives 0
// for every sector.  Lanes split the edges; the 16 minima are warp-reduced.  Moving
// solid rings (ttdqn_moving, observe_act_moving_kernel) spread their (ring, edge) pairs over the
// lanes instead (moving_minima).
//
// The Q-network (46-16-16-9 for the reference's ray model) runs on the TENSOR CORES in its own
// kernel, qnet_mma_kernel: 16 environments per warp tile, mma.sync.m16n8k8 TF32 with fp32
// accumulation, every operand split EXACTLY into three TF32 numbers (x = hi + mid + lo) and six
// products per term kept (everything above 2^-33 of it), which holds the 1e-5 Q-value parity a
// plain TF32 / bf16 product (~1e-3) or a two-way split (1.7e-5 measured) cannot
// (tests/test_gpu_parity.py, tools/qnet_diag.py).  Layer shapes other than
// 16-wide hidden layers fall back to the FMA-pipe path inside observe_act_kernel (fp64
// accumulation, one rounding per neuron).  Why mma.sync and not tcgen05: the whole network is
// 1.5 kFLOP per environment, 25 MFLOP for 16384 of them; the 16x8x8 warp tile matches the 16-wide
// layers, while a tcgen05 tile (M = 128 rows, operands through shared-memory descriptors,
// accumulator in TMEM, mbarrier hand-offs between three dependent layers) would spend more on
// its set-up than on the math.
#include <cuda_runtime.h>
#include <math.h>

#include <cstdlib>
#include <mutex>
#include <string>

#include "../../include/ttmpc.h"
#include "ttmpc_device.cuh"

namespace ttdqn {

constexpr unsigned FULL = 0xffffffffu;
constexpr int MAX_SEG = 16;

struct Args {
  ttdqn_scene_layout lay;
  int n_in, n_h1, n_h2, n_out;
  const float *w0, *b0, *w1, *b1, *w2, *b2;
  const double *agent, *poly_xy;
  const int *poly_off, *is_solid, *n_poly;
  const float *internal;
  float *old_ext, *ext, *q;
  int *action;
  double *seg_dist, *ray_dist;
  int n_envs;
  float *obs;     // [n_envs][obs_stride] network input rows (qnet_mma_kernel reads them) or null
  int obs_stride; // n_in padded to a multiple of 8
  int defer_net;  // 1: the MLP runs in qnet_mma_kernel, this kernel only writes `obs`
};

__device__ __forceinline__ double cross2(double ax, double ay, double bx, double by) {
  return ax * by - ay * bx;
}

struct Sector {  // per-sector constants in shared memory
  double V[3][2];
  double rx, ry;
};

__device__ __forceinline__ bool clip_to_triangle(const Sector &S, double p0x, double p0y, double dx,
                                                 double dy, double &t0, double &t1) {
  double lo = 0.0, hi = 1.0;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const int j = (i + 1) % 3;
    const double ex = S.V[j][0] - S.V[i][0], ey = S.V[j][1] - S.V[i][1];
    const double f0 = cross2(ex, ey, p0x - S.V[i][0], p0y - S.V[i][1]);
    const double f1 = cross2(ex, ey, dx, dy);
    if (f1 == 0.0) {
      if (f0 < 0.0) return false;
    } else {
      const double t = -f0 / f1;
      if (f1 > 0.0) { if (t > lo) lo = t; }
      else          { if (t < hi) hi = t; }
    }
    if (lo > hi) return false;
  }
  t0 = lo; t1 = hi;
  return true;
}

__device__ __forceinline__ double ray_seg_hit(double ax, double ay, double rx, double ry, double L,
                                              double p0x, double p0y, double p1x, double p1y) {
  const double dx = p1x - p0x, dy = p1y - p0y;
  const double wx = p0x - ax, wy = p0y - ay;
  const double den = cross2(rx, ry, dx, dy);
  if (den != 0.0) {
    const double s = cross2(wx, wy, dx, dy) / den;
    const double t = cross2(wx, wy, rx, ry) / den;
    if (t >= 0.0 && t <= 1.0 && s >= 0.0 && s <= L) return s;
    return INFINITY;
  }
  if (cross2(wx, wy, rx, ry) != 0.0) return INFINITY;
  const double s0 = wx * rx + wy * ry, s1 = (p1x - ax) * rx + (p1y - ay) * ry;
  const double lo = fmin(s0, s1), hi = fmax(s0, s1);
  if (hi < 0.0 || lo > L) return INFINITY;
  return fmax(lo, 0.0);
}

__device__ __forceinline__ float normalize_distance_f32(float d, float max_distance) {
  float t = -2.0f * d;
  t = t / max_distance;
  t = (float)exp((double)t); /* correctly rounded fp32 exp on both sides */
  t = 1.0f + t;
  t = 2.0f / t;
  return t - 1.0f;
}

__device__ __forceinline__ double wmin(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, o));
  return v;
}

// one edge p0 -> p1 into this lane's running sector and ray minima.  Only ray hits at s <= Lmax are
// taken: Lmax is L when no vertex of the environment lies beyond Lin, else Lin.  Hits up to Lin lie
// inside the sector triangle (the ray leaves it at L cos(pi / ns); Lin stays 2^-20 of that short of
// it), so their ring meets the triangle.  A hit beyond Lin counts only if some edge
// of its ring meets the triangle (the reference looks for a ring's ray hit only when the sector
// intersection is non-empty); such a hit needs a vertex farther than Lin from the agent, and only
// then are a ring's edges passed again, sector by sector, through far_edge_hit / take_ray.
__device__ __forceinline__ void edge_minima(const Sector *sec, int ns, double ax, double ay, double Lmax,
                                            double p0x, double p0y, double p1x, double p1y,
                                            double (&dseg)[MAX_SEG], double (&dray)[MAX_SEG]) {
  const double dx = p1x - p0x, dy = p1y - p0y;
  const double dd = dx * dx + dy * dy;
#pragma unroll
  for (int i = 0; i < MAX_SEG; i++) {
    if (i < ns) {
      const Sector &S = sec[i];
      double t0, t1;
      if (clip_to_triangle(S, p0x, p0y, dx, dy, t0, t1)) {
        double t = t0;
        if (dd > 0.0) {
          t = ((ax - p0x) * dx + (ay - p0y) * dy) / dd;
          t = fmin(fmax(t, t0), t1);
        }
        const double qx = p0x + t * dx - ax, qy = p0y + t * dy - ay;
        dseg[i] = fmin(dseg[i], sqrt(qx * qx + qy * qy));
      }
      dray[i] = fmin(dray[i], ray_seg_hit(ax, ay, S.rx, S.ry, Lmax, p0x, p0y, p1x, p1y));
    }
  }
}

// ray hit of the edge p0 -> p1 in sector i (a run-time index: one copy of the code for the rare
// rings that reach beyond Lin), and whether the edge meets sector i's triangle
__device__ __forceinline__ double far_edge_hit(const Sector &S, double ax, double ay, double L, double p0x,
                                               double p0y, double p1x, double p1y, bool &touch) {
  double t0, t1;
  touch = touch || clip_to_triangle(S, p0x, p0y, p1x - p0x, p1y - p0y, t0, t1);
  return ray_seg_hit(ax, ay, S.rx, S.ry, L, p0x, p0y, p1x, p1y);
}
// dray[i] = fmin(dray[i], h) for a run-time i, without indexing the register array
__device__ __forceinline__ void take_ray(double (&dray)[MAX_SEG], int i, double h) {
#pragma unroll
  for (int k = 0; k < MAX_SEG; k++)
    if (k == i) dray[k] = fmin(dray[k], h);
}

// Moving solid rings (ttdqn_moving): the (ring, edge) pairs are spread over the lanes, 32 / max_pv
// whole rings per pass, lane = slot * max_pv + edge.  Each lane forms its edge e -> e+1 of ring
// centre + offset and the even-odd crossing of the pair (e+1, e), which is the pair the static ring
// loop tests on lane e+1; a ballot masked to the ring's lanes gives the ring's parity.  Every edge
// is the same arithmetic as for a static ring and min / OR ignore the order, so the result equals
// that of the rings appended as static solid rings.  Returns whether the agent is inside any ring.
__device__ __forceinline__ bool moving_minima(const ttdqn_moving &M, int env, int lane, const Sector *sec, int ns,
                                              double ax, double ay, double L, double Lin, double Lfar2,
                                              double (&dseg)[MAX_SEG], double (&dray)[MAX_SEG]) {
  const int pv = M.max_pv, per = 32 / pv, slot = lane / pv, e = lane - slot * pv;
  const unsigned mask = slot < per ? ((pv == 32 ? FULL : (1u << pv) - 1u) << (slot * pv)) : 0u;
  const double *cen = M.centre + (size_t)env * M.n_live * 2;
  const double *sxy = M.shape_xy + (M.shape_shared ? 0 : (size_t)env * M.n_live * pv * 2);
  const int *snv = M.shape_nv + (M.shape_shared ? 0 : (size_t)env * M.n_live);
  bool inside = false;
  for (int o0 = 0; o0 < M.n_live; o0 += per) {
    const int o = o0 + slot;
    const int nv = (slot < per && o < M.n_live) ? min(snv[o], pv) : 0;
    const bool edge = nv >= 3 && e < nv;
    double p0x = 0.0, p0y = 0.0, p1x = 0.0, p1y = 0.0;
    int cross = 0;
    if (edge) {
      const double cx = cen[2 * o], cy = cen[2 * o + 1], *r = sxy + (size_t)o * pv * 2;
      const int e2 = (e + 1 == nv) ? 0 : e + 1;
      p0x = cx + r[2 * e]; p0y = cy + r[2 * e + 1];
      p1x = cx + r[2 * e2]; p1y = cy + r[2 * e2 + 1];
      if (((p1y > ay) != (p0y > ay)) && (ax < (p0x - p1x) * (ay - p1y) / (p0y - p1y) + p1x)) cross = 1;
    }
    const bool in_ring = (__popc(__ballot_sync(FULL, cross) & mask) & 1) != 0;
    inside = inside || in_ring;
    bool far = false;
    if (edge && !in_ring) {
      edge_minima(sec, ns, ax, ay, Lin, p0x, p0y, p1x, p1y, dseg, dray);
      far = (p0x - ax) * (p0x - ax) + (p0y - ay) * (p0y - ay) > Lfar2;
    }
    if (__any_sync(FULL, far)) {   // rings reaching beyond Lin: their ray hits count where they meet a triangle
      const int end = slot * pv + pv;
#pragma unroll 1
      for (int i = 0; i < ns; i++) {
        bool touch = false;
        double h = INFINITY;
        if (edge && !in_ring) h = far_edge_hit(sec[i], ax, ay, L, p0x, p0y, p1x, p1y, touch);
        // OR over the ring's lanes [slot * pv, end): lane l gathers [l, min(l + 2o, end))
        unsigned tv = touch ? 1u : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned v = __shfl_down_sync(FULL, tv, o);
          if (lane + o < end) tv |= v;
        }
        tv = __shfl_sync(FULL, tv, (slot * pv) & 31);
        if (tv) take_ray(dray, i, h);
      }
    }
  }
  return __any_sync(FULL, inside);
}

// shared memory per block: Q-net weights (once) + per-warp scratch.  MOVING: also the moving rings
// of ttdqn_moving (n_live > 0); the instantiation without them is observe_act_kernel.
template <bool MOVING>
__device__ __forceinline__ void observe_act_body(const Args A, const ttdqn_moving M) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ns = A.lay.num_segments;
  const int n_ext = A.lay.use_memory ? 4 * ns : 2 * ns;
  const int nw0 = A.n_in * A.n_h1, nw1 = A.n_h1 * A.n_h2, nw2 = A.n_h2 * A.n_out;
  float *W0 = reinterpret_cast<float *>(smem_raw);
  float *B0 = W0 + nw0, *W1 = B0 + A.n_h1, *B1 = W1 + nw1, *W2 = B1 + A.n_h2, *B2 = W2 + nw2;
  size_t off = ((size_t)(nw0 + A.n_h1 + nw1 + A.n_h2 + nw2 + A.n_out) * sizeof(float) + 15) / 16 * 16;
  const size_t per_warp = sizeof(Sector) * MAX_SEG + sizeof(float) * (size_t)(A.n_in + A.n_h1 + A.n_h2 + A.n_out + 4);
  unsigned char *wbase = smem_raw + off + (size_t)warp * ((per_warp + 15) / 16 * 16);
  Sector *sec = reinterpret_cast<Sector *>(wbase);
  float *x = reinterpret_cast<float *>(wbase + sizeof(Sector) * MAX_SEG);
  float *h1 = x + A.n_in, *h2 = h1 + A.n_h1, *qv = h2 + A.n_h2;

  const bool have_net = A.w0 != nullptr;
  if (have_net && !A.defer_net) {
    for (int i = threadIdx.x; i < nw0; i += blockDim.x) W0[i] = A.w0[i];
    for (int i = threadIdx.x; i < A.n_h1; i += blockDim.x) B0[i] = A.b0[i];
    for (int i = threadIdx.x; i < nw1; i += blockDim.x) W1[i] = A.w1[i];
    for (int i = threadIdx.x; i < A.n_h2; i += blockDim.x) B1[i] = A.b1[i];
    for (int i = threadIdx.x; i < nw2; i += blockDim.x) W2[i] = A.w2[i];
    for (int i = threadIdx.x; i < A.n_out; i += blockDim.x) B2[i] = A.b2[i];
  }
  __syncthreads();

  const double L = A.lay.ray_length;
  const double width = 2 * M_PI / ns;
  const double Lin = L * cos(width / 2) * (1.0 - 0x1p-20);  // ray hits up to here lie inside the triangle
  const double Lfar2 = Lin * Lin * (1.0 - 0x1p-20);          // a hit beyond Lin needs a vertex this far (squared)
  for (int env = blockIdx.x * warps + warp; env < A.n_envs; env += gridDim.x * warps) {
    const double ax = A.agent[3 * env], ay = A.agent[3 * env + 1], th = A.agent[3 * env + 2];
    const double *xy = A.poly_xy + (size_t)env * A.lay.max_vert * 2;
    const int *poff = A.poly_off + (size_t)env * (A.lay.max_poly + 1);
    const int *solid = A.is_solid + (size_t)env * A.lay.max_poly;
    const int npoly = A.n_poly[env];
    if (lane < ns) {
      const double angle = th + lane * width;
      const double a1 = angle - width / 2, a2 = angle + width / 2;
      Sector &S = sec[lane];
      S.V[0][0] = ax; S.V[0][1] = ay;
      S.V[1][0] = ax + L * cos(a1); S.V[1][1] = ay + L * sin(a1);
      S.V[2][0] = ax + L * cos(a2); S.V[2][1] = ay + L * sin(a2);
      S.rx = cos(angle); S.ry = sin(angle);
    }
    __syncwarp();
    // a ray hit beyond Lin needs a vertex farther than Lin: without one (every scene smaller than the
    // ray) all hits are taken in the edge loop, as they lie inside their triangle
    bool far_v = false;
    for (int v = lane; v < poff[npoly > 0 ? npoly : 0] - poff[0]; v += 32) {
      const double qx = xy[2 * (poff[0] + v)] - ax, qy = xy[2 * (poff[0] + v) + 1] - ay;
      far_v = far_v || qx * qx + qy * qy > Lfar2;
    }
    const bool far_env = __any_sync(FULL, far_v);
    const double Lx = far_env ? Lin : L;
    double dseg[MAX_SEG], dray[MAX_SEG];
#pragma unroll
    for (int i = 0; i < MAX_SEG; i++) { dseg[i] = INFINITY; dray[i] = INFINITY; }
    bool inside_any = false;
    for (int gidx = 0; gidx < npoly; gidx++) {
      const int v0 = poff[gidx], nv = poff[gidx + 1] - v0;
      if (nv < 2) continue;
      const double *r = xy + 2 * (size_t)v0;
      // even-odd point-in-ring, edges split over lanes
      if (solid[gidx]) {
        int cross = 0;
        for (int e = lane; e < nv; e += 32) {
          const int j = (e == 0) ? nv - 1 : e - 1;
          const double xi = r[2 * e], yi = r[2 * e + 1], xj = r[2 * j], yj = r[2 * j + 1];
          if (((yi > ay) != (yj > ay)) && (ax < (xj - xi) * (ay - yi) / (yj - yi) + xi)) cross ^= 1;
        }
        cross = __reduce_xor_sync(FULL, cross);
        if (cross) { inside_any = true; continue; }
      }
      for (int e = lane; e < nv; e += 32) {
        const int e2 = (e + 1 == nv) ? 0 : e + 1;
        edge_minima(sec, ns, ax, ay, Lx, r[2 * e], r[2 * e + 1], r[2 * e2], r[2 * e2 + 1], dseg, dray);
      }
      if (far_env) {   // ray hits beyond Lin count in the sectors whose triangle the ring meets
#pragma unroll 1
        for (int i = 0; i < ns; i++) {
          bool touch = false;
          double h = INFINITY;
          for (int e = lane; e < nv; e += 32) {
            const int e2 = (e + 1 == nv) ? 0 : e + 1;
            h = fmin(h, far_edge_hit(sec[i], ax, ay, L, r[2 * e], r[2 * e + 1], r[2 * e2], r[2 * e2 + 1], touch));
          }
          if (__any_sync(FULL, touch)) take_ray(dray, i, h);
        }
      }
    }
    if (MOVING && moving_minima(M, env, lane, sec, ns, ax, ay, L, Lin, Lfar2, dseg, dray)) inside_any = true;
#pragma unroll
    for (int i = 0; i < MAX_SEG; i++) {
      if (i < ns) {
        double s = wmin(dseg[i]), r_ = wmin(dray[i]);
        if (inside_any) { s = 0.0; r_ = 0.0; }
        if (lane == 0) {
          if (A.seg_dist) A.seg_dist[(size_t)env * ns + i] = s;
          if (A.ray_dist) A.ray_dist[(size_t)env * ns + i] = r_;
          x[i] = normalize_distance_f32((float)s, (float)A.lay.max_distance);
          x[ns + i] = normalize_distance_f32((float)r_, (float)A.lay.max_distance);
        }
      }
    }
    __syncwarp();
    if (A.lay.use_memory) {
      float *old = A.old_ext + (size_t)env * 2 * ns;
      for (int i = lane; i < 2 * ns; i += 32) {
        x[2 * ns + i] = old[i];
        old[i] = x[i];
      }
    }
    for (int i = lane; i < A.lay.n_internal; i += 32)
      x[n_ext + i] = A.internal ? A.internal[(size_t)env * A.lay.n_internal + i] : 0.0f;
    __syncwarp();
    if (A.ext)
      for (int i = lane; i < n_ext; i += 32) A.ext[(size_t)env * n_ext + i] = x[i];
    if (A.obs)
      for (int i = lane; i < A.obs_stride; i += 32) A.obs[(size_t)env * A.obs_stride + i] = i < A.n_in ? x[i] : 0.0f;
    if (have_net && !A.defer_net) {
      for (int o = lane; o < A.n_h1; o += 32) {
        double a = (double)B0[o];  // fp64 accumulation, one rounding to fp32 per neuron
        for (int i = 0; i < A.n_in; i++) a += (double)W0[o * A.n_in + i] * (double)x[i];
        const float acc = (float)a;
        h1[o] = acc < 0.0f ? 0.0f : acc;
      }
      __syncwarp();
      for (int o = lane; o < A.n_h2; o += 32) {
        double a = (double)B1[o];
        for (int i = 0; i < A.n_h1; i++) a += (double)W1[o * A.n_h1 + i] * (double)h1[i];
        const float acc = (float)a;
        h2[o] = acc < 0.0f ? 0.0f : acc;
      }
      __syncwarp();
      for (int o = lane; o < A.n_out; o += 32) {
        double a = (double)B2[o];
        for (int i = 0; i < A.n_h2; i++) a += (double)W2[o * A.n_h2 + i] * (double)h2[i];
        const float acc = (float)a;
        qv[o] = acc;
        if (A.q) A.q[(size_t)env * A.n_out + o] = acc;
      }
      __syncwarp();
      if (lane == 0 && A.action) {
        int best = 0;
        for (int o = 1; o < A.n_out; o++)
          if (qv[o] > qv[best]) best = o;
        A.action[env] = best;
      }
    }
    __syncwarp();
  }
}
__global__ void __launch_bounds__(128) observe_act_kernel(const __grid_constant__ Args A) {
  observe_act_body<false>(A, ttdqn_moving{});
}
__global__ void __launch_bounds__(128) observe_act_moving_kernel(const __grid_constant__ Args A,
                                                                 const __grid_constant__ ttdqn_moving M) {
  observe_act_body<true>(A, M);
}

// ------------------------------------------------------------------ Q-network on the tensor cores
struct QArgs {
  const float *obs; int obs_stride;  // [n][obs_stride], obs_stride = 8 * ksteps
  const float *w0, *b0, *w1, *b1, *w2, *b2;
  int n_in, n_out, n_envs;
  float *q; int *action;
};
__device__ __forceinline__ unsigned to_tf32(float x) {
  unsigned r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// x = hi + mid + lo EXACTLY, each part representable in TF32 (11 significant bits each cover the
// 24 of fp32).  With only two parts every operand is 2^-22 off, and at |Q| ~ 12 with terms that
// partly cancel that alone cost 1.7e-5 against torch (measured, tools/qnet_diag.py).
__device__ __forceinline__ void split_tf32(float x, unsigned &hi, unsigned &mid, unsigned &lo) {
  hi = to_tf32(x);
  const float r1 = x - __uint_as_float(hi);
  mid = to_tf32(r1);
  lo = to_tf32(r1 - __uint_as_float(mid));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// One layer for a 16-row tile: C[16 x 16] = A[16 x 8*ksteps] . W^T, A fp32 in shared memory (row
// stride as), W pre-split (hi / lo TF32 bit patterns, [16][ws] each).  Fragment layouts of
// mma.m16n8k8: g = lane / 4, t = lane % 4; A: (g, t) (g+8, t) (g, t+4) (g+8, t+4); B: (k = t, n = g)
// (k = t+4, n = g); C: (g, 2t) (g, 2t+1) (g+8, 2t) (g+8, 2t+1).
__device__ __forceinline__ void mlp_layer(const float *As, int as, const unsigned *W3, int ws,
                                          int ksteps, int lane, float (&c0)[4], float (&c1)[4]) {
  const int g = lane >> 2, t = lane & 3;
  const unsigned *Wh = W3, *Wm = W3 + 16 * ws, *Wl = W3 + 32 * ws;
  for (int ks = 0; ks < ksteps; ks++) {
    const int k = 8 * ks + t;
    unsigned ah[4], am[4], al[4];
    split_tf32(As[g * as + k], ah[0], am[0], al[0]);
    split_tf32(As[(g + 8) * as + k], ah[1], am[1], al[1]);
    split_tf32(As[g * as + k + 4], ah[2], am[2], al[2]);
    split_tf32(As[(g + 8) * as + k + 4], ah[3], am[3], al[3]);
#pragma unroll
    for (int nt = 0; nt < 2; nt++) {
      const int n = g + 8 * nt;
      const unsigned bh0 = Wh[n * ws + k], bh1 = Wh[n * ws + k + 4];
      const unsigned bm0 = Wm[n * ws + k], bm1 = Wm[n * ws + k + 4];
      const unsigned bl0 = Wl[n * ws + k], bl1 = Wl[n * ws + k + 4];
      // six products per term (everything down to 2^-33 of it), smallest first, into a fresh
      // accumulator; the k-steps are then summed with ordinary round-to-nearest FADDs (the tensor
      // core's own fp32 accumulation truncates)
      float p[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      mma_tf32(p, am, bm0, bm1);
      mma_tf32(p, al, bh0, bh1);
      mma_tf32(p, ah, bl0, bl1);
      mma_tf32(p, am, bh0, bh1);
      mma_tf32(p, ah, bm0, bm1);
      mma_tf32(p, ah, bh0, bh1);
      float (&c)[4] = nt ? c1 : c0;
      c[0] += p[0]; c[1] += p[1]; c[2] += p[2]; c[3] += p[3];
    }
  }
}
// 16 environments per warp tile, 4 warps per block, grid-stride over the tiles.  Hidden layers are
// 16 wide, n_out <= 16 (rows of W2 beyond n_out are zero).
__global__ void __launch_bounds__(128) qnet_mma_kernel(const __grid_constant__ QArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int ksteps = A.obs_stride / 8;
  const int ws0 = A.obs_stride + 4, ws1 = 20;           // padded strides: conflict-free fragment reads
  unsigned *W0 = reinterpret_cast<unsigned *>(smem_raw);  // [3 parts][16][ws0]
  unsigned *W1 = W0 + 48 * ws0, *W2 = W1 + 48 * ws1;       // [3][16][ws1] each
  float *B0 = reinterpret_cast<float *>(W2 + 48 * ws1), *B1 = B0 + 16, *B2 = B1 + 16;
  float *tiles = B2 + 16;
  float *X = tiles + (size_t)warp * (16 * ws0 + 16 * ws1);  // this warp's input tile, then its hidden tile
  float *H = X + 16 * ws0;
  for (int i = threadIdx.x; i < 16 * ws0; i += blockDim.x) {
    const int n = i / ws0, k = i - n * ws0;
    unsigned hi = 0, mid = 0, lo = 0;
    if (k < A.n_in) split_tf32(A.w0[n * A.n_in + k], hi, mid, lo);
    W0[i] = hi; W0[16 * ws0 + i] = mid; W0[32 * ws0 + i] = lo;
  }
  for (int i = threadIdx.x; i < 16 * ws1; i += blockDim.x) {
    const int n = i / ws1, k = i - n * ws1;
    unsigned hi = 0, mid = 0, lo = 0;
    if (k < 16) split_tf32(A.w1[n * 16 + k], hi, mid, lo);
    W1[i] = hi; W1[16 * ws1 + i] = mid; W1[32 * ws1 + i] = lo;
    hi = mid = lo = 0;
    if (k < 16 && n < A.n_out) split_tf32(A.w2[n * 16 + k], hi, mid, lo);
    W2[i] = hi; W2[16 * ws1 + i] = mid; W2[32 * ws1 + i] = lo;
  }
  if (threadIdx.x < 16) {
    B0[threadIdx.x] = A.b0[threadIdx.x]; B1[threadIdx.x] = A.b1[threadIdx.x];
    B2[threadIdx.x] = threadIdx.x < A.n_out ? A.b2[threadIdx.x] : 0.0f;
  }
  __syncthreads();
  const int n_tiles = (A.n_envs + 15) / 16, warps_total = gridDim.x * (blockDim.x >> 5);
  for (int tile = blockIdx.x * (blockDim.x >> 5) + warp; tile < n_tiles; tile += warps_total) {
    const int e0 = tile * 16;
    // input rows -> shared memory (coalesced: the 16 rows are contiguous in global memory)
    for (int i = lane; i < 16 * A.obs_stride; i += 32) {
      const int r = i / A.obs_stride, k = i - r * A.obs_stride;
      X[r * ws0 + k] = (e0 + r < A.n_envs) ? A.obs[(size_t)e0 * A.obs_stride + i] : 0.0f;
    }
    __syncwarp();
    float c0[4], c1[4];
    // layer 1
    c0[0] = c0[2] = B0[2 * t]; c0[1] = c0[3] = B0[2 * t + 1];
    c1[0] = c1[2] = B0[8 + 2 * t]; c1[1] = c1[3] = B0[8 + 2 * t + 1];
    mlp_layer(X, ws0, W0, ws0, ksteps, lane, c0, c1);
    H[g * ws1 + 2 * t] = fmaxf(c0[0], 0.0f); H[g * ws1 + 2 * t + 1] = fmaxf(c0[1], 0.0f);
    H[(g + 8) * ws1 + 2 * t] = fmaxf(c0[2], 0.0f); H[(g + 8) * ws1 + 2 * t + 1] = fmaxf(c0[3], 0.0f);
    H[g * ws1 + 8 + 2 * t] = fmaxf(c1[0], 0.0f); H[g * ws1 + 8 + 2 * t + 1] = fmaxf(c1[1], 0.0f);
    H[(g + 8) * ws1 + 8 + 2 * t] = fmaxf(c1[2], 0.0f); H[(g + 8) * ws1 + 8 + 2 * t + 1] = fmaxf(c1[3], 0.0f);
    __syncwarp();
    // layer 2 (reads H, writes H: the fragments are in registers before the tile is overwritten)
    c0[0] = c0[2] = B1[2 * t]; c0[1] = c0[3] = B1[2 * t + 1];
    c1[0] = c1[2] = B1[8 + 2 * t]; c1[1] = c1[3] = B1[8 + 2 * t + 1];
    mlp_layer(H, ws1, W1, ws1, 2, lane, c0, c1);
    __syncwarp();
    H[g * ws1 + 2 * t] = fmaxf(c0[0], 0.0f); H[g * ws1 + 2 * t + 1] = fmaxf(c0[1], 0.0f);
    H[(g + 8) * ws1 + 2 * t] = fmaxf(c0[2], 0.0f); H[(g + 8) * ws1 + 2 * t + 1] = fmaxf(c0[3], 0.0f);
    H[g * ws1 + 8 + 2 * t] = fmaxf(c1[0], 0.0f); H[g * ws1 + 8 + 2 * t + 1] = fmaxf(c1[1], 0.0f);
    H[(g + 8) * ws1 + 8 + 2 * t] = fmaxf(c1[2], 0.0f); H[(g + 8) * ws1 + 8 + 2 * t + 1] = fmaxf(c1[3], 0.0f);
    __syncwarp();
    // layer 3 (no activation)
    c0[0] = c0[2] = B2[2 * t]; c0[1] = c0[3] = B2[2 * t + 1];
    c1[0] = c1[2] = B2[8 + 2 * t]; c1[1] = c1[3] = B2[8 + 2 * t + 1];
    mlp_layer(H, ws1, W2, ws1, 2, lane, c0, c1);
    __syncwarp();
    H[g * ws1 + 2 * t] = c0[0]; H[g * ws1 + 2 * t + 1] = c0[1];
    H[(g + 8) * ws1 + 2 * t] = c0[2]; H[(g + 8) * ws1 + 2 * t + 1] = c0[3];
    H[g * ws1 + 8 + 2 * t] = c1[0]; H[g * ws1 + 8 + 2 * t + 1] = c1[1];
    H[(g + 8) * ws1 + 8 + 2 * t] = c1[2]; H[(g + 8) * ws1 + 8 + 2 * t + 1] = c1[3];
    __syncwarp();
    // Q-values out (coalesced) and the arg max of each row: first maximum, like the fold in
    // torch.argmax / the FMA path
    if (A.q)
      for (int i = lane; i < 16 * A.n_out; i += 32) {
        const int r = i / A.n_out, o = i - r * A.n_out;
        if (e0 + r < A.n_envs) A.q[(size_t)(e0 + r) * A.n_out + o] = H[r * ws1 + o];
      }
    if (A.action && lane < 16 && e0 + lane < A.n_envs) {
      int best = 0;
      for (int o = 1; o < A.n_out; o++)
        if (H[lane * ws1 + o] > H[lane * ws1 + best]) best = o;
      A.action[e0 + lane] = best;
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------ internal observation, rl_ref
// One thread per environment: a few dozen flops each, the work is the polyline walk.
__device__ __forceinline__ void rel_obs(double px, double py, const double *agent, double max_distance, float *o) {
  const double dx = px - agent[0], dy = py - agent[1];
  const double rel = atan2(dy, dx) - agent[2];
  o[0] = (float)cos(rel);
  o[1] = (float)sin(rel);
  o[2] = (float)(2.0 / (1.0 + exp(-2.0 * sqrt(dx * dx + dy * dy) / max_distance)) - 1.0);
}
__global__ void __launch_bounds__(128) internal_obs_kernel(int n, int max_nodes, int corner_samples, double offset,
                                                           double max_distance, const double *__restrict__ agent5,
                                                           const double *__restrict__ path_xy,
                                                           const int *__restrict__ path_n, float *__restrict__ obs_all,
                                                           double *__restrict__ progress) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const double *a = agent5 + 5 * e, *xy = path_xy + (size_t)e * max_nodes * 2;
  const int nn = path_n[e];
  float *obs = obs_all + (size_t)e * (5 + 3 * corner_samples);
  obs[0] = (float)(2.0 * (a[3] - (-0.5)) / (1.5 - (-0.5)) - 1.0);
  obs[1] = (float)(2.0 * (a[4] - (-3.0)) / (3.0 - (-3.0)) - 1.0);  // reference quirk: acceleration bounds
  // path.project(agent): arc length of the closest point, first closest segment wins
  double best = INFINITY, s = 0.0, cum = 0.0;
  for (int i = 0; i + 1 < nn; i++) {
    const double ax = xy[2 * i], ay = xy[2 * i + 1], dx = xy[2 * i + 2] - ax, dy = xy[2 * i + 3] - ay;
    const double len2 = dx * dx + dy * dy, len = sqrt(len2);
    double t = 0.0;
    if (len2 > 0.0) {
      t = ((a[0] - ax) * dx + (a[1] - ay) * dy) / len2;
      t = t < 0.0 ? 0.0 : (t > 1.0 ? 1.0 : t);
    }
    const double qx = ax + t * dx - a[0], qy = ay + t * dy - a[1];
    const double d = sqrt(qx * qx + qy * qy);
    if (d < best) { best = d; s = cum + t * len; }
    cum += len;
  }
  if (progress) progress[e] = s;
  // path.interpolate(path_progress + offset)
  {
    const double sq = s + offset;
    double px = xy[2 * (nn - 1)], py = xy[2 * (nn - 1) + 1];
    if (sq <= 0.0 || nn < 2) { px = xy[0]; py = xy[1]; }
    else {
      double c2 = 0.0;
      for (int i = 0; i + 1 < nn; i++) {
        const double ax = xy[2 * i], ay = xy[2 * i + 1], dx = xy[2 * i + 2] - ax, dy = xy[2 * i + 3] - ay;
        const double len = sqrt(dx * dx + dy * dy);
        if (sq <= c2 + len && len > 0.0) {
          const double t = (sq - c2) / len;
          px = ax + t * dx; py = ay + t * dy;
          break;
        }
        c2 += len;
      }
    }
    rel_obs(px, py, a, max_distance, obs + 2);
  }
  // upcoming corners (int_obsv_reference_path_corner.py:27-43)
  double length = 0.0;
  int i = 0;
  while (length < s && i + 1 < nn) {
    const double dx = xy[2 * (i + 1)] - xy[2 * i], dy = xy[2 * (i + 1) + 1] - xy[2 * i + 1];
    length += sqrt(dx * dx + dy * dy);
    i++;
  }
  for (int j = 0; j < corner_samples; j++) {
    if (i > nn - 1) i = nn - 1;
    rel_obs(xy[2 * i], xy[2 * i + 1], a, max_distance, obs + 5 + 3 * j);
    i++;
  }
}
__global__ void __launch_bounds__(128) rl_ref_kernel(int n, int steps, double ts, double ref_speed,
                                                     const double *__restrict__ agent5,
                                                     const int *__restrict__ action_all, double *__restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const double *a = agent5 + 5 * e;
  double x = a[0], y = a[1], th = a[2], v = a[3], w = a[4], s, c;
  const int action = action_all[e];
  for (int j = 0; j < steps; j++) {
    double sp;
    if (j == 0) {  // MobileRobot.step (agent.py:120-145)
      if (action / 3 == 0) v += ts * 1.0;
      if (action / 3 == 2) v += ts * -1.0;
      if (action % 3 == 0) w += ts * 3.0;
      if (action % 3 == 2) w += ts * -3.0;
      if (v > 1.5) v = 1.5;
      if (v < -0.5) v = -0.5;
      if (w > 0.5) w = 0.5;
      if (w < -0.5) w = -0.5;
      th += ts * w;
      sp = v;
    } else {       // step_with_ref_speed -> step_with_decay_angular_velocity (agent.py:86-101)
      w *= 0.95;
      th += ts * w;
      sp = ref_speed <= 0.0 ? 1.5 : ref_speed;
    }
    ttmpc::tt_sincos(th, &s, &c);
    x += (ts * sp) * c; y += (ts * sp) * s;
    out[((size_t)e * steps + j) * 2] = x; out[((size_t)e * steps + j) * 2 + 1] = y;
  }
}

}  // namespace ttdqn

static thread_local std::string g_dqn_err;
extern "C" const char *ttdqn_last_error(void) { return g_dqn_err.c_str(); }
namespace ttmpc { void set_last_error(const std::string &msg); }
static int dfail(int code, const std::string &m) { g_dqn_err = m; ttmpc::set_last_error(m); return code; }
#define DQN_TRY(x)                                                                   \
  do {                                                                               \
    cudaError_t e__ = (x);                                                           \
    if (e__ != cudaSuccess)                                                          \
      return dfail(TTMPC_ERR_CUDA, std::string(#x) + ": " + cudaGetErrorString(e__)); \
  } while (0)

extern "C" void ttdqn_default_layout(ttdqn_scene_layout *l) {
  l->num_segments = 8; l->max_poly = 16; l->max_vert = 512; l->n_internal = 14;
  l->use_memory = 1; l->_pad = 0; l->ray_length = 1000.0; l->max_distance = 10.0;
}

// num_segments 1 and 2 give sector "triangles" of zero area (the far vertices coincide, or lie on a
// line with the apex): whether anything is seen then hangs on the last bit of cos / sin
static int check_layout(const ttdqn_scene_layout *lay, int n) {
  if (!lay || n < 0) return dfail(TTMPC_ERR_BAD_ARG, "layout required, n >= 0");
  if (lay->num_segments < 3 || lay->num_segments > ttdqn::MAX_SEG)
    return dfail(TTMPC_ERR_BAD_CONFIG, "num_segments must be in 3..16");
  return TTMPC_OK;
}

static int observe_act(const ttdqn_scene_layout *lay, const ttdqn_qnet *qn, int n, const double *d_agent,
                       const double *d_poly_xy, const int *d_poly_off, const int *d_is_solid, const int *d_n_poly,
                       const ttdqn_moving *mv, const float *d_internal, float *d_old_ext, float *d_ext,
                       float *d_q, int *d_action, double *d_seg, double *d_ray, void *stream) {
  using namespace ttdqn;
  if (int rc = check_layout(lay, n)) return rc;
  if (lay->use_memory && !d_old_ext) return dfail(TTMPC_ERR_BAD_ARG, "use_memory needs d_old_ext");
  if (mv) {
    if (mv->n_live < 0) return dfail(TTMPC_ERR_BAD_ARG, "moving: n_live must be >= 0");
    if (mv->max_pv < 3 || mv->max_pv > 32) return dfail(TTMPC_ERR_BAD_ARG, "moving: max_pv must be in 3..32");
    if (mv->n_live > 0 && (!mv->centre || !mv->shape_xy || !mv->shape_nv))
      return dfail(TTMPC_ERR_BAD_ARG, "moving: centre, shape_xy and shape_nv are required with n_live > 0");
  }
  const bool moving = mv && mv->n_live > 0;
  if (n == 0) return TTMPC_OK;
  if (!d_agent || !d_poly_xy || !d_poly_off || !d_is_solid || !d_n_poly)
    return dfail(TTMPC_ERR_BAD_ARG, "agent and geometry pointers are required");
  Args A;
  A.lay = *lay;
  const int n_ext = lay->use_memory ? 4 * lay->num_segments : 2 * lay->num_segments;
  if (qn) {
    if (qn->n_in != n_ext + lay->n_internal)
      return dfail(TTMPC_ERR_BAD_CONFIG, "qnet n_in must equal n_ext + n_internal");
    if (qn->n_h1 < 1 || qn->n_h2 < 1 || qn->n_out < 1 || qn->n_h1 > 256 || qn->n_h2 > 256 || qn->n_out > 64)
      return dfail(TTMPC_ERR_BAD_CONFIG, "qnet layer sizes out of range");
    A.n_in = qn->n_in; A.n_h1 = qn->n_h1; A.n_h2 = qn->n_h2; A.n_out = qn->n_out;
    A.w0 = qn->w0; A.b0 = qn->b0; A.w1 = qn->w1; A.b1 = qn->b1; A.w2 = qn->w2; A.b2 = qn->b2;
  } else {
    A.n_in = n_ext + lay->n_internal; A.n_h1 = 1; A.n_h2 = 1; A.n_out = 1;
    A.w0 = A.b0 = A.w1 = A.b1 = A.w2 = A.b2 = nullptr;
  }
  A.agent = d_agent; A.poly_xy = d_poly_xy; A.poly_off = d_poly_off; A.is_solid = d_is_solid;
  A.n_poly = d_n_poly; A.internal = d_internal; A.old_ext = d_old_ext; A.ext = d_ext; A.q = d_q;
  A.action = d_action; A.seg_dist = d_seg; A.ray_dist = d_ray; A.n_envs = n;
  // tensor-core path of the Q-network: 16-wide hidden layers, up to 16 outputs (the reference's
  // SB3 [16, 16] MLP); TTDQN_QNET=fma forces the FMA-pipe path for A/B measurements
  int dev = 0, sms = 0, smem_max = 0;
  DQN_TRY(cudaGetDevice(&dev));
  bool mma = qn && qn->n_h1 == 16 && qn->n_h2 == 16 && qn->n_out <= 16 && qn->n_in <= 248;
  if (const char *e = std::getenv("TTDQN_QNET")) mma = mma && !(e[0] == 'f');
  A.obs = nullptr; A.obs_stride = (A.n_in + 7) / 8 * 8; A.defer_net = 0;
  // shared memory per block: the Q-network's weights and 4 warps' scratch (observe_act_body)
  const int warps = 4;
  size_t wbytes = ((size_t)(A.n_in * A.n_h1 + A.n_h1 + A.n_h1 * A.n_h2 + A.n_h2 + A.n_h2 * A.n_out + A.n_out) * sizeof(float) + 15) / 16 * 16;
  size_t per_warp = (sizeof(Sector) * MAX_SEG + sizeof(float) * (size_t)(A.n_in + A.n_h1 + A.n_h2 + A.n_out + 4) + 15) / 16 * 16;
  size_t smem = wbytes + per_warp * warps;
  DQN_TRY(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if (smem > (size_t)smem_max)
    return dfail(TTMPC_ERR_UNSUPPORTED, "observe_act needs " + std::to_string(smem) +
                                            " bytes of shared memory per block (Q-network weights and scratch), "
                                            "the device allows " + std::to_string(smem_max));
  float *d_obs = nullptr;
  if (mma) {
    // stream-ordered scratch from the device's default memory pool.  The pool's default release
    // threshold is 0 (memory goes back to the OS at every synchronisation and the next call pays
    // milliseconds to get it again): raise it once per device.
    {
      static std::mutex mu;
      static bool raised[64] = {};
      std::lock_guard<std::mutex> lk(mu);
      if (dev >= 0 && dev < 64 && !raised[dev]) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
          unsigned long long keep = ~0ull;
          cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
        raised[dev] = true;
      }
    }
    DQN_TRY(cudaMallocAsync((void **)&d_obs, sizeof(float) * (size_t)n * A.obs_stride, (cudaStream_t)stream));
    A.obs = d_obs; A.defer_net = 1;
  }
  DQN_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const void *kern = moving ? (const void *)observe_act_moving_kernel : (const void *)observe_act_kernel;
  DQN_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int bps = 0;
  DQN_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, warps * 32, smem));
  if (bps < 1) return dfail(TTMPC_ERR_UNSUPPORTED, "observe_act kernel does not fit");
  long long want = ((long long)n + warps - 1) / warps, cap = (long long)sms * bps;
  const int grid = (int)(want < cap ? want : cap);
  if (moving)
    observe_act_moving_kernel<<<grid, warps * 32, smem, (cudaStream_t)stream>>>(A, *mv);
  else
    observe_act_kernel<<<grid, warps * 32, smem, (cudaStream_t)stream>>>(A);
  DQN_TRY(cudaGetLastError());
  if (mma) {
    QArgs Q;
    Q.obs = d_obs; Q.obs_stride = A.obs_stride; Q.w0 = qn->w0; Q.b0 = qn->b0; Q.w1 = qn->w1; Q.b1 = qn->b1;
    Q.w2 = qn->w2; Q.b2 = qn->b2; Q.n_in = qn->n_in; Q.n_out = qn->n_out; Q.n_envs = n; Q.q = d_q; Q.action = d_action;
    const int ws0 = A.obs_stride + 4;
    const size_t qsmem = sizeof(unsigned) * (3 * 16 * ws0 + 6 * 16 * 20) + sizeof(float) * 48 +
                         sizeof(float) * (size_t)warps * (16 * ws0 + 16 * 20);
    DQN_TRY(cudaFuncSetAttribute(qnet_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qsmem));
    const long long tiles = ((long long)n + 15) / 16, qwant = (tiles + warps - 1) / warps, qcap = (long long)sms * 8;
    qnet_mma_kernel<<<(int)(qwant < qcap ? qwant : qcap), warps * 32, qsmem, (cudaStream_t)stream>>>(Q);
    DQN_TRY(cudaGetLastError());
    DQN_TRY(cudaFreeAsync(d_obs, (cudaStream_t)stream));
  }
  return TTMPC_OK;
}

extern "C" int ttdqn_observe_act_device(const ttdqn_scene_layout *lay, const ttdqn_qnet *qn, int n,
                                        const double *d_agent, const double *d_poly_xy,
                                        const int *d_poly_off, const int *d_is_solid,
                                        const int *d_n_poly, const float *d_internal,
                                        float *d_old_ext, float *d_ext, float *d_q, int *d_action,
                                        double *d_seg, double *d_ray, void *stream) {
  return observe_act(lay, qn, n, d_agent, d_poly_xy, d_poly_off, d_is_solid, d_n_poly, nullptr, d_internal,
                     d_old_ext, d_ext, d_q, d_action, d_seg, d_ray, stream);
}

extern "C" int ttdqn_observe_act_moving_device(const ttdqn_scene_layout *lay, const ttdqn_qnet *qn, int n,
                                               const double *d_agent, const double *d_poly_xy,
                                               const int *d_poly_off, const int *d_is_solid,
                                               const int *d_n_poly, const ttdqn_moving *mv,
                                               const float *d_internal, float *d_old_ext, float *d_ext,
                                               float *d_q, int *d_action, double *d_seg, double *d_ray,
                                               void *stream) {
  return observe_act(lay, qn, n, d_agent, d_poly_xy, d_poly_off, d_is_solid, d_n_poly, mv, d_internal,
                     d_old_ext, d_ext, d_q, d_action, d_seg, d_ray, stream);
}

extern "C" int ttdqn_observe_act_host(const ttdqn_scene_layout *lay, const ttdqn_qnet *qn, int n,
                                      const double *h_agent, const double *h_poly_xy,
                                      const int *h_poly_off, const int *h_is_solid,
                                      const int *h_n_poly, const float *h_internal,
                                      float *h_old_ext, float *h_ext, float *h_q, int *h_action,
                                      double *h_seg, double *h_ray) {
  if (int rc = check_layout(lay, n)) return rc;
  if (n == 0) return TTMPC_OK;
  const size_t nn = (size_t)n;
  const int ns = lay->num_segments;
  const int n_ext = lay->use_memory ? 4 * ns : 2 * ns;
  std::string err;
  void *ptrs[32]; int np = 0;
  auto dalloc = [&](size_t bytes, const void *src) -> void * {
    void *d = nullptr;
    if (cudaMalloc(&d, bytes ? bytes : 8) != cudaSuccess) { err = "cudaMalloc failed"; return nullptr; }
    ptrs[np++] = d;
    if (src && cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice) != cudaSuccess) err = "H2D copy failed";
    return d;
  };
  auto cleanup = [&]() { for (int i = 0; i < np; i++) cudaFree(ptrs[i]); };
  double *dag = (double *)dalloc(sizeof(double) * 3 * nn, h_agent);
  double *dxy = (double *)dalloc(sizeof(double) * 2 * nn * lay->max_vert, h_poly_xy);
  int *doff = (int *)dalloc(sizeof(int) * nn * (lay->max_poly + 1), h_poly_off);
  int *dsol = (int *)dalloc(sizeof(int) * nn * lay->max_poly, h_is_solid);
  int *dnp = (int *)dalloc(sizeof(int) * nn, h_n_poly);
  float *dint = h_internal ? (float *)dalloc(sizeof(float) * nn * lay->n_internal, h_internal) : nullptr;
  float *dold = lay->use_memory ? (float *)dalloc(sizeof(float) * nn * 2 * ns, h_old_ext) : nullptr;
  float *dext = (float *)dalloc(sizeof(float) * nn * n_ext, nullptr);
  double *dseg = (double *)dalloc(sizeof(double) * nn * ns, nullptr);
  double *dray = (double *)dalloc(sizeof(double) * nn * ns, nullptr);
  ttdqn_qnet dq; float *dqv = nullptr; int *dact = nullptr;
  if (qn) {
    dq = *qn;
    dq.w0 = (float *)dalloc(sizeof(float) * qn->n_in * qn->n_h1, qn->w0);
    dq.b0 = (float *)dalloc(sizeof(float) * qn->n_h1, qn->b0);
    dq.w1 = (float *)dalloc(sizeof(float) * qn->n_h1 * qn->n_h2, qn->w1);
    dq.b1 = (float *)dalloc(sizeof(float) * qn->n_h2, qn->b1);
    dq.w2 = (float *)dalloc(sizeof(float) * qn->n_h2 * qn->n_out, qn->w2);
    dq.b2 = (float *)dalloc(sizeof(float) * qn->n_out, qn->b2);
    dqv = (float *)dalloc(sizeof(float) * nn * qn->n_out, nullptr);
    dact = (int *)dalloc(sizeof(int) * nn, nullptr);
  }
  if (!err.empty()) { cleanup(); return dfail(TTMPC_ERR_CUDA, err); }
  int rc = ttdqn_observe_act_device(lay, qn ? &dq : nullptr, n, dag, dxy, doff, dsol, dnp, dint, dold,
                                    dext, dqv, dact, dseg, dray, 0);
  if (rc) { cleanup(); return rc; }
  cudaError_t e = cudaDeviceSynchronize();
  auto back = [&](void *h, const void *d, size_t bytes) {
    if (h && d && e == cudaSuccess) e = cudaMemcpy(h, d, bytes, cudaMemcpyDeviceToHost);
  };
  back(h_ext, dext, sizeof(float) * nn * n_ext);
  back(h_seg, dseg, sizeof(double) * nn * ns);
  back(h_ray, dray, sizeof(double) * nn * ns);
  if (lay->use_memory) back(h_old_ext, dold, sizeof(float) * nn * 2 * ns);
  if (qn) { back(h_q, dqv, sizeof(float) * nn * qn->n_out); back(h_action, dact, sizeof(int) * nn); }
  cleanup();
  if (e != cudaSuccess) return dfail(TTMPC_ERR_CUDA, cudaGetErrorString(e));
  return TTMPC_OK;
}

extern "C" int ttdqn_internal_obs_device(int n, int max_nodes, int corner_samples, double sample_offset,
                                         double max_distance, const double *d_agent5, const double *d_path_xy,
                                         const int *d_path_n, float *d_internal, double *d_progress, void *stream) {
  if (n < 0 || max_nodes < 2 || corner_samples < 0 || !(max_distance > 0.0))
    return dfail(TTMPC_ERR_BAD_ARG, "internal_obs: n >= 0, max_nodes >= 2, corner_samples >= 0, max_distance > 0");
  if (n == 0) return TTMPC_OK;
  if (!d_agent5 || !d_path_xy || !d_path_n || !d_internal)
    return dfail(TTMPC_ERR_BAD_ARG, "internal_obs: agent, path and output pointers are required");
  ttdqn::internal_obs_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      n, max_nodes, corner_samples, sample_offset, max_distance, d_agent5, d_path_xy, d_path_n, d_internal, d_progress);
  DQN_TRY(cudaGetLastError());
  return TTMPC_OK;
}
extern "C" int ttdqn_rl_ref_device(int n, int steps, double ts, double ref_speed, const double *d_agent5,
                                   const int *d_action, double *d_rl_ref, void *stream) {
  if (n < 0 || steps < 1 || !(ts > 0.0)) return dfail(TTMPC_ERR_BAD_ARG, "rl_ref: n >= 0, steps >= 1, ts > 0");
  if (n == 0) return TTMPC_OK;
  if (!d_agent5 || !d_action || !d_rl_ref) return dfail(TTMPC_ERR_BAD_ARG, "rl_ref: null pointer");
  ttdqn::rl_ref_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(n, steps, ts, ref_speed, d_agent5, d_action, d_rl_ref);
  DQN_TRY(cudaGetLastError());
  return TTMPC_OK;
}
