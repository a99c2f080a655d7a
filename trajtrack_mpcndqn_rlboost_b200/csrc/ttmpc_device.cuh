// ttmpc_device.cuh -- device side of the batched NMPC planner (sm_100a).
//
// One WARP solves one scene; lane k owns horizon step k: its controls
// (v_k, w_k), every PANOC vector's two entries, the state s_{k+1}, and the
// k-th column of the obstacle tables.  The sequential unicycle rollout and its
// adjoint become warp prefix / suffix scans; every inner product is a butterfly
// all-reduce, so all solver control flow is warp-uniform.
//
// ARITHMETIC CONTRACT.  This file is compiled with -fmad=false: the only fused
// multiply-adds are the explicit fma() calls below, trigonometry is tt_sincos
// (Cody-Waite + fdlibm kernels, +,*,fma only), divisions and square roots are
// IEEE.  The CPU oracle (oracle/ttmpc_oracle.c, WARP ordering) performs the same
// operations in the same order, so a GPU solve is reproducible bit for bit on
// the host.  Change an expression here and the oracle's mirror must change too.
//
// Reference for the maths:
//   cost / constraints : /root/reference/src/mpc_traj_tracker/mpc/mpc_generator.py:155-283
//   dynamics           : /root/reference/src/pkg_motion_model/motion_model.py:153-176
//   solver             : OpEn (optimization_engine 0.7.x) PANOC + ALM/PM, as
//                        called at src/mpc_traj_tracker/trajectory_generator.py:284
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/ttmpc.h"

namespace ttmpc {

constexpr unsigned FULL = 0xffffffffu;
constexpr int MAX_MEM = 16;
constexpr int MAX_EDGE = 8;
constexpr int DYN_FIELDS = 10;  // per (obstacle, step): see stage_scene
// live dynamic obstacles whose table rows are kept in shared memory; the rest stay in the warp's global
// table.  One, not more: each further slot costs 1.6 KB per warp (default shapes), and 12 warps of the
// rolled build must fit the shared memory of an SM.
constexpr int DYN_SLOTS = 1;

struct DevCfg {
  int N, Nother, Nstc, ne, nstcobs, Ndyn, mem, max_inner, max_outer;
  int off_s, off_q, off_r, off_vref, off_c, off_os, off_od, off_qdyn, np;
  int smem_per_warp;  // bytes
  int warps_per_block;
  double ts, inv_ts, h6, veh_d2, margin;
  double vmin, vmax, wmax, amin, amax, awmax;
  double tol, init_tol, delta_tol, c0, pen_factor, tol_factor, suff_dec;
  unsigned long long max_ns;  // wall-clock budget of one scene [ns], 0 = none
};

// ---------------------------------------------------------------- sincos
// Cody-Waite reduction by pi/2 (three fma steps, exact products) and the fdlibm
// __kernel_sin / __kernel_cos minimax polynomials.  <= 1 ulp on |x| < 1e9.
__host__ __device__ __forceinline__ void tt_sincos(double x, double *s, double *c) {
  const double kd = rint(x * 6.36619772367581382433e-01);
  double r = fma(-kd, 1.5707963267948966e+00, x);
  r = fma(-kd, 6.123233995736766e-17, r);
  r = fma(-kd, -1.4973849048591698e-33, r);
  const int q = (int)((long long)kd & 3);
  const double z = r * r;
  double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
  ps = fma(z, ps, 2.75573137070700676789e-06);
  ps = fma(z, ps, -1.98412698298579493134e-04);
  ps = fma(z, ps, 8.33333333332248946124e-03);
  ps = fma(z, ps, -1.66666666666666324348e-01);
  const double sr = fma(r * z, ps, r);
  double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
  pc = fma(z, pc, -2.75573143513906633035e-07);
  pc = fma(z, pc, 2.48015872894767294178e-05);
  pc = fma(z, pc, -1.38888888888741095749e-03);
  pc = fma(z, pc, 4.16666666666666019037e-02);
  const double cr = fma(z * z, pc, fma(-0.5, z, 1.0));
  // quadrant fix-up without branches: q odd swaps, bit 1 of q / q+1 negates
  const bool swap = (q & 1) != 0;
  const double sb = swap ? cr : sr, cb = swap ? sr : cr;
  double so = (q & 2) ? -sb : sb, co = ((q + 1) & 2) ? -cb : cb;
  if (!(fabs(x) < 1.0e9)) { so = x * 0.0 + NAN; co = so; }  // huge / non-finite argument
  *s = so; *c = co;
}

// ---------------------------------------------------------------- atan2
// fdlibm's __ieee754_atan2 / atan (argument reduction by atan(1/2), atan(1), atan(3/2), atan(inf),
// 11-term odd minimax polynomial, hi/lo table of atan at the reduction points) with Horner in fma
// and one correction fdlibm lacks: the rounding error of y/x, fma(-t, x, y) / x, enters through
// d atan / dt = 1 / (1 + t^2).  <= 1 ulp.  CUDA's atan2 and glibc's differ from each other in the
// last bit; this one is the same function on the device and in the CPU oracle (ttmpc_oracle_atan2).
__host__ __device__ __forceinline__ double tt_atan_ratio(double ay, double ax) {  // atan(ay / ax), ay, ax > 0
  const double t = ay / ax;
  if (!(t <= 0x1p60)) return 1.57079632679489655800e+00;  // |y/x| > 2^60 (or overflow): pi/2
  if (t < 0x1p-27) return t;                               // atan(t) = t to the last bit
  const double e = fma(-t, ax, ay) / ax / fma(t, t, 1.0);  // (y/x - t) / (1 + t^2)
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
__host__ __device__ __forceinline__ double tt_atan2(double y, double x) {
  const double pi = 3.1415926535897931160e+00, pi_lo = 1.2246467991473531772e-16;
  if (x != x || y != y) return x + y;
  const double ax = fabs(x), ay = fabs(y);
  const bool xneg = signbit(x);
  double z;
  if (ay == 0.0) z = xneg ? pi : 0.0;                             // atan2(+-0, x)
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

// Same function for the hot path (eval_psi): the coefficients come from the constant bank, so
// every DFMA takes its constant as an operand.  With literals ptxas materialises each 64-bit
// constant with two UMOVs -- 28 of the 85 instructions of one inlined tt_sincos, three of them per
// evaluation.  Identical operations in identical order: bit-identical results.
static __constant__ double TT_SC[16] = {
    6.36619772367581382433e-01, 1.5707963267948966e+00, 6.123233995736766e-17, -1.4973849048591698e-33,
    1.58969099521155010221e-10, -2.50507602534068634195e-08, 2.75573137070700676789e-06,
    -1.98412698298579493134e-04, 8.33333333332248946124e-03, -1.66666666666666324348e-01,
    -1.13596475577881948265e-11, 2.08757232129817482790e-09, -2.75573143513906633035e-07,
    2.48015872894767294178e-05, -1.38888888888741095749e-03, 4.16666666666666019037e-02};
__device__ __forceinline__ void tt_sincos_c(double x, double *s, double *c) {
  const double kd = rint(x * TT_SC[0]);
  double r = fma(-kd, TT_SC[1], x);
  r = fma(-kd, TT_SC[2], r);
  r = fma(-kd, TT_SC[3], r);
  const int q = (int)((long long)kd & 3);
  const double z = r * r;
  double ps = fma(z, TT_SC[4], TT_SC[5]);
  ps = fma(z, ps, TT_SC[6]);
  ps = fma(z, ps, TT_SC[7]);
  ps = fma(z, ps, TT_SC[8]);
  ps = fma(z, ps, TT_SC[9]);
  const double sr = fma(r * z, ps, r);
  double pc = fma(z, TT_SC[10], TT_SC[11]);
  pc = fma(z, pc, TT_SC[12]);
  pc = fma(z, pc, TT_SC[13]);
  pc = fma(z, pc, TT_SC[14]);
  pc = fma(z, pc, TT_SC[15]);
  const double cr = fma(z * z, pc, fma(-0.5, z, 1.0));
  const bool swap = (q & 1) != 0;
  const double sb = swap ? cr : sr, cb = swap ? sr : cr;
  double so = (q & 2) ? -sb : sb, co = ((q + 1) & 2) ? -cb : cb;
  if (!(fabs(x) < 1.0e9)) { so = x * 0.0 + NAN; co = so; }  // huge / non-finite argument
  *s = so; *c = co;
}

// IEEE division / square root: ~15 inlined instructions per use (MUFU seed, Newton steps, range
// check, slow-path call) and the PANOC step has a dozen of them, so they are out of line: one
// shared copy keeps the hot loop inside the instruction cache (DESIGN.md section 6)
static __device__ __noinline__ double tt_div(double a, double b) { return a / b; }
static __device__ __noinline__ double tt_sqrt(double a) { return sqrt(a); }

// ---------------------------------------------------------------- warp utils
// Hand-written shuffle primitives.  Round 1 left these to the compiler as rolled loops in
// __noinline__ functions to save instruction-cache bytes; the SASS of one rolled scan level was
// 20 instructions for two doubles (4 SHFL + 4 MOV + 2 DADD + 4 FSEL + loop / divergence-check
// overhead) and the moves in and out of the reduction functions were 15 % of all executed
// instructions (profiles/r2_*).  The versions below issue fewer instructions AND are not longer:
//  * scans use the shuffle's own "source lane in range" predicate to gate the add (no compare);
//  * all-reduces of several values do a reduce-scatter over the first levels (lanes keep half of
//    the values, send the other half), a butterfly over the rest and an all-gather: 10 double
//    shuffles instead of 20 for four values.  Every value still goes through the SAME addition
//    tree as in a plain xor-butterfly (x + y == y + x bit for bit), so results are unchanged and
//    the CPU oracle's w_sum() mirror stays valid.
template <int O>
__device__ __forceinline__ void up_add(double &v) {  // v += v[lane - O] on lanes >= O
  asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 lo, hi, tl, th;\n\t.reg .f64 t;\n\t"
               "mov.b64 {lo, hi}, %0;\n\t"
               "shfl.sync.up.b32 tl|p, lo, %1, 0, 0xffffffff;\n\t"
               "shfl.sync.up.b32 th, hi, %1, 0, 0xffffffff;\n\t"
               "mov.b64 t, {tl, th};\n\t"
               "@p add.rn.f64 %0, %0, t;\n\t}"
               : "+d"(v) : "n"(O));
}
template <int O>
__device__ __forceinline__ void down_add(double &v) {  // v += v[lane + O] on lanes < 32 - O
  asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 lo, hi, tl, th;\n\t.reg .f64 t;\n\t"
               "mov.b64 {lo, hi}, %0;\n\t"
               "shfl.sync.down.b32 tl|p, lo, %1, 31, 0xffffffff;\n\t"
               "shfl.sync.down.b32 th, hi, %1, 31, 0xffffffff;\n\t"
               "mov.b64 t, {tl, th};\n\t"
               "@p add.rn.f64 %0, %0, t;\n\t}"
               : "+d"(v) : "n"(O));
}
// inclusive prefix sum over lanes (Kogge-Stone)
__device__ __forceinline__ double wscan(double v, int) {
  up_add<1>(v); up_add<2>(v); up_add<4>(v); up_add<8>(v); up_add<16>(v);
  return v;
}
__device__ __forceinline__ void wscan2(double &a, double &b) {  // two scans, interleaved
  up_add<1>(a); up_add<1>(b); up_add<2>(a); up_add<2>(b); up_add<4>(a); up_add<4>(b);
  up_add<8>(a); up_add<8>(b); up_add<16>(a); up_add<16>(b);
}
// inclusive suffix sum over lanes
__device__ __forceinline__ double wsuffix(double v, int) {
  down_add<1>(v); down_add<2>(v); down_add<4>(v); down_add<8>(v); down_add<16>(v);
  return v;
}
__device__ __forceinline__ void wsuffix2(double &a, double &b) {
  down_add<1>(a); down_add<1>(b); down_add<2>(a); down_add<2>(b); down_add<4>(a); down_add<4>(b);
  down_add<8>(a); down_add<8>(b); down_add<16>(a); down_add<16>(b);
}
// v + v[lane ^ O] (the 64-bit shuffle intrinsic costs two extra moves per use)
template <int O>
__device__ __forceinline__ double xor_get(double v) {
  double t;
  asm volatile("{\n\t.reg .b32 lo, hi, tl, th;\n\t"
               "mov.b64 {lo, hi}, %1;\n\t"
               "shfl.sync.bfly.b32 tl, lo, %2, 31, 0xffffffff;\n\t"
               "shfl.sync.bfly.b32 th, hi, %2, 31, 0xffffffff;\n\t"
               "mov.b64 %0, {tl, th};\n\t}"
               : "=d"(t) : "d"(v), "n"(O));
  return t;
}
// all-reduce of one value: xor-butterfly, offsets 16 .. 1
__device__ __forceinline__ double wsum_inl(double v) {
  v += xor_get<16>(v); v += xor_get<8>(v); v += xor_get<4>(v); v += xor_get<2>(v); v += xor_get<1>(v);
  return v;
}
static __device__ __noinline__ double wsum(double v) { return wsum_inl(v); }
// all-reduce of four values: 10 double shuffles instead of 20
__device__ __forceinline__ void wsum4_inl(double &a, double &b, double &c, double &d, int lane) {
  const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0;
  double x = b4 ? c : a, y = b4 ? d : b;
  const double sx = b4 ? a : c, sy = b4 ? b : d;
  x += xor_get<16>(sx); y += xor_get<16>(sy);
  double z = b3 ? y : x;
  const double sz = b3 ? x : y;
  z += xor_get<8>(sz);
  z += xor_get<4>(z); z += xor_get<2>(z); z += xor_get<1>(z);
  a = __shfl_sync(FULL, z, 0); b = __shfl_sync(FULL, z, 8);
  c = __shfl_sync(FULL, z, 16); d = __shfl_sync(FULL, z, 24);
}
struct D4 { double a, b, c, d; };
// ONE out-of-line copy serves every 2-, 3- and 4-value all-reduce of the solve (unused slots carry
// zeros; each value goes through its own butterfly tree, so the zeros change nothing)
static __device__ __noinline__ D4 wsum4v(double a, double b, double c, double d) {
  wsum4_inl(a, b, c, d, threadIdx.x & 31);
  D4 r; r.a = a; r.b = b; r.c = c; r.d = d;
  return r;
}
__device__ __forceinline__ void wsum4(double &a, double &b, double &c, double &d, int) {
  const D4 r = wsum4v(a, b, c, d);
  a = r.a; b = r.b; c = r.c; d = r.d;
}
__device__ __forceinline__ void wsum2(double &a, double &b) {
  const D4 r = wsum4v(a, b, 0.0, 0.0);
  a = r.a; b = r.b;
}
__device__ __forceinline__ void wsum3(double &a, double &b, double &c) {
  const D4 r = wsum4v(a, b, c, 0.0);
  a = r.a; b = r.b; c = r.c;
}
__device__ __forceinline__ double clipd_ref(double z, double lo, double hi) {
  return fmin(fmax(z, lo), hi);
}
// Compare + select on doubles.  sm_100 has no DMNMX: fmax/fmin (and the C ternaries the
// compiler canonicalises to them) expand to ~9 instructions each with NaN quieting.  A
// setp/selp pair written in PTX stays 1 DSETP + 2 FSEL.  Semantics used below: the result is
// `x` only when the comparison is TRUE, so NaN inputs fall to the constant, exactly like
// fmax(x, 0) / fmin(., 1) do.
__device__ __forceinline__ double sel_gt(double a, double b, double x, double y) {  // a > b ? x : y
  double r;
  asm("{\n\t.reg .pred p;\n\tsetp.gt.f64 p, %1, %2;\n\tselp.f64 %0, %3, %4, p;\n\t}"
      : "=d"(r) : "d"(a), "d"(b), "d"(x), "d"(y));
  return r;
}
__device__ __forceinline__ double sel_lt(double a, double b, double x, double y) {  // a < b ? x : y
  double r;
  asm("{\n\t.reg .pred p;\n\tsetp.lt.f64 p, %1, %2;\n\tselp.f64 %0, %3, %4, p;\n\t}"
      : "=d"(r) : "d"(a), "d"(b), "d"(x), "d"(y));
  return r;
}
// fmin(fmax(z, lo), hi) for every input (NaN -> lo), 6 instructions
__device__ __forceinline__ double clipd(double z, double lo, double hi) {
  const double t = sel_gt(z, lo, z, lo);
  return sel_lt(t, hi, t, hi);
}
__device__ __forceinline__ double relu(double x) { return sel_gt(x, 0.0, x, 0.0); }
__device__ __forceinline__ double clamp01(double x) {
  const double t = sel_gt(x, 0.0, x, 0.0);
  return sel_lt(t, 1.0, t, 1.0);
}
// per-lane share of an inner product of two lane-distributed vectors
__device__ __forceinline__ double pdot(double a0, double a1, double b0, double b1) {
  return fma(a1, b1, a0 * b0);
}

// ---------------------------------------------------------------- per-warp state
// Everything a warp needs that is uniform across lanes lives in shared memory
// (broadcast reads), so the eval routine can be a real (non-inlined) function.
// PANOC scalars of the solve kernel (ttmpc_solve.cu) that are read a few times per iteration, away from the
// dependent chain of the line search: warp-uniform, kept in the warp's context rather than in registers.
struct PanocCold {
  double L, sigma, lb_gamma;
  double ip;              // <grad, fpr>, reduced together with |fpr|^2
  double env_dd, env_g2;  // |gstep - u_half|^2 and |grad|^2 of the current gradient step / half step: from the
                          // accepted line-search evaluation, or formed where the solver takes the step itself
  double tau;             // line-search step of the current candidate
  double rhs_ls;          // right-hand side of the line search's envelope test
  int iteration;          // PANOC steps taken in this inner solve
  int lb_active, lb_head, lb_first;  // L-BFGS ring: pairs held, newest slot, no pair yet
};
// The L-BFGS state panoc_step saves before it updates L-BFGS speculatively (tail helpers) and restores
// when the speculation is lost.
struct SpecSave {
  double lb_gamma;
  int lb_first, lb_head, lb_active;
};
struct WarpCtx {
  const double *p;   // this scene's packed parameter vector (global)
  double *dyn;       // this warp's dynamic-obstacle table (global scratch, L2 resident)
  double x0, y0, th0, xg, yg, thg, v_init, w_init;
  double qvel, rv, rw, qN, qthetaN, qrpd, acc_pen, wacc_pen;
  long long n_cost, n_grad, n_body;  // evaluation counters (lane 0 view)
  int nstc_active;                   // static obstacles that can ever be non-zero
  float fleet_thr;                   // fp32 contact prefilter threshold (padded d^2)
  // box-guarded compaction: obstacles / robots whose bounding circles never meet the box
  // |p - start|_inf < box_half are skipped while every rolled-out position stays in the box
  double box_half;
  unsigned long long dyn_live;       // bit j: dynamic obstacle j can matter inside the box
  unsigned fleet_live;               // bit j: other robot j can matter inside the box
  double lipc;                       // PANOC: GAMMA_L_COEFF / (2 gamma) of the current gamma
  double icm_c, icm;                 // 1 / max(c, 1) of the last penalty c this warp evaluated with
  // solve_scene's outer-loop (ALM) state: warp-uniform, changes once per outer iteration and is live
  // across every evaluation of the inner loop.  Kept here, not in registers, so that the rolled build
  // fits 168 registers per thread (12 resident scenes per SM) without spilling.
  PanocCold pc;
  SpecSave spec;
  double akkt_tol, f_final, last_fpr, dy_norm, dy_norm_plus, f2_norm, f2_norm_plus;
  unsigned long long t_start, panoc_iters;
  int inner_count, exit_status, num_outer, scene, in_time;
};

struct HelpHdr;
struct WarpSmem {
  WarpCtx *ctx;
  double *seg;    // [N][6]: s1x s1y | sx sy | inv_den pad  (three vector loads per segment)
  double *os;     // [Nstc*nstcobs] per obstacle: b[ne], -a0[ne], -a1[ne]
  double *D;      // [Ndyn] per-obstacle hard sums of the last evaluation
  double *vref;   // [N] speed reference
  float2 *fleet;  // [Nother][N] other robots' (x, y), fp32 copy for the contact prefilter
  float *dynb;    // [Ndyn][N][3] conservative fp32 bounding test: cx cy R2
  double *dynt;   // [DYN_SLOTS][DYN_FIELDS][N] table rows of the first live dynamic obstacles
  double2 *lbs;   // [(mem+1)][N]  L-BFGS s rows (lane k reads element k of a row: no bank conflict)
  double2 *lby;   // [(mem+1)][N]  L-BFGS y rows
  double *rho;    // [mem+1]
  double2 *gprev; // [N] previous gradient of the PANOC iteration (AKKT residual); lanes >= N: zero
  double2 *olds;  // [32] L-BFGS old_state of every lane (lanes >= N included: their entries need not be zero)
  double2 *oldg;  // [32] L-BFGS old_g
  // mailbox of the tail helpers (see ttmpc_solve.cu): the owner's request / the helper's answer
  double2 *hreq;  // [N] evaluation point (v, w)
  double2 *hres;  // [N] gradient (gv, gw): the same row as hreq
  double2 *yrow;  // [N] the owner's current multipliers (ya, yw)
  struct HelpHdr *hhdr;
};
struct HelpHdr {
  int state;        // 0 idle, 1 request posted, 2 result ready
  int grad;         // request: gradient wanted
  double c, gamma_ls;
  double psi, f, f2sq, S, dd, g2;  // result
};

// Compile-time problem dimensions (0 = take the value from DevCfg at run time).
// The default configuration (config/mpc_default.yaml) gets a fully specialised kernel.
__device__ __forceinline__ int first_bit(unsigned m) { return __ffs((int)m) - 1; }
__device__ __forceinline__ int first_bit(unsigned long long m) { return __ffsll((long long)m) - 1; }
__device__ __forceinline__ int pop_bits(unsigned m) { return __popc(m); }
__device__ __forceinline__ int pop_bits(unsigned long long m) { return __popcll(m); }
template <bool WIDE> struct DynMask { using type = unsigned long long; };
template <> struct DynMask<false> { using type = unsigned; };

template <int N_, int NO_, int NS_, int NE_, int ND_, int MEM_ = 0>
struct Dims {
  // bit mask over the dynamic obstacles: 32 bits when the compile-time count allows (64-bit
  // find-first-set / shifts are ~10 instructions each on sm_100)
  using dmask = typename DynMask<(N_ == 0 || ND_ > 32)>::type;
  static constexpr int kN = N_, kNstc = NS_;
  // unroll factor of the static-obstacle loop in eval_psi (see Rolled)
  static constexpr int kStaticUnroll = 4;
  __device__ __forceinline__ static int mem(const DevCfg &g) { return N_ ? MEM_ : g.mem; }
  __device__ __forceinline__ static int N(const DevCfg &g) { return N_ ? N_ : g.N; }
  __device__ __forceinline__ static int Nother(const DevCfg &g) { return N_ ? NO_ : g.Nother; }
  __device__ __forceinline__ static int Nstc(const DevCfg &g) { return N_ ? NS_ : g.Nstc; }
  __device__ __forceinline__ static int ne(const DevCfg &g) { return N_ ? NE_ : g.ne; }
  __device__ __forceinline__ static int Ndyn(const DevCfg &g) { return N_ ? ND_ : g.Ndyn; }
};
using DimsRuntime = Dims<0, 0, 0, 0, 0>;
using DimsDefault = Dims<20, 10, 10, 4, 15, 10>;
// The same dimensions with the static-obstacle loop rolled: the code of solve_kernel_small.  The
// kernel is bound by instruction-cache refills (DESIGN.md section 6), so an unroll factor trades
// dependent-issue latency against code bytes; with 12 warps per SM at different places of the loop,
// the smaller loop body wins.  Same arithmetic in the same order: bit-identical results.
template <class DM>
struct Rolled : DM {
  static constexpr int kStaticUnroll = 1;
};

__host__ __device__ inline int smem_bytes_per_warp(int N, int Nother, int Nstc, int nstcobs, int Ndyn,
                                                   int mem) {
  size_t b = 0;
  b += (sizeof(WarpCtx) + 15) / 16 * 16;
  b += sizeof(double) * 6 * N;
  b += sizeof(double) * ((Nstc * nstcobs + 1) / 2 * 2);
  b += sizeof(double) * ((Ndyn + 1) / 2 * 2);
  b += sizeof(double) * ((N + 1) / 2 * 2);
  b += (sizeof(float2) * (size_t)Nother * N + 15) / 16 * 16;
  b += (sizeof(float) * 3 * (size_t)Ndyn * N + 15) / 16 * 16;
  b += sizeof(double) * (size_t)(Ndyn ? DYN_SLOTS * DYN_FIELDS * N : 0);
  b += sizeof(double2) * (size_t)(mem + 1) * N * 2;
  b += sizeof(double) * ((mem + 2) / 2 * 2);
  b += sizeof(double2) * ((size_t)N + 64);
  b += sizeof(double2) * 2 * (size_t)N + (sizeof(HelpHdr) + 15) / 16 * 16;  // mailbox rows + header
  return (int)((b + 15) / 16 * 16);
}

// With compile-time dimensions (DimsDefault) every offset folds into the load / store
// immediates: one base register instead of ~20 pointers and their address arithmetic.
template <class DM>
__device__ __forceinline__ WarpSmem carve(unsigned char *base, const DevCfg &g) {
  WarpSmem w;
  unsigned char *q = base;
  const int N = DM::N(g), MEM = DM::mem(g), Nother = DM::Nother(g), Nstc = DM::Nstc(g),
            nstcobs = 3 * DM::ne(g), Ndyn = DM::Ndyn(g);
  w.ctx = reinterpret_cast<WarpCtx *>(q); q += (sizeof(WarpCtx) + 15) / 16 * 16;
  w.lbs = reinterpret_cast<double2 *>(q); q += sizeof(double2) * (size_t)(MEM + 1) * N;
  w.lby = reinterpret_cast<double2 *>(q); q += sizeof(double2) * (size_t)(MEM + 1) * N;
  w.fleet = reinterpret_cast<float2 *>(q); q += (sizeof(float2) * (size_t)Nother * N + 15) / 16 * 16;
  w.dynb = reinterpret_cast<float *>(q); q += (sizeof(float) * 3 * (size_t)Ndyn * N + 15) / 16 * 16;
  w.dynt = reinterpret_cast<double *>(q); q += sizeof(double) * (size_t)(Ndyn ? DYN_SLOTS * DYN_FIELDS * N : 0);
  w.seg = reinterpret_cast<double *>(q); q += sizeof(double) * 6 * N;
  w.os = reinterpret_cast<double *>(q); q += sizeof(double) * ((Nstc * nstcobs + 1) / 2 * 2);
  w.D = reinterpret_cast<double *>(q); q += sizeof(double) * ((Ndyn + 1) / 2 * 2);
  w.vref = reinterpret_cast<double *>(q); q += sizeof(double) * ((N + 1) / 2 * 2);
  w.rho = reinterpret_cast<double *>(q); q += sizeof(double) * ((MEM + 2) / 2 * 2);
  w.gprev = reinterpret_cast<double2 *>(q); q += sizeof(double2) * (size_t)N;
  w.olds = reinterpret_cast<double2 *>(q); q += sizeof(double2) * 32;
  w.oldg = reinterpret_cast<double2 *>(q); q += sizeof(double2) * 32;
  // the answer overwrites the request: the helper reads the point before it evaluates, and the owner
  // posts the next request only after it has collected the answer
  w.hreq = reinterpret_cast<double2 *>(q); q += sizeof(double2) * (size_t)N;
  w.hres = w.hreq;
  w.yrow = reinterpret_cast<double2 *>(q); q += sizeof(double2) * (size_t)N;
  w.hhdr = reinterpret_cast<HelpHdr *>(q);
  return w;
}

// Dynamic-obstacle table, field-major so that lane k reads element [f][j][k]
// coalesced.  Built once per solve from the raw (cx cy rx ry angle alpha) records
// (mpc_generator.py:225-237): the sincos and the four divisions leave the hot loop.
//   0 cx  1 cy  2 R2 (rejection radius^2)  3 cos  4 sin
//   5 1/(rx+1e-6)^2  6 1/(ry+1e-6)^2  7 1/(rx+m+1e-6)^2  8 1/(ry+m+1e-6)^2  9 alpha*qdyn[k]
__device__ __forceinline__ double &dynf(double *t, const DevCfg &g, int f, int j, int k) {
  return t[((size_t)f * g.Ndyn + j) * g.N + k];
}

// Row of obstacle j's table for this lane's column: shared memory for the first DYN_SLOTS live
// obstacles, the warp's global scratch otherwise.  field f of the row = p[f * sf].
struct DynRow { const double *p; int sf; };
template <class M>
__device__ __forceinline__ DynRow dyn_row(const WarpSmem &sm, const WarpCtx *cx, int j, int N, int Ndyn, int lk) {
  const M live = (M)cx->dyn_live;
  const int slot = pop_bits((M)(live & (((M)1 << j) - (M)1)));
  const bool in_s = (live >> j & (M)1) != (M)0 && slot < DYN_SLOTS;
  DynRow r;
  r.p = in_s ? sm.dynt + (size_t)slot * DYN_FIELDS * N + lk : cx->dyn + (size_t)j * N + lk;
  r.sf = in_s ? N : Ndyn * N;
  return r;
}

// Staging, part 1: everything before the dynamic-obstacle block.  `p` points at a copy of the
// row prefix [0, off_od) (shared-memory copy made by the bulk copy below, or the row itself).
__device__ inline void stage_part1(const DevCfg &g, const WarpSmem &sm, const double *p, const double *p_global,
                                   double *dyn_scratch, int lane) {
  WarpCtx *c = sm.ctx;
  if (lane == 0) {
    const double *s = p + g.off_s, *q = p + g.off_q;
    c->p = p_global; c->dyn = dyn_scratch;
    c->x0 = s[0]; c->y0 = s[1]; c->th0 = s[2];
    c->xg = s[3]; c->yg = s[4]; c->thg = s[5];
    c->v_init = s[6]; c->w_init = s[7];
    c->qvel = q[1]; c->rv = q[3]; c->rw = q[4]; c->qN = q[5]; c->qthetaN = q[6];
    c->qrpd = q[7]; c->acc_pen = q[8]; c->wacc_pen = q[9];
    c->n_cost = 0; c->n_grad = 0; c->n_body = 0;
    c->lipc = 0.0; c->icm_c = NAN; c->icm = 0.0;  // NaN never compares equal: the first evaluation fills the pair
  }
  // reference-path segments: path_ref has N+1 points, last duplicated (l.190-191)
  const double *r = p + g.off_r;
  for (int j = lane; j < g.N; j += 32) {
    int j2 = (j + 1 < g.N) ? j + 1 : g.N - 1;
    double s1x = r[3 * j], s1y = r[3 * j + 1];
    double sx = r[3 * j2] - s1x, sy = r[3 * j2 + 1] - s1y;
    double den = fma(sy, sy, sx * sx) + 1e-16;
    sm.seg[6 * j + 0] = s1x; sm.seg[6 * j + 1] = s1y;
    sm.seg[6 * j + 2] = sx;  sm.seg[6 * j + 3] = sy;
    sm.seg[6 * j + 4] = 1.0 / den; sm.seg[6 * j + 5] = 0.0;
  }
  // static half-spaces: keep b, store -a0 and -a1 (res = b + (-a0) x + (-a1) y).
  // An obstacle with an edge a0 = a1 = 0, b <= 0 (e.g. a zero-padded slot) has
  // max(0, res) = 0 on that edge for every position, so its product is exactly 0:
  // such obstacles are dropped here (same order for the rest), which changes no result.
  const double *os = p + g.off_os;
  {
    int n_act = 0;
    for (int i0 = 0; i0 < g.Nstc; i0 += 32) {
      const int i = i0 + lane;
      bool live = false;
      if (i < g.Nstc) {
        live = true;
        const double *b = os + i * g.nstcobs, *a0 = b + g.ne, *a1 = b + 2 * g.ne;
        for (int e = 0; e < g.ne; e++)
          if (a0[e] == 0.0 && a1[e] == 0.0 && !(b[e] > 0.0)) live = false;
      }
      const unsigned m = __ballot_sync(FULL, live);
      if (live) {
        const int slot = n_act + __popc(m & ((1u << lane) - 1u));
        const double *src = os + i * g.nstcobs;
        double *dst = sm.os + slot * g.nstcobs;
        for (int e = 0; e < g.nstcobs; e++) dst[e] = (e < g.ne) ? src[e] : -src[e];
      }
      n_act += __popc(m);
    }
    if (lane == 0) c->nstc_active = n_act;
  }
  for (int k = lane; k < g.N; k += 32) sm.vref[k] = p[g.off_vref + k];
  // other robots: c is robot-major, (x y theta) per step (mpc_generator.py:207-209)
  const double *cpar = p + g.off_c;
  for (int t = lane; t < g.Nother * g.N; t += 32)
    sm.fleet[t] = make_float2((float)cpar[(size_t)t * 3], (float)cpar[(size_t)t * 3 + 1]);
  // contact needs |p - o|^2 < d^2; the fp32 prefilter pads d by the worst rounding of the
  // fp32 copies (8 ulp_f32 of the largest coordinate of this scene) so it never rejects a contact
  double cmax = 0.0;
  bool cnan = false;
  for (int t = lane; t < g.Nother * g.N; t += 32) {
    const double ax = fabs(cpar[(size_t)t * 3]), ay = fabs(cpar[(size_t)t * 3 + 1]);
    cnan = cnan || !(ax == ax) || !(ay == ay);
    cmax = fmax(cmax, fmax(ax, ay));
  }
  for (int o = 16; o > 0; o >>= 1) cmax = fmax(cmax, __shfl_xor_sync(FULL, cmax, o));
  cnan = __any_sync(FULL, cnan);
  if (lane == 0) {
    if (cnan) cmax = NAN;
    const double d = sqrt(g.veh_d2), pad = 4.8e-7 * (2.0 * cmax + 2.0 * d + 1.0) + 1e-6;
    float thr = __double2float_ru((d + pad) * (d + pad) * (1.0 + 1e-6));
    if (!(cmax == cmax)) thr = INFINITY;  // NaN coordinates: let the exact test decide
    c->fleet_thr = thr;
  }
  // live mask of the box-guarded compaction, other robots (NaN / inf coordinates stay live)
  {
    const double x0 = p[g.off_s], y0 = p[g.off_s + 1];
    const double vm = fmax(fabs(g.vmax), fabs(g.vmin));
    const double bh = 2.0 * g.N * g.ts * vm + 1.0;
    unsigned fl = 0;
    const double dveh = sqrt(g.veh_d2) * 1.001 + 1e-3;
    for (int t = lane; t < g.Nother * g.N; t += 32) {
      const int j = t / g.N;
      const bool outside = fabs(cpar[(size_t)t * 3] - x0) > bh + dveh || fabs(cpar[(size_t)t * 3 + 1] - y0) > bh + dveh;
      if (!outside) fl |= 1u << j;
    }
    fl = __reduce_or_sync(FULL, fl);
    if (lane == 0) { c->box_half = bh; c->fleet_live = fl; }
  }
  __syncwarp();
}

// Staging, part 2: the dynamic-obstacle table.  od = the o_d block, qdyn = the q_dyn block.
__device__ inline void stage_part2(const DevCfg &g, const WarpSmem &sm, const double *od, const double *qdyn,
                                   double *dyn_scratch, int lane) {
  WarpCtx *c = sm.ctx;
  const int npair = g.Ndyn * g.N;
  // live mask of the box-guarded compaction, dynamic obstacles (NaN / inf coordinates stay live)
  unsigned long long live;
  {
    const double x0 = c->x0, y0 = c->y0;
    const double bh = c->box_half;
    unsigned long long dl = 0;
    for (int t = lane; t < npair; t += 32) {
      const int j = t / g.N;
      const double *e = od + (size_t)t * 6;
      const double rmax = fmax(fmax(fabs(e[2] + 1e-6), fabs(e[3] + 1e-6)),
                               fmax(fabs(e[2] + g.margin + 1e-6), fabs(e[3] + g.margin + 1e-6))) * 1.001 + 1e-3;
      const bool outside = fabs(e[0] - x0) > bh + rmax || fabs(e[1] - y0) > bh + rmax;
      if (!outside) dl |= 1ull << j;
    }
    const unsigned dlo = __reduce_or_sync(FULL, (unsigned)dl), dhi = __reduce_or_sync(FULL, (unsigned)(dl >> 32));
    live = ((unsigned long long)dhi << 32) | dlo;
    if (lane == 0) c->dyn_live = live;
  }
  for (int t = lane; t < npair; t += 32) {
    int j = t / g.N, k = t - j * g.N;
    const double *e = od + (size_t)t * 6;  // obstacle-major, then step: contiguous records
    double cx = e[0], cy = e[1], rx = e[2], ry = e[3], ang = e[4], alpha = e[5];
    double sa, ca;
    tt_sincos(ang, &sa, &ca);
    double Rx = rx + 1e-6, Ry = ry + 1e-6;
    double Rxm = rx + g.margin + 1e-6, Rym = ry + g.margin + 1e-6;
    double rmax = fmax(fmax(fabs(Rx), fabs(Ry)), fmax(fabs(Rxm), fabs(Rym)));
    double f[DYN_FIELDS];
    f[0] = cx; f[1] = cy; f[2] = rmax * rmax * (1.0 + 1e-9); f[3] = ca; f[4] = sa;
    f[5] = 1.0 / (Rx * Rx); f[6] = 1.0 / (Ry * Ry); f[7] = 1.0 / (Rxm * Rxm); f[8] = 1.0 / (Rym * Rym);
    f[9] = alpha * qdyn[k];
#pragma unroll
    for (int q = 0; q < DYN_FIELDS; q++) dynf(dyn_scratch, g, q, j, k) = f[q];
    // the first DYN_SLOTS live obstacles also get their rows in shared memory (eval_psi reads them
    // there: the obstacles a scene actually meets are few, their rows are read in every evaluation)
    {
      const int slot = __popcll(live & ((1ull << j) - 1ull));
      if ((live >> j & 1ull) && slot < DYN_SLOTS) {
#pragma unroll
        for (int q = 0; q < DYN_FIELDS; q++) sm.dynt[((size_t)slot * DYN_FIELDS + q) * g.N + k] = f[q];
      }
    }
    // conservative fp32 copy of the bounding test: the radius is padded by the worst
    // rounding of the fp32 centre / position (8 ulp_f32 of the coordinates) so a pair the
    // exact fp64 test accepts is never rejected here; rejected pairs contribute exactly 0
    {
      const double pad = 4.8e-7 * (fabs(cx) + fabs(cy) + 2.0 * rmax + 1.0) + 1e-6;
      const double rp = rmax + pad;
      float r2f = __double2float_ru(rp * rp * (1.0 + 1e-6));
      if (!(rmax == rmax) || !(cx == cx) || !(cy == cy)) r2f = 0.0f;  // NaN input: exact test is false too
      sm.dynb[3 * t] = (float)cx; sm.dynb[3 * t + 1] = (float)cy; sm.dynb[3 * t + 2] = r2f;
    }
  }
  __syncwarp();
}

// Staging = part 1 + part 2, straight from the scene's row of the parameter block (read once;
// ~35 us per scene, 1 % of an average solve: measured in round 1 with a cycle-counting build of the
// kernel, since removed; DESIGN.md section 6).
// A cp.async.bulk landing zone in the (then empty) L-BFGS ring was tried and dropped: part 2 is
// bound by its 300 sincos + 1200 divisions, not by the loads, and its 14.4 KB block does not fit the ring.
__device__ inline void stage_scene(const DevCfg &g, const WarpSmem &sm, const double *p,
                                   double *dyn_scratch, int lane) {
  stage_part1(g, sm, p, p, dyn_scratch, lane);
  stage_part2(g, sm, p + g.off_od, p + g.off_qdyn, dyn_scratch, lane);
}

// ---------------------------------------------------------------- evaluation
struct EvalOut {
  double psi;   // f + c/2 dist^2_C(F1 + y/max(c,1)) + c/2 |F2|^2
  double f;     // original cost (psi at c = 0)
  double f2sq;  // |F2|^2
  double S;     // static hard sum (F2_j = S + D_j, D in smem when any_hard, else 0)
  double gv, gw;  // this lane's gradient entries (GRAD only)
  // line-search fusion (GRAD and gamma_ls > 0): gradient step s = p - gamma*grad, half step
  // h = proj(s), and the two reduced scalars of the forward-backward envelope
  double h0, h1, dd, g2;
  bool any_hard;
};

// 1 / max(c, 1) for a penalty this warp has not evaluated with yet (see eval_psi); `store` = the calling warp
// owns the context
static __device__ __noinline__ double icm_miss(double c, WarpCtx *ctx, bool store) {
  const double icm = 1.0 / fmax(c, 1.0);
  if (store) {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) { ctx->icm = icm; ctx->icm_c = c; }
    __syncwarp();
  }
  return icm;
}

// Evaluate psi (and its gradient when GRAD) at this lane's (v, w).
// ya / yw are this lane's multipliers for the linear / angular acceleration rows.
// DM carries the problem dimensions (compile-time for the default configuration).
// GRAD is a run-time (warp-uniform) flag: one copy of the code serves both uses, which
// keeps the hot loop inside the instruction cache.
//
// Lanes >= N carry v = w = 0, so their state equals lane N-1's; they run the same
// instruction stream on lane N-1's table columns (no divergence regions) and their
// contributions are zeroed before the reductions.  Rare events (fleet contact, inside a
// static polygon, inside an ellipse's bounding circle) are entered through warp votes, so
// the common path has no divergent branch at all.
template <class DM>
__device__ __noinline__ EvalOut eval_psi(const DevCfg *gp, unsigned char *smem_base, double v_in,
                                         double w_in, double c, double ya, double yw,
                                         double *st_out, const bool GRAD, const double gamma_ls,
                                         double *Dalt = nullptr) {
  // Dalt: a helper warp evaluating on another warp's scene tables brings its own scratch for
  // the per-obstacle hard sums (and does not touch the owner's counters)
  const DevCfg &g = *gp;
  const WarpSmem sm = carve<DM>(smem_base, g);
  double *const Dv = Dalt ? Dalt : sm.D;
  const int lane = threadIdx.x & 31;
  const double v = lane < DM::N(g) ? v_in : 0.0, w = lane < DM::N(g) ? w_in : 0.0;
  const WarpCtx *cx = sm.ctx;
  const int N = DM::N(g), Nother = DM::Nother(g), Nstc = cx->nstc_active, ne = DM::ne(g),
            Ndyn = DM::Ndyn(g);
  const int nstcobs = 3 * ne;
  const bool act = lane < N;
  const int lk = act ? lane : N - 1;  // table column this lane reads
  const double ts = g.ts;

  // ---- terms of (v, w) alone: speed reference + control action (l.203-204), accelerations and the ALM
  //      distance (l.250-264).  Formed HERE, ahead of the rollout: the kernel runs two warps per scheduler
  //      and its top stall is the fixed-latency dependency wait, and the rollout that follows is one long
  //      chain (theta scan -> sincos -> position scan); in the same basic block these ~60 independent
  //      instructions fill its bubbles (+3 % solves/s, round 2).  They are ADDED to the cost at their
  //      original places below, so every accumulation keeps its order and the bits do not change.
  // 1 / max(c, 1): c changes once per outer iteration, the division (an out-of-line call, with the NaN-aware
  // fmax ~55 executed instructions, 4 % of an evaluation) ran in every evaluation.  The warp that owns the
  // scene keeps the last (c, 1 / max(c, 1)) pair in its context; a helper evaluating on another warp's
  // tables (Dalt) never touches the pair, so there is one reader / writer and no ordering to think about.
  // The miss path is a function of its own: inlined it sat in the middle of the hot instruction stream
  // (0.5 KB the sequential prefetch fetched for nothing: icc hit rate 90.2 -> 87.7 %, -3 % solves/s).
  const double icm = __builtin_expect(!Dalt && c == cx->icm_c, 1) ? cx->icm : icm_miss(c, sm.ctx, Dalt == nullptr);
  const double vr = sm.vref[lk];
  double t_vel, t_ctl, t_acc;
  double aa, aw, ea, ew, alm;
  {
    const double dv_ = v - vr;
    t_vel = cx->qvel * (dv_ * dv_);
    t_ctl = fma(cx->rw, w * w, cx->rv * (v * v));
    double vp = __shfl_up_sync(FULL, v, 1), wp = __shfl_up_sync(FULL, w, 1);
    if (lane == 0) { vp = cx->v_init; wp = cx->w_init; }
    aa = (v - vp) * g.inv_ts; aw = (w - wp) * g.inv_ts;
    t_acc = fma(aw * aw, cx->wacc_pen, (aa * aa) * cx->acc_pen);
    double z = fma(ya, icm, aa);
    ea = z - clipd(z, g.amin, g.amax);
    z = fma(yw, icm, aw);
    ew = z - clipd(z, -g.awmax, g.awmax);
    alm = fma(ew, ew, ea * ea);
  }
  // ---- rollout (motion_model.py:153-176; RK4 of the unicycle = Simpson in theta):
  //      theta and position are prefix sums over the lanes
  const double tw = ts * w;
  const double th_in = wscan(tw, lane);
  double th_ex = __shfl_up_sync(FULL, th_in, 1);
  if (lane == 0) th_ex = 0.0;
  const double tha = cx->th0 + th_ex;
  const double thb = fma(0.5, tw, tha), thc = tha + tw;
  double sa, ca, sb, cb, sc, cc;
  tt_sincos_c(tha, &sa, &ca);
  tt_sincos_c(thb, &sb, &cb);
  // heading at the end of step k = heading at the start of step k + 1 (lane k + 1 holds its sine
  // and cosine; lane N exists and carries w = 0 when N < 32): two sincos per evaluation, not three.
  // The two values differ by the rounding of (th0 + scan_{k-1}) + ts w_k against th0 + scan_k;
  // the oracle's WARP order does the same.
  if (N < 32) {
    sc = __shfl_down_sync(FULL, sa, 1); cc = __shfl_down_sync(FULL, ca, 1);
  } else {
    tt_sincos_c(thc, &sc, &cc);
  }
  const double Cs = fma(4.0, cb, ca) + cc, Ss = fma(4.0, sb, sa) + sc;
  const double hv = g.h6 * v;
  const double dx = hv * Cs, dy = hv * Ss;
  double X, Y;
  {  // two prefix scans, interleaved
    double a = dx, b = dy;
    wscan2(a, b);
    X = cx->x0 + a; Y = cx->y0 + b;
  }
  const double TH = cx->th0 + th_in;
  if (st_out && act) { st_out[3 * lane] = X; st_out[3 * lane + 1] = Y; st_out[3 * lane + 2] = TH; }

  // every rolled-out position inside the scene's box?  then only the "live" robots / obstacles
  // can contribute (the others are farther than their radius from every point of the box)
  const bool in_box = __all_sync(FULL, fabs(X - cx->x0) < cx->box_half && fabs(Y - cx->y0) < cx->box_half);
  double cost;               // this lane's share of f
  double gx = 0.0, gy = 0.0; // d psi / d position_{k+1}
  double S_loc = 0.0, gSx = 0.0, gSy = 0.0;

  // ---- one static obstacle (l.214-220): hard penalty only.  The edge products of an obstacle are formed
  //      once; its sum / gradient terms are entered through a warp vote by the lanes that are inside it.
  auto static_obstacle = [&](int i) {
    const double *b = sm.os + i * nstcobs, *na0 = b + ne, *na1 = b + 2 * ne;
    double m[MAX_EDGE], sq[MAX_EDGE];
    double inside = 1.0;
#pragma unroll
    for (int e = 0; e < MAX_EDGE; e++) {
      if (e < ne) {
        m[e] = relu(fma(na1[e], Y, fma(na0[e], X, b[e])));
        sq[e] = m[e] * m[e];
        inside *= sq[e];
      }
    }
    if (__builtin_expect(__any_sync(FULL, inside > 0.0), 0)) {
      if (inside > 0.0) {
        S_loc += inside;
        if (GRAD) {
#pragma unroll
          for (int e = 0; e < MAX_EDGE; e++) {
            if (e < ne) {
              double rest = 1.0;
#pragma unroll
              for (int e2 = 0; e2 < MAX_EDGE; e2++)
                if (e2 < ne && e2 != e) rest *= sq[e2];
              const double coef = rest * (2.0 * m[e]);
              gSx = fma(coef, na0[e], gSx);
              gSy = fma(coef, na1[e], gSy);
            }
          }
        }
      }
    }
  };
  // ---- reference-path deviation (l.124-139, 202): min over the remaining segments j >= k.
  //      Step k has N - k segments (lane 0 the most); the 32 - N lanes beyond the horizon take
  //      the upper half of the ranges of the first 32 - N steps, so the loop is ~N/2 long.
  //      min is exact and ties go to the lower segment index, as in the sequential fold.
  {
    const int nh = 32 - N;                                  // lanes available as helpers
    const bool is_helper = !act && (lane - N) < N;          // helper of step lane - N
    const int kq = is_helper ? lane - N : lk;               // the step whose position this lane tests
    const double Xq = __shfl_sync(FULL, X, kq), Yq = __shfl_sync(FULL, Y, kq);
    const bool split = kq < nh;                             // this step's range is shared
    const int mid = kq + (N - kq + 1) / 2;
    const int lo = is_helper ? mid : kq;
    const int hi = (act && split) ? mid : N;
    const int cnt = (act || is_helper) ? hi - lo : 0;
    const int trips = (nh >= N) ? (N + 1) / 2 : max((N + 1) / 2, N - nh);
    double dmin = INFINITY; int jmin = lo;
    const double2 *segv = reinterpret_cast<const double2 *>(sm.seg);
    // unrolled by 2 in both builds: two independent distance chains per trip
#pragma unroll 2
    for (int t = 0; t < trips; t++) {
      const int j = min(lo + t, N - 1);
      const double2 s1 = segv[3 * j], sd = segv[3 * j + 1];
      const double inv = sm.seg[6 * j + 4];
      const double px = Xq - s1.x, py = Yq - s1.y;
      const double t_hat = fma(py, sd.y, px * sd.x) * inv;
      const double tt = clamp01(t_hat);
      const double qx = fma(tt, sd.x, -px), qy = fma(tt, sd.y, -py);
      const double d2 = fma(qy, qy, qx * qx);
      const bool take = (t < cnt) && !(dmin <= d2);  // first minimum wins ties
      dmin = take ? d2 : dmin;
      jmin = take ? j : jmin;
    }
    {  // fold the helper's half into the owner (owner = lower indices wins ties)
      const int src = (act && split) ? N + lane : lane;
      const double dh = __shfl_sync(FULL, dmin, src);
      const int jh = __shfl_sync(FULL, jmin, src);
      if (act && split && !(dmin <= dh)) { dmin = dh; jmin = jh; }
    }
    cost = dmin * cx->qrpd;
    if (GRAD) {
      const int j = act ? jmin : N - 1;
      const double2 s1 = segv[3 * j], sd = segv[3 * j + 1];
      const double inv = sm.seg[6 * j + 4];
      const double px = X - s1.x, py = Y - s1.y;
      const double t_hat = fma(py, sd.y, px * sd.x) * inv;
      const double t = clamp01(t_hat);
      const double qx = fma(t, sd.x, -px), qy = fma(t, sd.y, -py);
      const double pass = (t_hat >= 0.0 && t_hat <= 1.0) ? 1.0 : 0.0;
      const double cs = fma(qy, sd.y, qx * sd.x) * pass * inv;
      gx = cx->qrpd * (2.0 * fma(cs, sd.x, -qx));
      gy = cx->qrpd * (2.0 * fma(cs, sd.y, -qy));
    }
  }
  // ---- speed reference + control action (l.203-204)
  cost += t_vel;
  cost += t_ctl;
  // ---- fleet collision (l.207-211): contacts are rare -> fp32 prefilter from shared memory,
  //      one vote, then the exact fp64 terms (parameters in global memory) for the flagged
  //      robots in the same order (Nother <= 32)
  //      Both obstacle blocks sit behind ONE warp-uniform test: a scene whose box meets no other
  //      robot and no moving obstacle (every scene of the static workload) walks around ~2 KB of code.
  const unsigned fleet_todo = in_box ? cx->fleet_live : (Nother >= 32 ? 0xffffffffu : ((1u << Nother) - 1u));
  using dmask = typename DM::dmask;
  const dmask dyn_todo = in_box ? (dmask)cx->dyn_live
                                : (Ndyn >= (int)(8 * sizeof(dmask)) ? ~(dmask)0 : (((dmask)1 << Ndyn) - (dmask)1));
  dmask hard_mask = 0;  // obstacles with a positive hard term on this lane
  bool any_hard = false;
  if (fleet_todo != 0u || dyn_todo != 0ull) {
  const float Xf = (float)X, Yf = (float)Y;
  {
    unsigned hit = 0;
    const float thr = cx->fleet_thr;
    unsigned todo = fleet_todo;
    while (todo) {
      const int j = __ffs(todo) - 1;
      todo &= todo - 1;
      const float2 o = sm.fleet[j * N + lk];
      const float exf = Xf - o.x, eyf = Yf - o.y;
      hit |= (!((exf * exf + eyf * eyf) >= thr) ? 1u : 0u) << j;
    }
    if (__builtin_expect(__any_sync(FULL, hit != 0), 0)) {
      const double *cp = cx->p + g.off_c + 3 * lk;
      double acc = 0.0, fx = 0.0, fy = 0.0;
      while (hit) {
        const int j = __ffs(hit) - 1;
        hit &= hit - 1;
        const double ex = X - cp[(size_t)j * 3 * N], ey = Y - cp[(size_t)j * 3 * N + 1];
        const double e = g.veh_d2 - fma(ey, ey, ex * ex);
        if (e > 0.0) {
          acc += e;
          if (GRAD) { fx = fma(-2.0, ex, fx); fy = fma(-2.0, ey, fy); }
        }
      }
      cost += 1000.0 * acc;
      if (GRAD) { gx = fma(1000.0, fx, gx); gy = fma(1000.0, fy, gy); }
    }
  }
  // ---- dynamic obstacles (l.225-237): hard penalty D_j and soft cost.
  //      fp32 bounding test from shared memory first; the exact fp64 body (global
  //      table) only runs for pairs that can be non-zero.
  {
    dmask near_mask = 0;
    dmask todo = dyn_todo;
    while (todo) {
      const int j = first_bit(todo);
      todo &= todo - 1;
      const float *b = sm.dynb + 3 * (j * N + lk);
      const float exf = Xf - b[0], eyf = Yf - b[1];
      near_mask |= (dmask)((exf * exf + eyf * eyf) < b[2] ? 1u : 0u) << j;
    }
    if (__builtin_expect(__any_sync(FULL, near_mask != 0), 0)) {
      double soft = 0.0;
      int bodies = 0;
      while (near_mask) {
        const int j = first_bit(near_mask);
        near_mask &= near_mask - 1;
        const DynRow T = dyn_row<dmask>(sm, cx, j, N, Ndyn, lk);
        const double ex = X - T.p[0];
        const double ey = Y - T.p[T.sf];
        if (fma(ey, ey, ex * ex) < T.p[2 * T.sf]) {
          bodies++;
          const double ca_ = T.p[3 * T.sf];
          const double sa_ = T.p[4 * T.sf];
          const double A = fma(ey, sa_, ex * ca_), B = fma(-ey, ca_, ex * sa_);
          const double A2 = A * A, B2 = B * B;
          const double in1 = fma(-B2, T.p[6 * T.sf], fma(-A2, T.p[5 * T.sf], 1.0));
          if (in1 > 0.0) hard_mask |= (dmask)1 << j;
          const double iRxm = T.p[7 * T.sf];
          const double iRym = T.p[8 * T.sf];
          const double in2 = fma(-B2, iRym, fma(-A2, iRxm, 1.0));
          if (in2 > 0.0) {
            const double ws = T.p[9 * T.sf];
            soft = fma(in2 * in2, ws, soft);
            if (GRAD) {
              const double wg = ws * (2.0 * in2);
              const double tA = A * iRxm, tB = B * iRym;
              gx = fma(wg, -2.0 * fma(tB, sa_, tA * ca_), gx);
              gy = fma(wg, -2.0 * fma(-tB, ca_, tA * sa_), gy);
            }
          }
        }
      }
      cost += soft;
      if (!act) { bodies = 0; hard_mask = 0; }
      bodies = __reduce_add_sync(FULL, bodies);
      if (lane == 0 && !Dalt) sm.ctx->n_body += bodies;
    }
  }
  // hard terms are rare: one vote for the whole loop, per-obstacle sums only when needed
  any_hard = __any_sync(FULL, hard_mask != 0);
  if (__builtin_expect(any_hard, 0)) {
    dmask warp_hard;
    if constexpr (sizeof(dmask) == 4) {
      warp_hard = __reduce_or_sync(FULL, (unsigned)hard_mask);
    } else {
      const unsigned lo = __reduce_or_sync(FULL, (unsigned)hard_mask);
      const unsigned hi = __reduce_or_sync(FULL, (unsigned)((unsigned long long)hard_mask >> 32));
      warp_hard = (dmask)(((unsigned long long)hi << 32) | lo);
    }
    for (int j = lane; j < Ndyn; j += 32) Dv[j] = 0.0;
    __syncwarp();
    // per-obstacle sums only for the obstacles some lane is inside of
    while (warp_hard) {
      const int j = first_bit(warp_hard);
      warp_hard &= warp_hard - 1;
      double in1 = 0.0;
      if (hard_mask >> j & (dmask)1) {
        const DynRow T = dyn_row<dmask>(sm, cx, j, N, Ndyn, lk);
        const double ex = X - T.p[0];
        const double ey = Y - T.p[T.sf];
        const double ca_ = T.p[3 * T.sf];
        const double sa_ = T.p[4 * T.sf];
        const double A = fma(ey, sa_, ex * ca_), B = fma(-ey, ca_, ex * sa_);
        in1 = fma(-(B * B), T.p[6 * T.sf], fma(-(A * A), T.p[5 * T.sf], 1.0));
      }
      const double Dj = wsum(in1);
      if (lane == 0) Dv[j] = Dj;
    }
    __syncwarp();
  }
  }  // fleet_todo | dyn_todo
  // ---- terminal cost (l.242)
  double gt = 0.0;
  // both terminal weights zero (config/mpc_default.yaml): every term below is a signed zero; the block is
  // a divergent branch of ~25 instructions run by one lane while 31 wait.  Mirrored in the oracle's WARP order.
  if (lane == N - 1 && (cx->qN != 0.0 || cx->qthetaN != 0.0)) {
    const double dxg = X - cx->xg, dyg = Y - cx->yg, dtg = TH - cx->thg;
    cost += fma(cx->qthetaN, dtg * dtg, cx->qN * fma(dyg, dyg, dxg * dxg));
    if (GRAD) {
      gx = fma(2.0 * cx->qN, dxg, gx);
      gy = fma(2.0 * cx->qN, dyg, gy);
      gt = 2.0 * cx->qthetaN * dtg;
    }
  }
  // ---- static obstacles (l.214-220), in obstacle order like the reference fold
  {
#pragma unroll(DM::kStaticUnroll)
    for (int i = 0; i < Nstc; i++) static_obstacle(i);
  }
  // ---- accelerations: cost (l.250-264) and the ALM set C = acc bounds
  cost += t_acc;
  // ---- lanes beyond the horizon contribute nothing
  if (!act) {
    cost = 0.0; gx = 0.0; gy = 0.0; S_loc = 0.0; gSx = 0.0; gSy = 0.0;
    aa = 0.0; aw = 0.0; ea = 0.0; ew = 0.0; alm = 0.0;
  }
  // ---- static sum: needed before the gradient (weight c * sum F2); zero in most evaluations
  double S = 0.0;
  if (__builtin_expect(__any_sync(FULL, S_loc != 0.0), 0)) S = wsum(S_loc);
  double f2sq = 0.0, sumF2 = 0.0;
  if (__builtin_expect(any_hard, 0)) {
#pragma unroll 1
    for (int j = 0; j < Ndyn; j++) {
      const double F2j = S + Dv[j];
      f2sq = fma(F2j, F2j, f2sq);
      sumF2 += F2j;
    }
  } else if (__builtin_expect(S != 0.0, 0)) {  // every D_j is zero: F2_j = S + 0.0 = S (same operations, no loads)
    // taken by every second evaluation of the static workload (a robot inside a polygon): two dependent
    // chains of Ndyn links; unrolled by 5 the 15 trips cost 39 instructions instead of 75
#pragma unroll 5
    for (int j = 0; j < Ndyn; j++) {
      f2sq = fma(S, S, f2sq);
      sumF2 += S;
    }
  }  // S == 0 and no hard term: the loop would leave f2sq = sumF2 = +0
  EvalOut out;
  out.f2sq = f2sq; out.S = S; out.any_hard = any_hard;
  out.gv = 0.0; out.gw = 0.0;
  out.h0 = out.h1 = out.dd = out.g2 = 0.0;
  double ddp = 0.0, g2p = 0.0;

  if (GRAD) {
    double gv = 0.0, gw = 0.0;
    // hard-penalty gradient: c * sum_j F2_j * (grad S + grad D_j)
    if (c != 0.0) {
      const double cs_ = c * sumF2;
      gx = fma(cs_, gSx, gx);
      gy = fma(cs_, gSy, gy);
      if (__builtin_expect(any_hard, 0)) {
        dmask mk = hard_mask;
        while (mk) {
          const int j = first_bit(mk);
          mk &= mk - 1;
          const DynRow T = dyn_row<dmask>(sm, cx, j, N, Ndyn, lk);
          const double ex = X - T.p[0];
          const double ey = Y - T.p[T.sf];
          const double ca_ = T.p[3 * T.sf];
          const double sa_ = T.p[4 * T.sf];
          const double iRx = T.p[5 * T.sf];
          const double iRy = T.p[6 * T.sf];
          const double A = fma(ey, sa_, ex * ca_), B = fma(-ey, ca_, ex * sa_);
          const double wg = c * (S + Dv[j]);
          const double tA = A * iRx, tB = B * iRy;
          gx = fma(wg, -2.0 * fma(tB, sa_, tA * ca_), gx);
          gy = fma(wg, -2.0 * fma(-tB, ca_, tA * sa_), gy);
        }
      }
    }
    // adjoint of the rollout: suffix scans (d pos_{k+1}/d theta_k = (-dy, dx))
    const double dxdv = g.h6 * Cs, dydv = g.h6 * Ss;
    const double hvt = hv * ts;
    const double dxdw = -(hvt * fma(2.0, sb, sc)), dydw = hvt * fma(2.0, cb, cc);
    double lx = gx, ly = gy;
    wsuffix2(lx, ly);
    const double m = fma(ly, dx, -(lx * dy));
    const double lt = wsuffix(gt + m, lane) - m;
    // direct control terms
    const double aa_n = __shfl_down_sync(FULL, aa, 1), aw_n = __shfl_down_sync(FULL, aw, 1);
    const double ea_n = __shfl_down_sync(FULL, ea, 1), ew_n = __shfl_down_sync(FULL, ew, 1);
    if (act) {
      const bool last = lane == N - 1;
      double dv = 2 * cx->qvel * (v - vr) + 2 * cx->rv * v;
      double dw = 2 * cx->rw * w;
      dv += (2 * cx->acc_pen * (aa - (last ? 0.0 : aa_n)) + c * (ea - (last ? 0.0 : ea_n))) * g.inv_ts;
      dw += (2 * cx->wacc_pen * (aw - (last ? 0.0 : aw_n)) + c * (ew - (last ? 0.0 : ew_n))) * g.inv_ts;
      gv = dv + lx * dxdv + ly * dydv;
      gw = dw + lx * dxdw + ly * dydw + lt * ts;
    }
    out.gv = gv; out.gw = gw;
    if (gamma_ls > 0.0 && act) {  // PANOC line search: gradient step, projection, envelope terms
      const double s0 = fma(-gamma_ls, gv, v), s1 = fma(-gamma_ls, gw, w);
      out.h0 = clipd(s0, g.vmin, g.vmax); out.h1 = clipd(s1, -g.wmax, g.wmax);
      const double q0 = out.h0 - s0, q1 = out.h1 - s1;
      ddp = pdot(q0, q1, q0, q1);
      g2p = pdot(gv, gw, gv, gw);
    }
  }
  // ---- one batched reduction: f, ALM distance (and the line-search scalars)
  wsum4(cost, alm, ddp, g2p, lane);
  out.f = cost; out.dd = ddp; out.g2 = g2p;
  out.psi = cost + c * alm / 2 + c * f2sq / 2;
  return out;
}

}  // namespace ttmpc
