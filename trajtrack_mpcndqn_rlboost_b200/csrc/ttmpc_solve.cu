// ttmpc_solve.cu -- persistent warp-per-scene PANOC + ALM/PM solve kernel and the
// batched evaluation kernel.  See ttmpc_device.cuh for the data layout.
//
// Solver structure follows OpEn (optimization_engine 0.7.x), the solver the
// reference calls at src/mpc_traj_tracker/trajectory_generator.py:284:
//   outer loop  : AlmOptimizer::solve / step       (alm_optimizer.rs)
//   inner loop  : PANOCOptimizer::solve, PANOCEngine::{init,step} (panoc_*.rs)
//   direction   : lbfgs crate two-loop recursion with C-BFGS safeguard
// but is laid out for a warp: vectors are 2 registers per lane, the L-BFGS
// history is a ring of double2 rows in shared memory, dot products are
// butterfly all-reduces.
#include "ttmpc_device.cuh"
#include "ttmpc_launch.cuh"
#include <algorithm>
#include <cstdlib>
#include <map>
#include <mutex>
#include <tuple>

// This file is compiled twice (Makefile).  ttmpc_solve.o: hot loops unrolled -- lowest latency of a
// single scene, ~47 KB of SASS per PANOC iteration.  ttmpc_solve_small.o (ttmpc_solve_small.cu,
// -DTTMPC_SMALL_CODE): every hot loop rolled -- same arithmetic in the same order, bit-identical
// results, smaller loop body, better instruction-cache behaviour with 12 warps per SM at different
// places of the loop; the API launches it for batches larger than the resident warps.  Only the
// solve kernel and its launcher exist in that build, under these names:
#ifndef TTMPC_MIN_BLOCKS
// CTAs of TTMPC_MAX_THREADS threads per SM the register budget is sized for.  Unrolled build: 2 of 128
// -> up to 255 registers, 8 resident scenes per SM.  Rolled build (Makefile): 3 of 128 -> 168 registers,
// 12 resident scenes per SM (six 64-thread CTAs for the default shapes), without spills: the PANOC / ALM state that is read a few times per
// iteration lives in the warp's shared memory (WarpCtx, the L-BFGS old_state / old_g rows), not in
// registers (DESIGN.md section 3.1).
#define TTMPC_MIN_BLOCKS 2
#endif
#ifndef TTMPC_MIN_BLOCKS_RUNTIME
// the same for the run-time-dimension kernel (DimsRuntime), which needs more registers than the
// specialised shapes: it keeps its 255 registers in both builds
#define TTMPC_MIN_BLOCKS_RUNTIME TTMPC_MIN_BLOCKS
#endif
#ifndef TTMPC_MAX_THREADS
#define TTMPC_MAX_THREADS 128  // CTA size the register budget is computed for (the API launches 64)
#endif
#ifdef TTMPC_SMALL_CODE
#define solve_kernel solve_kernel_small
#define launch_solve launch_solve_small
#define solve_occupancy solve_occupancy_small
#endif

namespace ttmpc {

// PANOC constants (panoc_engine.rs)
constexpr double GAMMA_L_COEFF = 0.95;
constexpr double DELTA_LIPSCHITZ = 1e-12;
constexpr double EPSILON_LIPSCHITZ = 1e-6;
constexpr double LIPSCHITZ_UPDATE_EPSILON = 1e-6;
constexpr int MAX_LIPSCHITZ_UPDATE_ITERATIONS = 10;
constexpr double MAX_LIPSCHITZ_CONSTANT = 1e9;
constexpr int MAX_LINESEARCH_ITERATIONS = 10;
// The line search's tau starts at 1 and only halves, so tau = 2^-k exactly after k halvings:
// k < MAX_LINESEARCH_ITERATIONS  <=>  tau > 2^-MAX_LINESEARCH_ITERATIONS
constexpr double MIN_LINESEARCH_TAU = 1.0 / (1 << MAX_LINESEARCH_ITERATIONS);
constexpr double MIN_L_ESTIMATE = 1e-10;
// lbfgs settings chosen by PANOCCache::new
constexpr double CBFGS_EPSILON = 1e-8;
constexpr double SY_EPSILON = 1e-10;

// per-lane L-BFGS + PANOC state
struct Lane {
  double u0, u1;          // current iterate
  double g0, g1;          // gradient at u (or u_plus during the line search)
  double h0, h1;          // u_half_step
  double d0, d1;          // L-BFGS direction
  double f0, f1;          // gamma * fixed point residual
};

struct Uni {  // warp-uniform scalars
  double gamma, cost, norm_fpr;
  PanocCold *pc;  // the rest, in the warp's context
};

__device__ __forceinline__ void project(const DevCfg &g, double a0, double a1, double &o0, double &o1) {
  o0 = clipd(a0, g.vmin, g.vmax);
  o1 = clipd(a1, -g.wmax, g.wmax);
}

// The two scalars PANOC derives from gamma alone.  OpEn recomputes them in every iteration from an
// unchanged gamma (update_lipschitz_constant: the right-hand side of the check and sigma); a division
// is a 22-instruction call, so they are formed where gamma changes -- same operands, same IEEE
// division, same bits.
// (The coefficient of the check lives in the warp's shared-memory context: a 256th register does
// not exist and a spill costs more than the broadcast load.)
__device__ __forceinline__ void set_lip_coeff(const Uni &U, const WarpSmem &sm) {
  const double lc = tt_div(GAMMA_L_COEFF, 2.0 * U.gamma);
  __syncwarp();
  if ((threadIdx.x & 31) == 0) sm.ctx->lipc = lc;
  __syncwarp();
}
__device__ __forceinline__ void set_gamma_terms(Uni &U, const WarpSmem &sm) {
  U.pc->sigma = tt_div(1.0 - GAMMA_L_COEFF, 4.0 * U.gamma);
  set_lip_coeff(U, sm);
}
// x / gamma for the forward-backward envelope.  x = |gradient step - half step|^2 / 2 is exactly zero
// whenever no box bound is active, and a zero numerator sends the IEEE division down its slow path
// (~60 instructions and 1.5 KB of otherwise cold code in the instruction cache, taken by 11 % of all
// divisions of a static4096 batch).  0 / y = 0 with the sign of x for every y > 0: same bits.
__device__ __forceinline__ double div_env(double x, double y) {
  if (x == 0.0 && y > 0.0) return x;
  return tt_div(x, y);
}

// ---------------------------------------------------------------- L-BFGS, two-loop recursion
// lbfgs crate (0.2.x) update_hessian / apply_hessian as OpEn's PANOCCache configures it: same
// pairs, same C-BFGS acceptance test, same H0 = gamma I, the literal two-loop recursion with one
// butterfly all-reduce per inner product.
//
// Round 1 ran the two loops in compact (Gram) form: half the dependent latency of one apply
// (3.5 k instead of 7 k cycles), but 8 KB of hot code (Gram maintenance, lane-per-dot pass, two
// triangular recurrences).  Round 2 measured what that costs with the GPU full: the hot loop of the
// solve is walked by 8 warps per SM out of phase, every line of it missed the 32 KB instruction
// cache once per pass, and removing the L-BFGS code alone (experiment, profiles/r2_c_*) took the
// instruction-cache hit rate from 69 % to 94 % and the issue rate up by 43 %.  The literal recursion
// is ~1.5 KB, executes fewer instructions (no Gram upkeep), and its reduction latency is hidden
// by the other warps.  The CPU oracle's WARP order mirrors it (lb_apply with butterfly dots).
// lbfgs old_state / old_g := the current iterate and residual (per-lane rows of the warp's shared memory)
__device__ __forceinline__ void set_old(const WarpSmem &sm, const Lane &z, int lane) {
  sm.olds[lane] = make_double2(z.u0, z.u1);
  sm.oldg[lane] = make_double2(z.f0, z.f1);
}
// Returns whether the pair was accepted.  keep_old = false leaves old_state / old_g unchanged: the
// speculative update of panoc_step stores them (z.os = z.u, z.og = z.f) only once the speculation holds,
// so that a lost speculation has nothing per lane to restore.
template <class DM>
__device__ __forceinline__ bool lbfgs_update(const DevCfg &g, const WarpSmem &sm, Lane &z, Uni &U,
                                             int lane, bool keep_old = true) {
  const int N = DM::N(g), MEM = DM::mem(g), M1 = MEM + 1;
  const double2 os = sm.olds[lane], og = sm.oldg[lane];
  const double sv0 = z.u0 - os.x, sv1 = z.u1 - os.y;
  const double yv0 = z.f0 - og.x, yv1 = z.f1 - og.y;
  bool accept = true;
  double ys = 0.0, yy = 0.0;
  if (!U.pc->lb_first) {
    double ss = pdot(sv0, sv1, sv0, sv1);
    ys = pdot(sv0, sv1, yv0, yv1); yy = pdot(yv0, yv1, yv0, yv1);
    wsum3(ys, ss, yy);
    const double lhs = tt_div(ys, ss);
    const double rhs = CBFGS_EPSILON * U.norm_fpr;  // cbfgs_alpha = 1: pow(x, 1) == x
    accept = !(ss <= 2.2250738585072014e-308 || ys <= SY_EPSILON) &&
             (lhs > rhs && isfinite(lhs) && isfinite(rhs));
  }
  if (!accept) return false;
  if (keep_old) set_old(sm, z, lane);
  if (U.pc->lb_first) {
    __syncwarp();
    U.pc->lb_first = 0;
    return true;
  }
  // rotate_right(1): scratch slot becomes slot 0
  int k0 = U.pc->lb_head + MEM; if (k0 >= M1) k0 -= M1;
  const int active = min(MEM, U.pc->lb_active + 1);
  const double rho = tt_div(1.0, ys);
  if (lane < N) {
    sm.lbs[k0 * N + lane] = make_double2(sv0, sv1);
    sm.lby[k0 * N + lane] = make_double2(yv0, yv1);
  }
  if (lane == 0) sm.rho[k0] = rho;
  U.pc->lb_gamma = tt_div(tt_div(1.0, rho), yy);
  __syncwarp();
  U.pc->lb_head = k0; U.pc->lb_active = active;
  return true;
}

// lbfgs::apply_hessian on the direction.  The 2 m inner products of the recursion are one dependent chain
// (each needs the vector the previous one left), and with two warps per scheduler the solve follows the
// length of its dependent chains: their butterfly is inlined (no call, no argument / result moves on that
// chain) at the price of ~0.5 KB of hot code (DESIGN.md section 6).
template <class DM>
__device__ __forceinline__ void lbfgs_apply(const DevCfg &g, const WarpSmem &sm, Lane &z,
                                            const Uni &U, int lane) {
  const int m = U.pc->lb_active;
  if (m == 0) return;
  const int N = DM::N(g), M1 = DM::mem(g) + 1;
  const bool act = lane < N;
  const int lk = act ? lane : N - 1;
  double q0 = z.d0, q1 = z.d1, a_me = 0.0;  // lane i keeps alpha_i
  int k = U.pc->lb_head;
#pragma unroll 1
  for (int i = 0; i < m; i++) {  // newest to oldest
    const double2 s = sm.lbs[k * N + lk], y = sm.lby[k * N + lk];
    const double a = sm.rho[k] * wsum_inl(act ? pdot(s.x, s.y, q0, q1) : 0.0);
    if (lane == i) a_me = a;
    q0 = fma(-a, y.x, q0); q1 = fma(-a, y.y, q1);
    k = (k + 1 == M1) ? 0 : k + 1;
  }
  q0 = U.pc->lb_gamma * q0; q1 = U.pc->lb_gamma * q1;
#pragma unroll 1
  for (int i = m - 1; i >= 0; i--) {  // oldest to newest
    k = (k == 0) ? M1 - 1 : k - 1;
    const double2 s = sm.lbs[k * N + lk], y = sm.lby[k * N + lk];
    const double beta = sm.rho[k] * wsum_inl(act ? pdot(y.x, y.y, q0, q1) : 0.0);
    const double cf = __shfl_sync(FULL, a_me, i) - beta;
    q0 = fma(cf, s.x, q0); q1 = fma(cf, s.y, q1);
  }
  z.d0 = act ? q0 : 0.0; z.d1 = act ? q1 : 0.0;
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

#ifdef TTMPC_PROFILE
#define PROF_BEGIN(v) const long long v = clock64();
#define PROF_END(v, slot) if (lane == 0) sm.ctx->prof[slot] += clock64() - v;
#else
#define PROF_BEGIN(v)
#define PROF_END(v, slot)
#endif

// ---------------------------------------------------------------- tail helpers
// When the scene queue is empty, warps without work help the CTA-mates that still own a
// long-running scene: the owner posts evaluation points into a mailbox, the helper evaluates
// them on the owner's shared-memory tables.  The owner uses this to (a) overlap the Lipschitz
// check psi(u_half) with the L-BFGS update/apply and (b) evaluate the next line-search
// candidate speculatively.  Results never depend on whether a helper was there: speculative
// work is discarded when the sequential algorithm would not have asked for it.
struct CtaHelp {
  int busy[8];    // warp w owns a scene
  int helper[8];  // helper[m] = warp helping owner m, or -1
  int epoch[8];   // serial number of warp w's current scene (a helper serves one scene)
};
// Dynamic shared memory of a solve CTA: the CtaHelp table first, at a fixed address (a warp finds its
// helper slot from its own index instead of holding a pointer in registers), then one region per warp.
extern __shared__ __align__(16) unsigned char smem_raw[];
__device__ __forceinline__ CtaHelp *cta_help() { return reinterpret_cast<CtaHelp *>(smem_raw); }
__device__ __forceinline__ unsigned char *warp_region(const DevCfg &g, int w) {
  return smem_raw + sizeof(CtaHelp) + (size_t)w * g.smem_per_warp;
}
struct HelpCtl {
  bool enabled;              // helpers exist in this launch and none has timed out on this warp
  bool timed_out;            // a request was abandoned after the time-out: helpers stay off for this
                             // warp until the launch ends, and the abandoned request is waited for
                             // before the scene tables are re-staged (see solve_kernel)
  bool pending;              // a posted request has not been collected yet
};
__device__ __forceinline__ int ld_volatile_shared(unsigned addr) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
// HELP = false: the instantiation of panoc_step without any request path (see solve_scene)
template <bool HELP>
__device__ __forceinline__ bool help_available(const HelpCtl &hc) {
  if constexpr (!HELP) return false;
  else return hc.enabled && ld_volatile_shared((unsigned)__cvta_generic_to_shared(&cta_help()->helper[threadIdx.x >> 5])) >= 0;
}
// Collect the posted evaluation.  false = the helper did not answer in time (treated as gone).
__device__ __forceinline__ bool help_wait(HelpCtl &hc, const WarpSmem &sm, int lane, int N, EvalOut &e) {
  int ok = 1;
  if (lane == 0) {
    const volatile int *st = reinterpret_cast<volatile int *>(&sm.hhdr->state);
    const unsigned long long t0 = globaltimer_ns();
    int spins = 0;
    while (*st != 2) {
      if (((++spins) & 1023) == 0 && globaltimer_ns() - t0 > 50000000ull) { ok = 0; break; }
    }
  }
  ok = __shfl_sync(FULL, ok, 0);
  hc.pending = false;
  if (!ok) {
    hc.enabled = false;
    hc.timed_out = true;
    return false;
  }
  __threadfence_block();
  const volatile HelpHdr *h = sm.hhdr;
  e.psi = h->psi; e.f = h->f; e.f2sq = h->f2sq; e.S = h->S; e.dd = h->dd; e.g2 = h->g2;
  {
    const volatile double *hr = reinterpret_cast<const volatile double *>(sm.hres);
    e.gv = lane < N ? hr[2 * lane] : 0.0;
    e.gw = lane < N ? hr[2 * lane + 1] : 0.0;
  }
  e.any_hard = false;
  e.h0 = e.h1 = 0.0;
  __syncwarp();
  if (lane == 0) *reinterpret_cast<volatile int *>(&sm.hhdr->state) = 0;
  return true;
}
// The mailbox lives in the owner's shared-memory region (request row, answer row, header).
__device__ __forceinline__ void help_post(HelpCtl &hc, const WarpSmem &sm, int lane, int N, double v,
                                          double w, double c, int grad, double gamma_ls) {
  if (hc.pending) {  // a speculative evaluation nobody needed: let it finish first
    EvalOut tmp;
    if (!help_wait(hc, sm, lane, N, tmp)) return;
  }
  if (lane < N) sm.hreq[lane] = make_double2(v, w);
  if (lane == 0) { sm.hhdr->c = c; sm.hhdr->gamma_ls = gamma_ls; sm.hhdr->grad = grad; }
  __threadfence_block();
  __syncwarp();
  if (lane == 0) *reinterpret_cast<volatile int *>(&sm.hhdr->state) = 1;
  hc.pending = true;
}
__device__ __forceinline__ void help_drain(HelpCtl &hc, const WarpSmem &sm, int lane, int N) {
  if (hc.pending) { EvalOut tmp; help_wait(hc, sm, lane, N, tmp); }
}

struct Problem {  // what eval needs besides the point
  double c, ya, yw;
};

template <class DM>
__device__ __forceinline__ double eval_cost(const DevCfg &g, const WarpSmem &sm, int lane,
                                            const Problem &pb, double a0, double a1, HelpCtl &hc) {
  PROF_BEGIN(t0)
  EvalOut e = eval_psi<DM>(&g, reinterpret_cast<unsigned char *>(sm.ctx), a0, a1, pb.c, pb.ya,
                           pb.yw, nullptr, false, 0.0);
  PROF_END(t0, 0)
  if (lane == 0) sm.ctx->n_cost++;
  return e.psi;
}
template <class DM>
__device__ __forceinline__ double eval_grad(const DevCfg &g, const WarpSmem &sm, int lane,
                                            const Problem &pb, double a0, double a1, double &o0,
                                            double &o1, HelpCtl &hc) {
  PROF_BEGIN(t0)
  EvalOut e = eval_psi<DM>(&g, reinterpret_cast<unsigned char *>(sm.ctx), a0, a1, pb.c, pb.ya, pb.yw,
                           nullptr, true, 0.0);
  PROF_END(t0, 1)
  if (lane == 0) sm.ctx->n_grad++;
  o0 = e.gv; o1 = e.gw;
  return e.psi;
}

// fixed point residual, its norm and <grad, fpr> in one batched reduction
__device__ __forceinline__ void compute_fpr(Lane &z, Uni &U) {
  z.f0 = z.u0 - z.h0; z.f1 = z.u1 - z.h1;
  double nf = pdot(z.f0, z.f1, z.f0, z.f1), ip = pdot(z.g0, z.g1, z.f0, z.f1);
  wsum2(nf, ip);
  U.norm_fpr = tt_sqrt(nf);
  U.pc->ip = ip;
}
// The gradient step s = a - gamma g lives only here and in eval_psi: nothing reads it later except the two
// envelope scalars, which are formed right away where the solver needs them (ENV).
template <bool ENV>
__device__ __forceinline__ void gradient_and_half_step(const DevCfg &g, Lane &z, Uni &U,
                                                       double a0, double a1) {
  const double s0 = fma(-U.gamma, z.g0, a0), s1 = fma(-U.gamma, z.g1, a1);
  project(g, s0, s1, z.h0, z.h1);
  if constexpr (ENV) {
    const double e0 = s0 - z.h0, e1 = s1 - z.h1;
    double dist2 = pdot(e0, e1, e0, e1), gg = pdot(z.g0, z.g1, z.g0, z.g1);
    wsum2(dist2, gg);
    U.pc->env_dd = dist2; U.pc->env_g2 = gg;
  }
}

// Serve owner m (helper slot already taken) until its current scene ends.
// false = nothing happened for 3 s (the caller gives up helping).
template <class DM>
__device__ bool serve_owner(const DevCfg &g, CtaHelp *cta, int m, int epoch_m,
                            const WarpSmem &mine, int lane) {
  unsigned char *base_m = warp_region(g, m);
  const WarpSmem own = carve<DM>(base_m, g);
  const int N = g.N;
  unsigned long long t_idle = globaltimer_ns();
  int idle_polls = 0;
  while (true) {
    int st = 0, alive = 1;
    if (lane == 0) {
      st = *reinterpret_cast<volatile int *>(&own.hhdr->state);
      alive = *reinterpret_cast<volatile int *>(&cta->busy[m]) &&
              *reinterpret_cast<volatile int *>(&cta->epoch[m]) == epoch_m;
    }
    st = __shfl_sync(FULL, st, 0);
    alive = __shfl_sync(FULL, alive, 0);
    if (st == 1 && alive) {
      __threadfence_block();
      const volatile HelpHdr *h = own.hhdr;
      double2 pt = make_double2(0.0, 0.0), yv = make_double2(0.0, 0.0);
      if (lane < N) {
        const volatile double *rq = reinterpret_cast<const volatile double *>(own.hreq);
        const volatile double *yr = reinterpret_cast<const volatile double *>(own.yrow);
        pt.x = rq[2 * lane]; pt.y = rq[2 * lane + 1];
        yv.x = yr[2 * lane]; yv.y = yr[2 * lane + 1];
      }
      const double c = h->c, gamma_ls = h->gamma_ls;
      const int grad = h->grad;
      const EvalOut e = eval_psi<DM>(&g, base_m, pt.x, pt.y, c, yv.x, yv.y, nullptr, grad != 0, gamma_ls, mine.D);
      if (lane < N) own.hres[lane] = make_double2(e.gv, e.gw);
      if (lane == 0) {
        own.hhdr->psi = e.psi; own.hhdr->f = e.f; own.hhdr->f2sq = e.f2sq; own.hhdr->S = e.S;
        own.hhdr->dd = e.dd; own.hhdr->g2 = e.g2;
      }
      __threadfence_block();
      __syncwarp();
      if (lane == 0) *reinterpret_cast<volatile int *>(&own.hhdr->state) = 2;
      t_idle = globaltimer_ns();
      idle_polls = 0;
    } else if (!alive) {
      if (lane == 0) atomicExch(&cta->helper[m], -1);
      return true;
    } else {
      // the next request usually follows within a few thousand cycles: poll tightly first
      if (++idle_polls > 96) {
        __nanosleep(32);
        if ((idle_polls & 255) == 0 && globaltimer_ns() - t_idle > 3000000000ull) {
          if (lane == 0) atomicExch(&cta->helper[m], -1);
          return false;
        }
      }
    }
  }
}

// A warp that ran out of scenes serves its CTA-mates until none of them owns a scene.
template <class DM>
__device__ void helper_loop(const DevCfg &g, const SolveArgs &A, CtaHelp *cta, int warp, int lane) {
  const int W = g.warps_per_block;
  const WarpSmem mine = carve<DM>(warp_region(g, warp), g);
  const unsigned long long t_start = globaltimer_ns();
  while (true) {
    int m = -1, any_busy = 0, ep = 0;
    if (lane == 0) {
      for (int k = 1; k < W; k++) {
        const int cand = (warp + k) % W;
        if (*reinterpret_cast<volatile int *>(&cta->busy[cand])) {
          any_busy = 1;
          ep = *reinterpret_cast<volatile int *>(&cta->epoch[cand]);
          if (atomicCAS(&cta->helper[cand], -1, warp) == -1) { m = cand; break; }
        }
      }
    }
    m = __shfl_sync(FULL, m, 0);
    any_busy = __shfl_sync(FULL, any_busy, 0);
    ep = __shfl_sync(FULL, ep, 0);
    if (m < 0) {
      if (!any_busy || globaltimer_ns() - t_start > 20000000000ull) return;
      __nanosleep(2000);
      continue;
    }
    if (!serve_owner<DM>(g, cta, m, ep, mine, lane)) return;
  }
}

// While the queue is not empty: a warp that is about to fetch its next scene first looks for a
// CTA-mate whose scene has already taken several times the average number of evaluations and
// has no helper, and serves that scene to its end instead (a batch ends when its slowest scene
// does; the few warps this takes out of the pool cost ~1 % of the bulk rate).
// run_stats = {sum of evaluations, count} over finished scenes.
template <class DM>
__device__ bool help_long_running_mate(const DevCfg &g, const SolveArgs &A, CtaHelp *cta,
                                       int warp, int lane) {
  int m = -1, ep = 0;
  if (lane == 0) {
    const unsigned long long nd = *reinterpret_cast<volatile unsigned long long *>(A.run_stats + 1);
    if (nd >= 64) {
      const unsigned long long sum = *reinterpret_cast<volatile unsigned long long *>(A.run_stats);
      const long long thr = 4 * (long long)(sum / nd);
      const int W = g.warps_per_block;
      for (int k = 1; k < W; k++) {
        const int cand = (warp + k) % W;
        if (!*reinterpret_cast<volatile int *>(&cta->busy[cand]) ||
            *reinterpret_cast<volatile int *>(&cta->helper[cand]) != -1)
          continue;
        const volatile WarpCtx *cx = reinterpret_cast<const volatile WarpCtx *>(warp_region(g, cand));
        ep = *reinterpret_cast<volatile int *>(&cta->epoch[cand]);
        if (cx->n_cost + cx->n_grad > thr && atomicCAS(&cta->helper[cand], -1, warp) == -1) { m = cand; break; }
      }
    }
  }
  m = __shfl_sync(FULL, m, 0);
  ep = __shfl_sync(FULL, ep, 0);
  if (m < 0) return false;
  const WarpSmem mine = carve<DM>(warp_region(g, warp), g);
  serve_owner<DM>(g, cta, m, ep, mine, lane);
  return true;
}

__device__ __forceinline__ void halve_tau(Uni &U) {
  const double t = U.pc->tau / 2.0;
  __syncwarp();  // every lane has read tau
  U.pc->tau = t;
}

// PANOCEngine::step.  Returns true to continue.
template <class DM, bool HELP>
__device__ __forceinline__ bool panoc_step(const DevCfg &g, const WarpSmem &sm, int lane, const Problem &pb,
                           Lane &z, Uni &U, double tolerance, HelpCtl &hc) {
  PROF_BEGIN(t_step)
  const bool act = lane < DM::N(g);
  if (U.pc->iteration >= 1 && act) sm.gprev[lane] = make_double2(z.g0, z.g1);
  compute_fpr(z, U);
  if (__builtin_expect(U.norm_fpr < tolerance, 0)) {
    const double2 gp = act ? sm.gprev[lane] : make_double2(0.0, 0.0);
    const double r0 = fma(U.gamma, z.g0 - gp.x, z.f0), r1 = fma(U.gamma, z.g1 - gp.y, z.f1);
    if (sqrt(wsum(pdot(r0, r1, r0, r1))) < sm.ctx->akkt_tol) return false;
  }
  // update_lipschitz_constant (+ lbfgs_direction).  With a helper the Lipschitz check
  // psi(u_half) runs on the helper while this warp already updates / applies L-BFGS on the
  // current residual; if the check then asks for backtracking, the speculative L-BFGS state
  // is rolled back and the sequential path below runs unchanged.
  // One L-BFGS call site for both orders (the update + apply pair is ~7 KB of SASS; two inlined
  // copies -- one for owners with a helper, one for owners without -- sat in the instruction cache
  // of every SM at once; measured: same speed, 18 KB less code).  pass 0: L-BFGS first if a helper evaluates psi(u_half) meanwhile, then
  // the Lipschitz check; pass 1: L-BFGS if it has not been done or the speculation was lost.
  bool lbfgs_done = false;
  {
    double cost_half = 0.0;
    const bool spec = __builtin_expect(help_available<HELP>(hc), 0);
    bool s_accept = false;
    SpecSave &sv = sm.ctx->spec;
    if (spec) {
      PROF_BEGIN(tp)
      help_post(hc, sm, lane, DM::N(g), z.h0, z.h1, pb.c, 0, 0.0);
      PROF_END(tp, 4)  // helper timeline: post
      sv.lb_first = U.pc->lb_first; sv.lb_head = U.pc->lb_head; sv.lb_active = U.pc->lb_active;
      sv.lb_gamma = U.pc->lb_gamma;
    }
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
      if (pass == 0 ? spec : !lbfgs_done) {
        PROF_BEGIN(tl)
        {
          PROF_BEGIN(t0)
          const bool acc = lbfgs_update<DM>(g, sm, z, U, lane, pass != 0);
          if (pass == 0) s_accept = acc;
          PROF_END(t0, 2)
        }
        if (U.pc->iteration > 0) {
          PROF_BEGIN(t0)
          z.d0 = z.f0; z.d1 = z.f1;
          lbfgs_apply<DM>(g, sm, z, U, lane);
          PROF_END(t0, 3)
        }
        if (pass == 0) { PROF_END(tl, 5) }  // speculative L-BFGS
      }
      if (pass == 1) break;
      bool got = false;
      if (spec) {
        EvalOut r;
        PROF_BEGIN(tw)
        got = hc.pending && help_wait(hc, sm, lane, DM::N(g), r);
        PROF_END(tw, 6)  // waiting for the helper's psi(u_half)
        if (got) {
          cost_half = r.psi;
          if (lane == 0) sm.ctx->n_cost++;
        }
      }
      if (!got) cost_half = eval_cost<DM>(g, sm, lane, pb, z.h0, z.h1, hc);
      if (spec) {
        const double rhs0 = U.cost + LIPSCHITZ_UPDATE_EPSILON * fabs(U.cost) - U.pc->ip +
                            sm.ctx->lipc * (U.norm_fpr * U.norm_fpr);
        if (cost_half > rhs0 && U.pc->L < MAX_LIPSCHITZ_CONSTANT) {  // speculation lost
          U.pc->lb_first = sv.lb_first; U.pc->lb_head = sv.lb_head; U.pc->lb_active = sv.lb_active;
          U.pc->lb_gamma = sv.lb_gamma;
        } else {
          lbfgs_done = true;
          if (s_accept) set_old(sm, z, lane);
        }
      }
      int it = 0;
      while (true) {
        const double rhs = U.cost + LIPSCHITZ_UPDATE_EPSILON * fabs(U.cost) - U.pc->ip +
                           sm.ctx->lipc * (U.norm_fpr * U.norm_fpr);
        if (!(cost_half > rhs && it < MAX_LIPSCHITZ_UPDATE_ITERATIONS &&
              U.pc->L < MAX_LIPSCHITZ_CONSTANT))
          break;
        U.pc->lb_active = 0; U.pc->lb_first = 1;  // lbfgs.reset()
        const double L2 = U.pc->L * 2.0;
        __syncwarp();
        U.pc->L = L2;
        U.gamma /= 2.0;
        set_lip_coeff(U, sm);
        gradient_and_half_step<false>(g, z, U, z.u0, z.u1);
        cost_half = eval_cost<DM>(g, sm, lane, pb, z.h0, z.h1, hc);
        compute_fpr(z, U);
        it++;
      }
      // gamma moved: the envelope scalars of the new gradient step / half step (iteration 0 takes its own step below)
      if (it > 0 && U.pc->iteration > 0) gradient_and_half_step<true>(g, z, U, z.u0, z.u1);
      if (it > 0) U.pc->sigma = tt_div(1.0 - GAMMA_L_COEFF, 4.0 * U.gamma);  // gamma moved
    }
  }
  if (U.pc->iteration == 0) {
    // update_no_linesearch
    z.u0 = z.h0; z.u1 = z.h1;
    U.cost = eval_grad<DM>(g, sm, lane, pb, z.u0, z.u1, z.g0, z.g1, hc);
    gradient_and_half_step<true>(g, z, U, z.u0, z.u1);
  } else {
    // linesearch on the forward-backward envelope
    const double dist2 = U.pc->env_dd, gg = U.pc->env_g2;  // same vectors as in the evaluation / step that produced this iterate
    const double fbe = U.cost - 0.5 * U.gamma * gg + div_env(0.5 * dist2, U.gamma);
    U.pc->rhs_ls = fbe - U.pc->sigma * (U.norm_fpr * U.norm_fpr);
    U.pc->tau = 1.0;
    double p0, p1;
    while (true) {
      const double one_m = 1.0 - U.pc->tau;
      p0 = fma(-U.pc->tau, z.d0, fma(-one_m, z.f0, z.u0));
      p1 = fma(-U.pc->tau, z.d1, fma(-one_m, z.f1, z.u1));
      // with a helper: the next candidate (tau/2) is evaluated speculatively at the same time
      bool posted = false;
      double n0 = 0.0, n1 = 0.0;
      if (__builtin_expect(U.pc->tau > MIN_LINESEARCH_TAU && help_available<HELP>(hc), 0)) {
        const double tau2 = U.pc->tau / 2.0, one_m2 = 1.0 - tau2;
        n0 = fma(-tau2, z.d0, fma(-one_m2, z.f0, z.u0));
        n1 = fma(-tau2, z.d1, fma(-one_m2, z.f1, z.u1));
        help_post(hc, sm, lane, DM::N(g), n0, n1, pb.c, 1, U.gamma);
        posted = hc.pending;
      }
      // cost, gradient, gradient step, half step and both envelope scalars in one evaluation
      PROF_BEGIN(t0)
      EvalOut e = eval_psi<DM>(&g, reinterpret_cast<unsigned char *>(sm.ctx), p0, p1, pb.c,
                               pb.ya, pb.yw, nullptr, true, U.gamma);
      PROF_END(t0, 1)
      if (lane == 0) sm.ctx->n_grad++;
      U.cost = e.psi;
      z.g0 = e.gv; z.g1 = e.gw; z.h0 = e.h0; z.h1 = e.h1;
      double lhs_ls = U.cost - 0.5 * U.gamma * e.g2 + div_env(0.5 * e.dd, U.gamma);
      U.pc->env_dd = e.dd; U.pc->env_g2 = e.g2;
      if (!(lhs_ls > U.pc->rhs_ls && U.pc->tau > MIN_LINESEARCH_TAU)) break;
      halve_tau(U);
      if (posted && help_wait(hc, sm, lane, DM::N(g), e)) {  // the helper's evaluation is the one at this tau
        if (lane == 0) sm.ctx->n_grad++;
        p0 = n0; p1 = n1;
        U.cost = e.psi;
        z.g0 = e.gv; z.g1 = e.gw;
        gradient_and_half_step<false>(g, z, U, p0, p1);  // same s = p - gamma g, h = proj(s) the evaluation formed
        lhs_ls = U.cost - 0.5 * U.gamma * e.g2 + div_env(0.5 * e.dd, U.gamma);
        U.pc->env_dd = e.dd; U.pc->env_g2 = e.g2;
        if (!(lhs_ls > U.pc->rhs_ls && U.pc->tau > MIN_LINESEARCH_TAU)) break;
        halve_tau(U);
      }
    }
    z.u0 = p0; z.u1 = p1;
  }
  {
    const int it1 = U.pc->iteration + 1;
    __syncwarp();
    U.pc->iteration = it1;
  }
  PROF_END(t_step, 7)  // whole step
  return true;
}

__device__ __forceinline__ void panoc_reset(Uni &U) {
  U.pc->lb_active = 0; U.pc->lb_first = 1; U.pc->env_dd = 0.0; U.pc->env_g2 = 0.0;
  U.pc->tau = 1.0; U.pc->L = 0.0; U.pc->sigma = 0.0; U.cost = 0.0; U.pc->iteration = 0; U.gamma = 0.0;
}

// One scene, start to finish.
// The outer-loop (ALM) scalars live in the warp's context (WarpCtx).  They are warp-uniform: every lane
// stores the same value, and where a value is read and replaced in the same outer iteration, every lane
// reads it before the __syncwarp() that precedes the stores.
template <class DM>
__device__ void solve_scene(const DevCfg &g, const WarpSmem &sm, const SolveArgs &A, int scene,
                            int lane, HelpCtl &hc) {
  const int N = g.N;
  const bool act = lane < N;
  WarpCtx *const cx = sm.ctx;
  cx->t_start = __shfl_sync(FULL, globaltimer_ns(), 0);
#ifdef TTMPC_PROFILE
  const long long t_clk0 = clock64();
#endif
  Lane z;
  Uni U;
  U.pc = &cx->pc;
  Problem pb;
  z.u0 = z.u1 = 0.0;
  pb.ya = pb.yw = 0.0;
  if (act) {
    if (A.use_u0) {
      z.u0 = A.u[(size_t)scene * 2 * N + 2 * lane];
      z.u1 = A.u[(size_t)scene * 2 * N + 2 * lane + 1];
    }
    if (A.use_y0 && A.y) {
      pb.ya = A.y[(size_t)scene * 2 * N + lane];
      pb.yw = A.y[(size_t)scene * 2 * N + N + lane];
    }
  }
  pb.c = A.c0 ? A.c0[scene] : g.c0;
  z.g0 = z.g1 = z.h0 = z.h1 = 0.0;
  if (act) sm.gprev[lane] = make_double2(0.0, 0.0);
  z.d0 = z.d1 = z.f0 = z.f1 = 0.0;
  sm.olds[lane] = make_double2(0.0, 0.0);
  sm.oldg[lane] = make_double2(0.0, 0.0);
  U.pc->lb_head = 0; U.pc->lb_gamma = 1.0; U.norm_fpr = 0.0;
  panoc_reset(U);
  cx->akkt_tol = g.init_tol;

  double yp_a = 0.0, yp_w = 0.0;  // y_plus
  cx->dy_norm = 0.0; cx->dy_norm_plus = 0.0; cx->f2_norm = 0.0; cx->f2_norm_plus = 0.0;
  cx->last_fpr = 0.0; cx->f_final = 0.0;
  cx->inner_count = 0; cx->exit_status = TTMPC_CONVERGED; cx->panoc_iters = 0;
  cx->num_outer = 0;
  cx->scene = scene;
  const double SMALL_EPSILON = 2.220446049250313e-16;

  cx->in_time = 1;  // OpEn: max_duration (AlmOptimizer::solve / PANOCOptimizer::solve)
  for (int outer = 1; outer <= g.max_outer; outer = cx->num_outer + 1) {  // the counter lives in the context
    if (g.max_ns) {  // no time left before this outer iteration: NotConvergedOutOfTime
      unsigned long long el = globaltimer_ns() - cx->t_start;
      el = __shfl_sync(FULL, el, 0);
      if (el > g.max_ns) { cx->exit_status = TTMPC_NOT_CONVERGED_OUT_OF_TIME; cx->in_time = 0; break; }
    }
    cx->num_outer = outer;
    pb.ya = clipd(pb.ya, -1e12, 1e12);
    pb.yw = clipd(pb.yw, -1e12, 1e12);
    help_drain(hc, sm, lane, N);
    if (act) sm.yrow[lane] = make_double2(pb.ya, pb.yw);  // what a helper evaluates with
    __syncwarp();
    // ---------------- inner problem: PANOCOptimizer::solve
    int inner_status;
    {
      panoc_reset(U);
      // init: cost, gradient, local Lipschitz estimate
      U.cost = eval_grad<DM>(g, sm, lane, pb, z.u0, z.u1, z.g0, z.g1, hc);
      if (lane == 0) sm.ctx->n_cost++;  // the reference evaluates cost and gradient separately
      {
        double h0 = 0.0, h1 = 0.0;
        if (act) {
          h0 = (EPSILON_LIPSCHITZ * z.u0 > DELTA_LIPSCHITZ) ? EPSILON_LIPSCHITZ * z.u0 : DELTA_LIPSCHITZ;
          h1 = (EPSILON_LIPSCHITZ * z.u1 > DELTA_LIPSCHITZ) ? EPSILON_LIPSCHITZ * z.u1 : DELTA_LIPSCHITZ;
        }
        double t0, t1;
        eval_grad<DM>(g, sm, lane, pb, z.u0 + h0, z.u1 + h1, t0, t1, hc);
        const double e0 = t0 - z.g0, e1 = t1 - z.g1;
        double nh = pdot(h0, h1, h0, h1);
        double nd = pdot(e0, e1, e0, e1);
        wsum2(nh, nd);
        U.pc->L = sqrt(nd) / sqrt(nh);
      }
      U.gamma = GAMMA_L_COEFF / fmax(U.pc->L, MIN_L_ESTIMATE);
      set_gamma_terms(U, sm);
      gradient_and_half_step<false>(g, z, U, z.u0, z.u1);

      // PANOCOptimizer::solve main loop (one call site: step, then count).  OpEn's iteration count
      // num_iter is the step counter after every step that continues, and one less after a step that
      // continues but ends the loop by the iteration or time limit; OpEn's `cont` is num_iter < max_inner
      // of the steps before the current one.
      bool flag;
      while (true) {
        // Two instantiations of the step: the plain one (no request path at all) runs while no
        // helper is attached to this warp -- every iteration of a bulk batch -- and keeps the hot
        // loop ~2 KB shorter (it is bound by the instruction cache, DESIGN.md section 6); the
        // helper-aware one takes over the moment a helper attaches (tail of a batch, one scene
        // alone).  Same arithmetic: results do not depend on which one ran.
        if (__builtin_expect(help_available<true>(hc), 0))
          flag = panoc_step<DM, true>(g, sm, lane, pb, z, U, g.tol, hc);
        else
          flag = panoc_step<DM, false>(g, sm, lane, pb, z, U, g.tol, hc);
        if (!(flag && U.pc->iteration - 1 < g.max_inner && cx->in_time)) break;
        if (g.max_ns) {
          unsigned long long el = globaltimer_ns() - cx->t_start;
          el = __shfl_sync(FULL, el, 0);
          cx->in_time = el <= g.max_ns;
        }
      }
      const int num_iter = flag ? U.pc->iteration - 1 : U.pc->iteration;
      const bool cont = num_iter < g.max_inner;
      const bool finite = isfinite(z.u0) && isfinite(z.u1);
      const int ic = cx->inner_count + num_iter;
      const unsigned long long pi = cx->panoc_iters + num_iter;
      const bool all_finite = __all_sync(FULL, finite);
      __syncwarp();
      cx->inner_count = ic;
      if (!all_finite) { cx->exit_status = TTMPC_NOT_FINITE; break; }
      z.u0 = z.h0; z.u1 = z.h1;
      inner_status = !cont ? TTMPC_NOT_CONVERGED_ITERATIONS
                           : (!cx->in_time ? TTMPC_NOT_CONVERGED_OUT_OF_TIME : TTMPC_CONVERGED);
      cx->panoc_iters = pi;
      cx->last_fpr = U.norm_fpr;
    }
    // ---------------- multipliers, infeasibility (alm_optimizer.rs step())
    double F1a = 0.0, F1w = 0.0;
    {
      double vp = __shfl_up_sync(FULL, z.u0, 1), wp = __shfl_up_sync(FULL, z.u1, 1);
      if (lane == 0) { vp = sm.ctx->v_init; wp = sm.ctx->w_init; }
      if (act) { F1a = (z.u0 - vp) * g.inv_ts; F1w = (z.u1 - wp) * g.inv_ts; }
    }
    {
      const double icm = 1.0 / fmax(pb.c, 1.0);
      double t = clipd(fma(pb.ya, icm, F1a), g.amin, g.amax);
      yp_a = pb.ya + pb.c * (F1a - t);
      t = clipd(fma(pb.yw, icm, F1w), -g.awmax, g.awmax);
      yp_w = pb.yw + pb.c * (F1w - t);
      if (!act) { yp_a = 0.0; yp_w = 0.0; }
    }
    double f2_norm_plus;
    {
      // c = 0: the multipliers do not enter f, F2
      const EvalOut e = eval_psi<DM>(&g, reinterpret_cast<unsigned char *>(sm.ctx), z.u0, z.u1, 0.0, 0.0,
                                     0.0, nullptr, false, 0.0);
      if (lane == 0) sm.ctx->n_cost++;
      f2_norm_plus = sqrt(e.f2sq);
      cx->f2_norm_plus = f2_norm_plus;
      cx->f_final = e.f;
    }
    double delta_y_norm_plus;
    {
      const double da = yp_a - pb.ya, dw = yp_w - pb.yw;
      delta_y_norm_plus = sqrt(wsum(pdot(da, dw, da, dw)));
      cx->dy_norm_plus = delta_y_norm_plus;
    }
    const double akkt_tol = cx->akkt_tol;
    const int alm_iter = cx->num_outer - 1;  // AlmOptimizer's iteration counter
    const bool crit1 = alm_iter > 0 && delta_y_norm_plus <= pb.c * g.delta_tol + SMALL_EPSILON;
    const bool crit2 = f2_norm_plus <= g.delta_tol + SMALL_EPSILON;
    const bool crit3 = akkt_tol <= g.tol + SMALL_EPSILON;
    if (crit1 && crit2 && crit3) { cx->exit_status = inner_status; break; }
    // is_penalty_stall_criterion: iteration 0, or both infeasibilities decreased enough
    const bool crit_alm = delta_y_norm_plus <= g.suff_dec * cx->dy_norm + SMALL_EPSILON;
    const bool crit_pm = g.Ndyn == 0 || f2_norm_plus <= g.suff_dec * cx->f2_norm + SMALL_EPSILON;
    const bool stall = alm_iter == 0 || (crit_alm && crit_pm);
    if (!stall) pb.c *= g.pen_factor;
    __syncwarp();
    cx->akkt_tol = fmax(akkt_tol * g.tol_factor, g.tol);
    if (act) sm.gprev[lane] = make_double2(0.0, 0.0);  // set_akkt_tolerance allocates a fresh zero vector
    cx->dy_norm = delta_y_norm_plus;
    cx->f2_norm = f2_norm_plus;
    pb.ya = yp_a; pb.yw = yp_w;
  }
  help_drain(hc, sm, lane, N);  // no evaluation on this scene's tables may still be in flight
  __syncwarp();
  int exit_status = cx->exit_status;
  const int num_outer = cx->num_outer;
  if (exit_status != TTMPC_NOT_FINITE && cx->in_time && num_outer == g.max_outer)
    exit_status = TTMPC_NOT_CONVERGED_ITERATIONS;

  // ---------------- results
  scene = cx->scene;
  if (act) {
    A.u[(size_t)scene * 2 * N + 2 * lane] = z.u0;
    A.u[(size_t)scene * 2 * N + 2 * lane + 1] = z.u1;
    if (A.y) {
      A.y[(size_t)scene * 2 * N + lane] = pb.ya;
      A.y[(size_t)scene * 2 * N + N + lane] = pb.yw;
    }
  }
  if (A.pred_states)
    eval_psi<DM>(&g, reinterpret_cast<unsigned char *>(sm.ctx), z.u0, z.u1, 0.0, 0.0, 0.0,
                 A.pred_states + (size_t)scene * N * 3, false, 0.0);
  if (lane == 0) {
    if (A.cost) A.cost[scene] = cx->f_final;
    if (A.exit_status) A.exit_status[scene] = exit_status;
    if (A.outer_iters) A.outer_iters[scene] = num_outer;
    if (A.inner_iters) A.inner_iters[scene] = cx->inner_count;
    if (A.last_fpr) A.last_fpr[scene] = cx->last_fpr;
    if (A.f1_infeas) A.f1_infeas[scene] = cx->dy_norm_plus / pb.c;
    if (A.f2_norm) A.f2_norm[scene] = cx->f2_norm_plus;
    if (A.penalty) A.penalty[scene] = pb.c;
    if (A.evals) {
      A.evals[4 * scene] = sm.ctx->n_cost; A.evals[4 * scene + 1] = sm.ctx->n_grad;
      A.evals[4 * scene + 2] = (long long)(globaltimer_ns() - cx->t_start);
      A.evals[4 * scene + 3] = (long long)cx->t_start;
    }
    // device-wide counters, added once per scene (a per-warp running sum would hold 8 registers
    // for the whole kernel)
    if (A.stats) {
      atomicAdd(A.stats + 0, (unsigned long long)sm.ctx->n_cost);
      atomicAdd(A.stats + 1, (unsigned long long)sm.ctx->n_grad);
      atomicAdd(A.stats + 2, (unsigned long long)sm.ctx->n_body);
      atomicAdd(A.stats + 3, cx->panoc_iters);
#ifdef TTMPC_PROFILE
      // 4: cost evals, 5: grad evals, 6: lbfgs update + apply, 7: whole solve (cycles)
      atomicAdd(A.stats + 4, (unsigned long long)sm.ctx->prof[0]);
      atomicAdd(A.stats + 5, (unsigned long long)sm.ctx->prof[1]);
      atomicAdd(A.stats + 6, (unsigned long long)(sm.ctx->prof[2] + sm.ctx->prof[3]));
      atomicAdd(A.stats + 7, (unsigned long long)(clock64() - t_clk0));
#endif
    }
#ifdef TTMPC_PROFILE
#ifndef TTMPC_PROFILE_STAGE
    sm.ctx->eprof[9] = sm.ctx->prof[3];  // L-BFGS apply alone (slot 6 holds update + apply)
#else
    sm.ctx->eprof[9] = 0;
    sm.ctx->eprof[8] = sm.ctx->prof[4]; sm.ctx->eprof[7] = sm.ctx->prof[5];  // staging part 1 / part 2
#endif
#ifdef TTMPC_PROFILE_HELP
    for (int i = 0; i < 4; i++) sm.ctx->eprof[i] = sm.ctx->prof[4 + i];  // helper timeline instead of eval sections
#endif
    if (A.eprof) for (int i = 0; i < 10; i++) atomicAdd(A.eprof + i, (unsigned long long)sm.ctx->eprof[i]);
#endif
  }
}

template <class DM>
__global__ void __launch_bounds__(TTMPC_MAX_THREADS, DM::kN ? TTMPC_MIN_BLOCKS : TTMPC_MIN_BLOCKS_RUNTIME) solve_kernel(const __grid_constant__ DevCfg g,
                                                    const __grid_constant__ SolveArgs A) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const WarpSmem sm = carve<DM>(warp_region(g, warp), g);
  CtaHelp *cta = cta_help();
  if (threadIdx.x < 8) { cta->busy[threadIdx.x] = 0; cta->helper[threadIdx.x] = -1; cta->epoch[threadIdx.x] = 0; }
  __syncthreads();
  HelpCtl hc;
  hc.enabled = A.helpers != 0;
  hc.timed_out = false;
  hc.pending = false;
  if (lane == 0) sm.hhdr->state = 0;
  bool had_scene = false;
  while (true) {
    if (had_scene && A.helpers && A.run_stats && help_long_running_mate<DM>(g, A, cta, warp, lane))
      continue;
    int scene = 0;
    if (lane == 0) scene = atomicAdd(A.work_counter, 1);
    scene = __shfl_sync(FULL, scene, 0);
    if (scene >= A.n_scenes) break;
    had_scene = true;
    if (A.order) scene = A.order[scene];  // likely-long scenes first (rank_scenes_kernel)
    // owner from here on: warps that find the queue empty may attach as helpers already while
    // the tables are being staged (requests are only posted from solve_scene)
    if (lane == 0) {
      *reinterpret_cast<volatile int *>(&cta->epoch[warp]) = cta->epoch[warp] + 1;
      *reinterpret_cast<volatile int *>(&cta->busy[warp]) = 1;
    }
    if (__builtin_expect(hc.timed_out, 0)) {
      // A request of an earlier scene was abandoned (the helper did not answer within the time-out:
      // the context was preempted or time-sliced).  The helper may still be evaluating on this
      // warp's tables: it detaches when it sees busy == 0 / a new epoch, so wait (bounded) until the
      // helper slot is empty or the abandoned request has been answered, then clear the mailbox.
      if (lane == 0) {
        const unsigned long long t0 = globaltimer_ns();
        const volatile int *stp = reinterpret_cast<volatile int *>(&sm.hhdr->state);
        while (*reinterpret_cast<volatile int *>(&cta->helper[warp]) >= 0 && *stp == 1) {
          __nanosleep(1000);
          if (globaltimer_ns() - t0 > 5000000000ull) break;
        }
      }
      __syncwarp();
    }
    if (lane == 0) *reinterpret_cast<volatile int *>(&sm.hhdr->state) = 0;  // mailbox empty at scene start
    __syncwarp();
    if (A.ready) {  // parameters of this scene may still be on their way from the host
      int ok = 1;
      if (lane == 0) {
        const volatile int *rdy = A.ready;
        const unsigned long long t0 = globaltimer_ns();
        while (*rdy <= scene) {
          __nanosleep(200);
          if (globaltimer_ns() - t0 > 2000000000ull) {  // copies are not arriving: never hang the GPU
            ok = 0; if (A.timeout_flag) atomicExch(A.timeout_flag, 1); break;
          }
        }
      }
      ok = __shfl_sync(FULL, ok, 0);
      if (!ok) {
        if (lane == 0) *reinterpret_cast<volatile int *>(&cta->busy[warp]) = 0;
        break;
      }
      __threadfence();
    }
#ifdef TTMPC_PROFILE_STAGE
    const long long t_stage0 = clock64();
#endif
    {
      const int gwarp = blockIdx.x * g.warps_per_block + warp;
      stage_scene(g, sm, A.p + (size_t)scene * g.np, A.dyn_scratch + (size_t)gwarp * DYN_FIELDS * g.Ndyn * g.N, lane);
    }
#ifdef TTMPC_PROFILE_STAGE
    if (lane == 0 && A.eprof) atomicAdd(A.eprof + 9, (unsigned long long)(clock64() - t_stage0));  // staging cycles (slot of the apply timer)
#endif
    hc.enabled = A.helpers != 0 && !hc.timed_out;
    solve_scene<DM>(g, sm, A, scene, lane, hc);
    if (lane == 0) {
      *reinterpret_cast<volatile int *>(&cta->busy[warp]) = 0;
      if (A.run_stats) {
        atomicAdd(A.run_stats, (unsigned long long)(sm.ctx->n_cost + sm.ctx->n_grad));
        atomicAdd(A.run_stats + 1, 1ull);
      }
    }
    __syncwarp();
  }
  // out of scenes: help the CTA-mates that still own one
  if (A.helpers) helper_loop<DM>(g, A, cta, warp, lane);
}



#ifndef TTMPC_SMALL_CODE  // everything below exists once, in the unrolled build
// ------------------------------------------------------------------ dispatch order
// Solve lengths span 50x and a batch ends when its slowest scene does, so scenes that are likely
// to run long should start first.  A cheap, result-neutral predictor: how many points of the
// reference trajectory lie strictly inside a static polygon or inside the bounding circle of a
// dynamic ellipse at the same step (on the synthetic workloads 98 of the 100 longest scenes have
// a non-zero count).  rank_scenes_kernel (one warp per scene, lane = horizon step) computes the
// count and a histogram of min(count, 15); order_scenes_kernel scatters the scene indices by
// class, highest class first.  The solve kernel then takes order[counter++].
constexpr int RANK_CLASSES = 16;
__global__ void __launch_bounds__(128) rank_scenes_kernel(const DevCfg g, const double *__restrict__ p_all,
                                                          int n, int *__restrict__ cls, int *__restrict__ hist) {
  const int scene = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (scene >= n) return;
  const double *p = p_all + (size_t)scene * g.np;
  int cnt = 0;
  if (lane < g.N) {
    const double x = p[g.off_r + 3 * lane], y = p[g.off_r + 3 * lane + 1];
    const double *os = p + g.off_os;
    for (int i = 0; i < g.Nstc; i++) {
      const double *b = os + i * g.nstcobs, *a0 = b + g.ne, *a1 = b + 2 * g.ne;
      bool inside = true, live = false;
      for (int e = 0; e < g.ne; e++) {
        inside = inside && (b[e] - a0[e] * x - a1[e] * y > 0.0);
        live = live || a0[e] != 0.0 || a1[e] != 0.0;
      }
      cnt += (inside && live) ? 1 : 0;
    }
    const double *od = p + g.off_od;
    for (int j = 0; j < g.Ndyn; j++) {
      const double *e = od + ((size_t)j * g.N + lane) * 6;
      const double dx = x - e[0], dy = y - e[1], r = fmax(e[2], e[3]) + g.margin;
      cnt += (e[5] > 0.0 && r > g.margin && dx * dx + dy * dy < r * r) ? 1 : 0;
    }
  }
  cnt = __reduce_add_sync(FULL, cnt);
  if (lane == 0) {
    const int c = cnt < RANK_CLASSES - 1 ? cnt : RANK_CLASSES - 1;
    cls[scene] = c;
    atomicAdd(hist + c, 1);
  }
}
__global__ void __launch_bounds__(256) order_scenes_kernel(int n, const int *__restrict__ cls,
                                                           const int *__restrict__ hist, int *__restrict__ cursor,
                                                           int *__restrict__ order) {
  const int scene = blockIdx.x * blockDim.x + threadIdx.x;
  if (scene >= n) return;
  const int c = cls[scene];
  int base = 0;
  for (int k = RANK_CLASSES - 1; k > c; k--) base += hist[k];
  order[base + atomicAdd(cursor + c, 1)] = scene;
}

// ------------------------------------------------------------------ batched evaluation
template <class DM>
__global__ void __launch_bounds__(128) eval_kernel(const __grid_constant__ DevCfg g,
                                                   const __grid_constant__ EvalArgs A) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const WarpSmem sm = carve<DM>(smem_raw + (size_t)warp * g.smem_per_warp, g);  // no CtaHelp table here
  const int gwarp = blockIdx.x * g.warps_per_block + warp;
  const int nwarps = gridDim.x * g.warps_per_block;
  double *dyn = A.dyn_scratch + (size_t)gwarp * DYN_FIELDS * g.Ndyn * g.N;
  const int N = g.N;
  for (int scene = gwarp; scene < A.n_scenes; scene += nwarps) {
    stage_scene(g, sm, A.p + (size_t)scene * g.np, dyn, lane);
    const bool act = lane < N;
    double v = 0.0, w = 0.0, ya = 0.0, yw = 0.0;
    if (act) {
      v = A.u[(size_t)scene * 2 * N + 2 * lane];
      w = A.u[(size_t)scene * 2 * N + 2 * lane + 1];
      if (A.y) { ya = A.y[(size_t)scene * 2 * N + lane]; yw = A.y[(size_t)scene * 2 * N + N + lane]; }
    }
    const double c = A.c ? A.c[scene] : 0.0;
    EvalOut e = eval_psi<DM>(&g, reinterpret_cast<unsigned char *>(sm.ctx), v, w, c, ya, yw, nullptr, true, 0.0);
    const double gv = e.gv, gw = e.gw;
    double vp = __shfl_up_sync(FULL, v, 1), wp = __shfl_up_sync(FULL, w, 1);
    if (lane == 0) { vp = sm.ctx->v_init; wp = sm.ctx->w_init; }
    if (act) {
      if (A.grad) { A.grad[(size_t)scene * 2 * N + 2 * lane] = gv; A.grad[(size_t)scene * 2 * N + 2 * lane + 1] = gw; }
      if (A.F1) {
        A.F1[(size_t)scene * 2 * N + lane] = (v - vp) * g.inv_ts;
        A.F1[(size_t)scene * 2 * N + N + lane] = (w - wp) * g.inv_ts;
      }
    }
    if (A.F2)
      for (int j = lane; j < g.Ndyn; j += 32)
        A.F2[(size_t)scene * g.Ndyn + j] = e.S + (e.any_hard ? sm.D[j] : 0.0);
    if (lane == 0) {
      if (A.f) A.f[scene] = e.f;
      if (A.psi) A.psi[scene] = e.psi;
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------ latency probe (diagnostics)
// One warp, one scene: cycles of a cost-only eval, a gradient eval, a butterfly sum, a
// 10-pair L-BFGS apply and a double division, each averaged over `reps` back-to-back calls.
template <class DM>
__global__ void __launch_bounds__(128, 3) probe_kernel(const __grid_constant__ DevCfg g, const double *p,
                                                       double *dyn, long long *out, int reps,
                                                       int warps) {
  // `warps` warps of every CTA run the same measurement on their own copy of the scene
  // (grid x warps > 1 shows how the latencies change when the SM is shared); block 0 /
  // warp 0 reports
  extern __shared__ __align__(16) unsigned char smem_all[];
  const int lane = threadIdx.x & 31, warp_id = threadIdx.x >> 5;
  if (warp_id >= warps) return;
  unsigned char *smem_raw = smem_all + (size_t)warp_id * g.smem_per_warp;
  const WarpSmem sm = carve<DM>(smem_raw, g);
  stage_scene(g, sm, p, dyn, lane);
  {  // desynchronise the warps
    const long long until = clock64() + ((blockIdx.x * 4 + warp_id) * 7919) % 9000;
    while (clock64() < until) {}
  }
  double v = lane < g.N ? 0.8 : 0.0, w = lane < g.N ? 0.05 : 0.0, acc = 0.0;
  long long t0 = clock64();
  for (int i = 0; i < reps; i++) {
    EvalOut e = eval_psi<DM>(&g, smem_raw, v, w, 10.0, 0.0, 0.0, nullptr, false, 0.0);
    v += 1e-9 * e.psi * 0.0 + 1e-12;
    acc += e.psi;
  }
  long long t1 = clock64();
  for (int i = 0; i < reps; i++) {
    EvalOut e = eval_psi<DM>(&g, smem_raw, v, w, 10.0, 0.0, 0.0, nullptr, true, 1e-3);
    v += e.gv * 1e-300; w += e.gw * 1e-300;
    acc += e.psi;
  }
  long long t2 = clock64();
  for (int i = 0; i < reps; i++) acc = wsum(acc * 1e-3 + v);
  long long t3 = clock64();
  Lane z; Uni U;
  U.pc = &sm.ctx->pc;
  z.d0 = v; z.d1 = w; U.pc->lb_active = g.mem; U.pc->lb_head = 0; U.pc->lb_gamma = 0.7;
  if (lane < g.N)
    for (int k = 0; k <= g.mem; k++) {
      sm.lbs[k * g.N + lane] = make_double2(0.01 * (k + 1), 0.02);
      sm.lby[k * g.N + lane] = make_double2(0.03, 0.01 * (k + 2));
    }
  if (lane <= g.mem) sm.rho[lane] = 0.5;
  __syncwarp();
  for (int i = 0; i < reps; i++) { lbfgs_apply<DM>(g, sm, z, U, lane); z.d0 *= 1e-3; z.d1 *= 1e-3; }
  long long t4 = clock64();
  double d = 1.0 + acc * 1e-30;
  for (int i = 0; i < reps; i++) d = 1.0 / (d + 0.5);
  long long t5 = clock64();
  for (int i = 0; i < reps; i++) d = sqrt(d + 0.5);
  long long t6 = clock64();
  double f = d;
  for (int i = 0; i < reps; i++) f = fma(f, 0.999, 1e-3);
  long long t7 = clock64();
  if (lane == 0 && blockIdx.x == 0 && warp_id == 0) {
    out[0] = (t1 - t0) / reps; out[1] = (t2 - t1) / reps; out[2] = (t3 - t2) / reps;
    out[3] = (t4 - t3) / reps; out[4] = (t5 - t4) / reps; out[5] = (t6 - t5) / reps;
    out[6] = (t7 - t6) / reps; out[7] = (long long)(acc + z.d0 + d + f);
  }
}

// ------------------------------------------------------------------ FP64 peak probe
__global__ void fp64_peak_kernel(double *out, int iters) {
  double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5,
         a6 = a0 + 6, a7 = a0 + 7;
  const double b = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
    a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

#endif  // !TTMPC_SMALL_CODE
}  // namespace ttmpc

// ------------------------------------------------------------------ launch helpers (host)
namespace ttmpc {

static bool is_default_dims(const DevCfg &g) {
  return g.N == 20 && g.Nother == 10 && g.Nstc == 10 && g.ne == 4 && g.Ndyn == 15 && g.mem == 10;
}

// cudaFuncSetAttribute / occupancy queries cost microseconds each and used to run on every call
// (they matter for the one-scene latency path): both are cached per (kernel, device).
static std::mutex g_attr_mu;
static std::map<std::pair<const void *, int>, size_t> g_attr_smem;
static std::map<std::tuple<const void *, int, int, size_t>, int> g_attr_occ;
template <class K>
static cudaError_t set_smem(K kernel, size_t smem) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const auto key = std::make_pair(reinterpret_cast<const void *>(kernel), dev);
  {
    std::lock_guard<std::mutex> lk(g_attr_mu);
    auto it = g_attr_smem.find(key);
    if (it != g_attr_smem.end() && it->second >= smem) return cudaSuccess;
  }
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) {
    std::lock_guard<std::mutex> lk(g_attr_mu);
    size_t &v = g_attr_smem[key];
    if (v < smem) v = smem;
  }
  return e;
}
template <class K>
static cudaError_t cached_occupancy(K kernel, int block, size_t smem, int *blocks_per_sm) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const auto key = std::make_tuple(reinterpret_cast<const void *>(kernel), dev, block, smem);
  {
    std::lock_guard<std::mutex> lk(g_attr_mu);
    auto it = g_attr_occ.find(key);
    if (it != g_attr_occ.end()) { *blocks_per_sm = it->second; return cudaSuccess; }
  }
  if ((e = set_smem(kernel, smem)) != cudaSuccess) return e;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, kernel, block, smem);
  if (e == cudaSuccess) {
    std::lock_guard<std::mutex> lk(g_attr_mu);
    g_attr_occ[key] = *blocks_per_sm;
  }
  return e;
}

// Shapes with a fully specialised solve kernel: config/mpc_default.yaml and the horizon /
// obstacle-count sweep of BASELINE configs[4]; everything else runs the run-time-dimension build.
//        N  Nother Nstc ne Ndyn mem
#define TTMPC_SOLVE_SHAPES(X) \
  X(20, 10, 10, 4, 15, 10)    \
  X(10, 10, 10, 4, 15, 10)    \
  X(32, 10, 10, 4, 15, 10)    \
  X(20, 10, 4, 4, 4, 10)      \
  X(20, 10, 20, 4, 30, 10)
template <class F>
static cudaError_t with_solve_dims(const DevCfg &g, F &&f) {
#define X(n, no, ns, e, nd, m) \
  if (g.N == n && g.Nother == no && g.Nstc == ns && g.ne == e && g.Ndyn == nd && g.mem == m) return f(Dims<n, no, ns, e, nd, m>{});
  TTMPC_SOLVE_SHAPES(X)
#undef X
  return f(DimsRuntime{});
}

cudaError_t launch_solve(const DevCfg &g, const SolveArgs &A, int grid, cudaStream_t st) {
  const size_t smem = (size_t)g.smem_per_warp * g.warps_per_block + sizeof(CtaHelp);
  return with_solve_dims(g, [&](auto dm) -> cudaError_t {
    using DM = decltype(dm);
    cudaError_t e;
    if ((e = set_smem(solve_kernel<DM>, smem)) != cudaSuccess) return e;
    solve_kernel<DM><<<grid, g.warps_per_block * 32, smem, st>>>(g, A);
    return cudaGetLastError();
  });
}
// resident blocks per SM of the kernel launch_solve would pick
cudaError_t solve_occupancy(const DevCfg &g, int *blocks_per_sm) {
  const size_t smem = (size_t)g.smem_per_warp * g.warps_per_block + sizeof(CtaHelp);
  return with_solve_dims(g, [&](auto dm) -> cudaError_t {
    using DM = decltype(dm);
    return cached_occupancy(solve_kernel<DM>, g.warps_per_block * 32, smem, blocks_per_sm);
  });
}
#ifndef TTMPC_SMALL_CODE
// scratch: cls[n] | hist[16] | cursor[16]   (ints; hist and cursor zeroed here)
cudaError_t launch_rank_scenes(const DevCfg &g, const double *p, int n, int *scratch, int *order,
                               cudaStream_t st) {
  int *cls = scratch, *hist = scratch + n, *cursor = hist + RANK_CLASSES;
  cudaError_t e = cudaMemsetAsync(hist, 0, 2 * RANK_CLASSES * sizeof(int), st);
  if (e != cudaSuccess) return e;
  rank_scenes_kernel<<<(n + 3) / 4, 128, 0, st>>>(g, p, n, cls, hist);
  order_scenes_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, cls, hist, cursor, order);
  return cudaGetLastError();
}
cudaError_t launch_eval(const DevCfg &g, const EvalArgs &A, int grid, cudaStream_t st) {
  const size_t smem = (size_t)g.smem_per_warp * g.warps_per_block;
  cudaError_t e;
  if (is_default_dims(g)) {
    if ((e = set_smem(eval_kernel<DimsDefault>, smem)) != cudaSuccess) return e;
    eval_kernel<DimsDefault><<<grid, g.warps_per_block * 32, smem, st>>>(g, A);
  } else {
    if ((e = set_smem(eval_kernel<DimsRuntime>, smem)) != cudaSuccess) return e;
    eval_kernel<DimsRuntime><<<grid, g.warps_per_block * 32, smem, st>>>(g, A);
  }
  return cudaGetLastError();
}
cudaError_t launch_probe(const DevCfg &g, const double *p, double *dyn, long long *out, int reps,
                         cudaStream_t st) {
  const size_t smem = (size_t)g.smem_per_warp * g.warps_per_block;
  cudaError_t e;
  int grid = 1, warps = 1;  // diagnostics: TTMPC_PROBE_GRID x TTMPC_PROBE_WARPS warps run the probe together
  if (const char *s = std::getenv("TTMPC_PROBE_GRID")) grid = std::max(1, std::atoi(s));
  if (const char *s = std::getenv("TTMPC_PROBE_WARPS")) warps = std::min(std::max(1, std::atoi(s)), g.warps_per_block);
  if (is_default_dims(g)) {
    if ((e = set_smem(probe_kernel<DimsDefault>, smem)) != cudaSuccess) return e;
    probe_kernel<DimsDefault><<<grid, 128, smem, st>>>(g, p, dyn, out, reps, warps);
  } else {
    if ((e = set_smem(probe_kernel<DimsRuntime>, smem)) != cudaSuccess) return e;
    probe_kernel<DimsRuntime><<<grid, 128, smem, st>>>(g, p, dyn, out, reps, warps);
  }
  return cudaGetLastError();
}
cudaError_t launch_fp64_peak(double *out, int blocks, int threads, int iters, cudaStream_t st) {
  fp64_peak_kernel<<<blocks, threads, 0, st>>>(out, iters);
  return cudaGetLastError();
}

#endif  // !TTMPC_SMALL_CODE
}  // namespace ttmpc
