// ttmpc_launch.cuh -- kernel argument blocks and host launch helpers shared by
// ttmpc_solve.cu (kernels) and ttmpc_api.cu (C-ABI).
#pragma once
#include "ttmpc_device.cuh"

namespace ttmpc {

struct SolveArgs {
  const double *p;      // [n][np]
  const double *c0;     // [n] or null
  double *u;            // [n][2N] in/out
  double *y;            // [n][2N] in/out or null
  double *cost, *last_fpr, *f1_infeas, *f2_norm, *penalty;
  int *exit_status, *outer_iters, *inner_iters;
  double *pred_states;  // [n][N][3] or null
  long long *evals;     // [n][4] or null
  double *dyn_scratch;  // [total_warps][DYN_FIELDS*Ndyn*N]
  int *work_counter;    // dynamic scene queue
  const int *order;     // optional dispatch order (likely-long scenes first) or null
  int helpers;          // 1: warps that run out of scenes help their CTA-mates (tail of a batch)
  int *timeout_flag;    // set to 1 if a wait on `ready` timed out (host then re-runs unstreamed)
  const int *ready;     // optional: number of scenes whose parameters have landed in d_p
                        // (host path streams p in chunks while the kernel already runs)
  unsigned long long *stats;  // [4]: cost evals, grad evals, dyn bodies, panoc iterations
  unsigned long long *run_stats;  // [2]: evaluations and count of finished scenes (early helpers) or null
  const int *skip_status;  // [n] or null: scenes whose entry is non-zero are not solved (fleet
                           // status of stopped robots); their result rows are left untouched
  int n_scenes;
  int use_u0, use_y0;
};

struct EvalArgs {
  const double *p, *u, *c, *y;
  double *f, *F1, *F2, *psi, *grad;
  double *dyn_scratch;
  int n_scenes;
};

// rolled: solve_kernel_small (bulk batches) instead of solve_kernel, see ttmpc_solve.cu
cudaError_t launch_solve(const DevCfg &g, const SolveArgs &A, int grid, bool rolled, cudaStream_t st);
cudaError_t launch_rank_scenes(const DevCfg &g, const double *p, int n, int *scratch, int *order,
                               cudaStream_t st);
cudaError_t launch_eval(const DevCfg &g, const EvalArgs &A, int grid, cudaStream_t st);
cudaError_t solve_occupancy(const DevCfg &g, bool rolled, int *blocks_per_sm);
// fleet step (ttmpc_fleet.cu)
struct FleetDims { int N, np, n_other, n_stc, n_dyn; double ts; };
// prev_u: the previous step's solutions, required when warm_exit != null or action_steps > 1
// (the goal test then reads their first control).  warm_exit != null: warm start -- prev_u is
// shifted in place into the initial guess of every robot that is RUNNING after the goal test.
// tasks != null with max_tasks > 0: REACHED robots take their next queued task (checked by the API).
cudaError_t launch_fleet_pack(const ttmpc_fleet &f, const FleetDims &d, double *p, double *prev_u,
                              const int *warm_exit, const ttmpc_fleet_tasks *tasks, cudaStream_t st);
cudaError_t launch_fleet_advance(const ttmpc_fleet &f, const FleetDims &d, const double *u,
                                 const int *exit_status, cudaStream_t st);
cudaError_t launch_fleet_monitor(const ttmpc_fleet &f, const ttmpc_fleet_monitor &m, cudaStream_t st);
// K = Nstcobs (<= 32), ns = nstcobs
cudaError_t launch_fleet_world_select(const ttmpc_fleet &f, const ttmpc_fleet_world &w, int K, int ns,
                                      double *stc_out, int *slot_poly, int *n_reach, cudaStream_t st);
cudaError_t launch_fp64_peak(double *out, int blocks, int threads, int iters, cudaStream_t st);

}  // namespace ttmpc
