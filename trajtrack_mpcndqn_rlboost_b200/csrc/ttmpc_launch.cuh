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
  unsigned long long *eprof;  // [10] eval section cycles (diagnostic build) or null
  int helpers;          // 1: warps that run out of scenes help their CTA-mates (tail of a batch)
  int *timeout_flag;    // set to 1 if a wait on `ready` timed out (host then re-runs unstreamed)
  const int *ready;     // optional: number of scenes whose parameters have landed in d_p
                        // (host path streams p in chunks while the kernel already runs)
  unsigned long long *stats;  // [4]: cost evals, grad evals, dyn bodies, panoc iterations
  unsigned long long *run_stats;  // [2]: evaluations and count of finished scenes (early helpers) or null
  int n_scenes;
  int use_u0, use_y0;
};

struct EvalArgs {
  const double *p, *u, *c, *y;
  double *f, *F1, *F2, *psi, *grad;
  double *dyn_scratch;
  int n_scenes;
};

cudaError_t launch_solve(const DevCfg &g, const SolveArgs &A, int grid, cudaStream_t st);
// the rolled-loop build of the same kernel (ttmpc_solve_small.cu): bulk batches
cudaError_t launch_solve_small(const DevCfg &g, const SolveArgs &A, int grid, cudaStream_t st);
cudaError_t launch_rank_scenes(const DevCfg &g, const double *p, int n, int *scratch, int *order,
                               cudaStream_t st);
cudaError_t launch_eval(const DevCfg &g, const EvalArgs &A, int grid, cudaStream_t st);
cudaError_t solve_occupancy(const DevCfg &g, int *blocks_per_sm);
cudaError_t solve_occupancy_small(const DevCfg &g, int *blocks_per_sm);  // the rolled build
cudaError_t launch_probe(const DevCfg &g, const double *p, double *dyn, long long *out, int reps,
                         cudaStream_t st);
// fleet step (ttmpc_fleet.cu)
struct FleetDims { int N, np, n_other, n_stc, n_dyn; double ts; };
cudaError_t launch_fleet_pack(const ttmpc_fleet &f, const FleetDims &d, double *p, cudaStream_t st);
cudaError_t launch_fleet_advance(const ttmpc_fleet &f, const FleetDims &d, const double *u,
                                 const int *exit_status, cudaStream_t st);
cudaError_t launch_fp64_peak(double *out, int blocks, int threads, int iters, cudaStream_t st);

}  // namespace ttmpc
