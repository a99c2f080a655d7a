/*
 * ttmpc.h -- C-ABI of the B200-native batched NMPC planner + DQN companion.
 *
 * This is the drop-in boundary for ONE path of Woodenonez/TrajTrack-MPCnDQN-RLBoost:
 * the call that the reference makes into its OpEn-generated (Rust, PyO3) solver
 *
 *     solution = self.solver.run(parameters, initial_guess)
 *         -- src/mpc_traj_tracker/trajectory_generator.py:284
 *     class Solver: def run(self, p, initial_guess, initial_lagrange_multipliers,
 *                           initial_penalty) -> SolverStatus
 *         -- src/mpc_traj_tracker/trajectory_generator.py:27-29
 *
 * and, for the DQN-boosted loop, the observation + policy call
 *
 *     obsv['external'] = SectorAndRayObservation.external_obs()
 *         -- src/pkg_dqn/environment/components/ext_obsv_sector_and_ray.py:33-83
 *     action_index, _ = model.predict(obsv, deterministic=True)
 *         -- src/main.py:148 (SB3 DQN MultiInputPolicy, net_arch [16,16])
 *
 * Everything is plain pointers and sizes.  No torch types, no C++ types.
 * Pointers named d_* are DEVICE pointers, h_* are HOST pointers.
 * All entry points return 0 on success, a negative ttmpc error code otherwise;
 * ttmpc_last_error() gives a human-readable string for the calling thread.
 *
 * The packed parameter vector p of one scene is laid out exactly as the
 * reference assembles it (trajectory_generator.py:251-254, mpc_generator.py:175-184):
 *
 *   s     [2*ns+nu]              x y theta | x_goal y_goal theta_goal | v_init w_init
 *   q     [nq = 10]              qpos qvel qtheta rv rw qN qthetaN qrpd acc_pen wacc_pen
 *   r     [ns*N + N]             (x y theta) * N reference states, then N speed refs
 *   c     [ns*N*Nother]          predicted states of other robots, robot-major
 *   o_s   [Nstcobs*nstcobs]      per obstacle: b[ne] a0[ne] a1[ne]   (ne = nstcobs/3)
 *   o_d   [Ndynobs*ndynobs*N]    per obstacle, per step: cx cy rx ry angle alpha
 *   q_stc [N]                    static-obstacle weights (unused by the cost, kept)
 *   q_dyn [N]                    dynamic-obstacle soft weights
 *
 * Batches are scene-major: p[scene][np], u[scene][nu*N], y[scene][2*N].
 */
#ifndef TTMPC_H
#define TTMPC_H

#ifdef __cplusplus
extern "C" {
#endif

#define TTMPC_VERSION 102

/* exit_status codes; names are the strings the OpEn python binding returns
 * (format!("{:?}", ExitStatus)), which the reference matches against
 * config.bad_exit_codes (config/mpc_default.yaml:58).  */
enum {
  TTMPC_CONVERGED = 0,                 /* "Converged"              */
  TTMPC_NOT_CONVERGED_ITERATIONS = 1,  /* "NotConvergedIterations" */
  TTMPC_NOT_CONVERGED_OUT_OF_TIME = 2, /* "NotConvergedOutOfTime"  */
  TTMPC_NOT_FINITE = 3                 /* SolverError::NotFiniteComputation: the
                                          binding returns None -> reference raises */
};

enum {
  TTMPC_OK = 0,
  TTMPC_ERR_BAD_CONFIG = -1,
  TTMPC_ERR_BAD_ARG = -2,
  TTMPC_ERR_CUDA = -3,
  TTMPC_ERR_UNSUPPORTED = -4
};

/* Problem + solver configuration.
 * Problem fields mirror config/mpc_default.yaml; solver fields mirror
 * opengen.config.SolverConfiguration as used at mpc_generator.py:268-276
 * (initial_penalty 10, everything else opengen 0.7.1 defaults).          */
typedef struct ttmpc_config {
  /* dimensions */
  int N_hor;    /* horizon, 1..32 (one lane per step)                  */
  int nu;       /* must be 2 (v, omega)                                */
  int ns;       /* must be 3 (x, y, theta)                             */
  int nq;       /* must be 10                                          */
  int Nother;   /* other-robot slots                                   */
  int Nstcobs;  /* static obstacle slots                               */
  int nstcobs;  /* doubles per static obstacle = 3*edges, edges<=8     */
  int Ndynobs;  /* dynamic obstacle slots                              */
  int ndynobs;  /* must be 6                                           */
  int _pad0;
  /* model */
  double ts;
  double vehicle_width;  /* fleet safe distance                         */
  double social_margin;  /* soft-ellipse inflation                      */
  double lin_vel_min, lin_vel_max, ang_vel_max; /* box on u              */
  double lin_acc_min, lin_acc_max, ang_acc_max; /* set C of the ALM map  */
  /* solver (OpEn) */
  double tolerance;              /* epsilon, 1e-4                        */
  double initial_tolerance;      /* initial inner AKKT tolerance, 1e-4   */
  double delta_tolerance;        /* constraints tolerance, 1e-4          */
  double initial_penalty;        /* 10 (mpc_generator.py:269)            */
  double penalty_update_factor;  /* 5                                    */
  double inner_tolerance_update_factor; /* 0.1                           */
  double sufficient_decrease_coeff;     /* 0.1                           */
  int lbfgs_memory;              /* 10, max 16                           */
  int max_inner_iterations;      /* 500                                  */
  int max_outer_iterations;      /* 10                                   */
  int max_duration_ms;           /* wall-clock budget of ONE scene's solve, 5000 =
                                    MAX_SOVLER_TIME (mpc_generator.py:22,270: with_max_duration_micros);
                                    0 = no limit.  Measured on the device from the moment the scene's
                                    solve starts; checked where OpEn checks it (after every PANOC step,
                                    before every outer iteration) -> TTMPC_NOT_CONVERGED_OUT_OF_TIME.
                                    Like in the reference, a solve that hits the budget is not
                                    reproducible; the CPU oracle ignores the field.               */
} ttmpc_config;

/* Fill cfg with config/mpc_default.yaml + opengen defaults. */
void ttmpc_default_config(ttmpc_config *cfg);
/* Number of doubles in one packed parameter vector / decision vector / F1 / F2. */
int ttmpc_num_params(const ttmpc_config *cfg);
int ttmpc_num_decision(const ttmpc_config *cfg);
int ttmpc_num_alm(const ttmpc_config *cfg);     /* n1 = 2*N_hor */
int ttmpc_num_penalty(const ttmpc_config *cfg); /* n2 = Ndynobs */
const char *ttmpc_last_error(void);
const char *ttmpc_exit_status_name(int code);
int ttmpc_version(void);
/* The CUDA device of the CALLING THREAD (cudaSetDevice / cudaGetDevice): every entry point works on
 * the calling thread's current device, so a host thread that serves GPU k calls ttmpc_set_device(k)
 * once before its first solve (new threads start on device 0).                                  */
int ttmpc_set_device(int device);
int ttmpc_get_device(int *device);

/* Per-scene outputs of a batched solve.  Any pointer may be NULL (skipped)
 * except u.  Mirrors the fields of OpEn's python OptimizerSolution that the
 * reference reads (trajectory_generator.py:286-289) plus the diagnostics.  */
typedef struct ttmpc_result {
  double *u;            /* [n][nu*N]  in: initial guess (see use_u0), out: solution */
  double *cost;         /* [n]  f(u*) (psi with c = 0)                              */
  int *exit_status;     /* [n]                                                      */
  int *outer_iters;     /* [n]                                                      */
  int *inner_iters;     /* [n]                                                      */
  double *last_fpr;     /* [n]  last_problem_norm_fpr                               */
  double *f1_infeas;    /* [n]  delta_y_norm / c                                    */
  double *f2_norm;      /* [n]                                                      */
  double *penalty;      /* [n]  final c                                             */
  double *y;            /* [n][2*N] in: initial multipliers (see use_y0), out: final */
  double *pred_states;  /* [n][N][ns] rollout of u* from p.s, i.e. from the state the solve STARTED in.
                           NOTE: the reference's list (trajectory_generator.py:296-301) starts from the
                           state AFTER u[0] was applied (taken_states[-1]) and re-applies u from there, so
                           it is this rollout shifted by one step; the Python TrajectoryGenerator mirror
                           rebuilds the reference's list on the host from u.                          */
  long long *evals;     /* [n][4] cost-only evals, cost+gradient evals, solve time [ns],
                           solve start [ns, %globaltimer] (diagnostics)              */
} ttmpc_result;

/* ------------------------------------------------------------------------
 * Batched NMPC solve, device-resident.  All pointers in res and d_p are
 * device pointers.  Asynchronous on `stream` (a cudaStream_t passed as void*).
 *   use_u0 = 0: initial guess is all-zero, like solver.run(p) with
 *               initial_guess=None; res->u is output only.
 *   use_y0 = 0: multipliers start at zero.  (The reference's Solver object
 *               keeps them between run() calls; the host mirror does that.)
 *   d_c0      : optional per-scene initial penalty (NULL -> cfg value).
 * Batches in flight: solves issued on the SAME stream run one after the other;
 * solves issued on DIFFERENT streams (each with its own result buffers; 16 stream
 * bindings per device, a 17th stream drains the device once and rebinds) may overlap -- every stream has its own scene queue and scratch
 * tables inside the library, and the CTAs of the next batch become resident as
 * the CTAs of the running one drain.  Results do not depend on what else runs.
 * ------------------------------------------------------------------------ */
int ttmpc_solve_batch_device(const ttmpc_config *cfg, int n_scenes,
                             const double *d_p, int use_u0, int use_y0,
                             const double *d_c0, const ttmpc_result *res,
                             void *stream);

/* Same call with HOST buffers: stages p/u/y through pinned memory, launches,
 * copies results back, synchronises.  This is what the python Solver.run
 * mirror and the `e2e` bench leg use.  Thread-safe: calls from several host
 * threads each take their own staging buffers / streams (8 sets per device, a
 * ninth caller waits) and overlap on the GPU.                              */
int ttmpc_solve_batch_host(const ttmpc_config *cfg, int n_scenes,
                           const double *h_p, int use_u0, int use_y0,
                           const double *h_c0, const ttmpc_result *res);

/* Evaluate the problem functions on device for a batch (testing / parity):
 * f, F1 [n][2N], F2 [n][Ndynobs], and psi/grad psi at xi = (c, y).
 * Any output may be NULL.  d_c [n], d_y [n][2N] may be NULL (c=0, y=0).   */
int ttmpc_eval_batch_device(const ttmpc_config *cfg, int n_scenes,
                            const double *d_p, const double *d_u,
                            const double *d_c, const double *d_y, double *d_f,
                            double *d_F1, double *d_F2, double *d_psi,
                            double *d_grad, void *stream);
int ttmpc_eval_batch_host(const ttmpc_config *cfg, int n_scenes,
                          const double *h_p, const double *h_u,
                          const double *h_c, const double *h_y, double *h_f,
                          double *h_F1, double *h_F2, double *h_psi,
                          double *h_grad);

/* ------------------------------------------------------------------------
 * DQN companion: sector+ray ("lidar") observation against the obstacle set,
 * then Q-network inference and argmax, one environment per warp.
 *
 * Geometry of one env (all fp64, world frame, already padded as the reference
 * pads them: obstacle.py:158-163,248-254):
 *   polygons: n_poly closed rings, ring i has poly_nv[i] vertices stored at
 *             poly_xy[poly_off[i] .. ], (x,y) pairs.  is_solid[i] != 0 for an
 *             obstacle (filled Polygon), 0 for the boundary ring (LineString).
 * Batched layout: fixed capacity per env: max_poly rings, max_vert vertices.
 * ------------------------------------------------------------------------ */
typedef struct ttdqn_scene_layout {
  int num_segments; /* 8 (rays_reward1.py:20); 3..16, else TTMPC_ERR_BAD_CONFIG */
  int max_poly;     /* ring slots per env                                  */
  int max_vert;     /* vertex slots per env (sum over rings)               */
  int n_internal;   /* 14 internal observation entries                     */
  int use_memory;   /* 1: external obs = [seg, ray, old_seg, old_ray]      */
  int _pad;
  double ray_length;   /* L = 1000 (ext_obsv_sector_and_ray.py:34): the sector
                        * triangles reach L, the centre rays are L long     */
  double max_distance; /* normalize_distance max_distance = 10 (utils.py:10) */
} ttdqn_scene_layout;

/* Q-network weights, fp32 row-major [out][in] like torch.nn.Linear.
 * Input is concat(external[4*num_segments or 2*num_segments], internal[n_internal])
 * (SB3 CombinedExtractor concatenates Dict keys in sorted order:
 *  'external' then 'internal').                                           */
typedef struct ttdqn_qnet {
  int n_in, n_h1, n_h2, n_out; /* 46, 16, 16, 9; n_h1, n_h2 1..256, n_out 1..64 */
  const float *w0, *b0, *w1, *b1, *w2, *b2;
} ttdqn_qnet;

void ttdqn_default_layout(ttdqn_scene_layout *lay);
/* Last failure of a ttdqn_* entry point on the calling thread (the same text is also what
 * ttmpc_last_error() returns, so one query serves the whole library).                     */
const char *ttdqn_last_error(void);

/* Device-resident batched observe + act.
 *   d_agent    [n][3]   x y theta (fp64)
 *   d_poly_xy  [n][max_vert][2], d_poly_off [n][max_poly+1] (prefix offsets),
 *   d_is_solid [n][max_poly], d_n_poly [n]
 *   d_internal [n][n_internal] fp32 internal observation
 *   d_old_ext  [n][2*num_segments] fp32 in/out memory of previous (seg, ray) obs
 *              (NULL when use_memory == 0)
 * outputs (any may be NULL): d_ext [n][n_ext] fp32, d_q [n][n_out] fp32,
 *   d_action [n] int32, d_seg_dist / d_ray_dist [n][num_segments] fp64 raw distances.
 * qnet pointers are device pointers.
 * Sector i is the triangle with apex at the agent and far vertices at ray_length, at angles
 * theta + i * 2 pi / num_segments -+ pi / num_segments; its ray is the centre line, ray_length long.
 * A ring's ray hit counts only in the sectors whose triangle the ring meets (the reference
 * intersects the ray only when the sector intersection is non-empty).
 * Q-network: 16-wide hidden layers with n_out <= 16 and n_in <= 248 run on the tensor cores (an
 * exact three-way TF32 split of every operand); every other shape runs on the FMA pipe with fp64
 * accumulation and one rounding to fp32 per neuron.  The FMA path keeps all weights in shared
 * memory: 4 * (n_in*n_h1 + n_h1 + n_h1*n_h2 + n_h2 + n_h2*n_out + n_out) bytes rounded up to 16,
 * plus 4 warps x (1024 + 4 * (n_in + n_h1 + n_h2 + n_out + 4) rounded up to 16) of scratch.  More
 * than the device's opt-in shared memory per block -> TTMPC_ERR_UNSUPPORTED before any device work
 * (ttdqn_last_error names both numbers).                                  */
int ttdqn_observe_act_device(const ttdqn_scene_layout *lay, const ttdqn_qnet *qnet,
                             int n_envs, const double *d_agent,
                             const double *d_poly_xy, const int *d_poly_off,
                             const int *d_is_solid, const int *d_n_poly,
                             const float *d_internal, float *d_old_ext,
                             float *d_ext, float *d_q, int *d_action,
                             double *d_seg_dist, double *d_ray_dist, void *stream);
int ttdqn_observe_act_host(const ttdqn_scene_layout *lay, const ttdqn_qnet *qnet,
                           int n_envs, const double *h_agent,
                           const double *h_poly_xy, const int *h_poly_off,
                           const int *h_is_solid, const int *h_n_poly,
                           const float *h_internal, float *h_old_ext,
                           float *h_ext, float *h_q, int *h_action,
                           double *h_seg_dist, double *h_ray_dist);

/* Moving obstacles in the observation: n_live solid rings per env, each a vertex template placed
 * at its obstacle's current centre.  Ring o of env e has vertices
 *   centre[e][o] + shape_xy[e or 0][o][v],  v < shape_nv[e or 0][o]
 * (one fp64 add per coordinate).  Like a static solid ring it is even-odd filled: an agent inside
 * one gives 0 in every sector and on every ray.  A template with shape_nv < 3 is not seen; counts
 * above max_pv are read as max_pv.  All arrays are device pointers.                               */
typedef struct ttdqn_moving {
  int n_live;              /* moving obstacles per env, >= 0                                   */
  int max_pv;              /* vertex slots per template, 3..32                                 */
  int shape_shared;        /* != 0: one template block for every env                           */
  int _pad;
  const double *centre;    /* [n][n_live][2] current centres, e.g. ttmpc_fleet.dyn_cur         */
  const double *shape_xy;  /* [n or 1][n_live][max_pv][2] vertex offsets from the centre       */
  const int *shape_nv;     /* [n or 1][n_live] vertex counts (< 3: not seen)                   */
} ttdqn_moving;
/* ttdqn_observe_act_device with the moving rings of mv.  The result equals that of
 * ttdqn_observe_act_device given the same rings (centre + offset) appended as static solid rings,
 * bit for bit; mv == NULL or n_live == 0 computes exactly what ttdqn_observe_act_device computes.
 * n_live < 0, max_pv outside 3..32 or a NULL array with n_live > 0 -> TTMPC_ERR_BAD_ARG before
 * any device work. */
int ttdqn_observe_act_moving_device(const ttdqn_scene_layout *lay, const ttdqn_qnet *qnet,
                                    int n_envs, const double *d_agent,
                                    const double *d_poly_xy, const int *d_poly_off,
                                    const int *d_is_solid, const int *d_n_poly,
                                    const ttdqn_moving *mv,
                                    const float *d_internal, float *d_old_ext,
                                    float *d_ext, float *d_q, int *d_action,
                                    double *d_seg_dist, double *d_ray_dist, void *stream);

/* ------------------------------------------------------------------------
 * Fleet step: the caller side of the solve, batched on the device.
 *
 * One control step of n independent robots, each following the reference's
 * InterfaceMpc.get_action -> TrajectoryGenerator.run_step sequence
 * (src/interface_mpc.py:80-92, src/mpc_traj_tracker/trajectory_generator.py:203-274):
 *
 *   pack    : termination test (check_termination_condition, :158-164), closest point of
 *             the global reference trajectory in the window [idx-k, idx+5k) (k = action_steps)
 *             and the N reference states from there (get_local_ref_traj, :203-230), speed
 *             reference from the distance to the goal (:248-255), dynamic-obstacle rows
 *             extrapolated from two consecutive positions (main.py:80-89,
 *             est_dyn_obs_positions), and the packed parameter vector in the block
 *             order of :257-260.
 *   solve   : ttmpc_solve_batch_device.
 *   advance : state <- unicycle RK4 step with u[k-1] (run_solver, :291-294;
 *             motion_model.py:153-176), last action, solver failure flag
 *             (NotFiniteComputation -> the reference raises), obstacle positions moved by
 *             their per-step displacement.
 *
 * All pointers are device pointers unless the struct member says otherwise; in/out
 * members persist between steps, so K steps run without touching the host.
 * ------------------------------------------------------------------------ */
enum {
  TTMPC_FLEET_RUNNING = 0,  /* get_action returned an action                      */
  TTMPC_FLEET_REACHED = 1,  /* check_termination_condition: get_action -> None    */
  TTMPC_FLEET_FAILED = 2,   /* solver error (the reference raises RuntimeError)   */
  TTMPC_FLEET_BAD_TASK = 3, /* ttmpc_fleet_step_tasks_device: the task taken next cannot be
                               driven (see ttmpc_fleet_tasks); the robot stops       */
  TTMPC_FLEET_COLLIDED = 4  /* ttmpc_fleet_monitor_device with stop_on_contact: the robot
                               touched an obstacle while RUNNING; the robot stops    */
};
/* ttmpc_fleet.options: bit mask of opt-in behaviours of ttmpc_fleet_step_device (0 = none; the
 * pack and advance entry points ignore it).  Other bits -> TTMPC_ERR_BAD_ARG.                  */
enum {
  /* Start the solve of every robot that is RUNNING after this step's goal test from its previous
   * solution shifted by the k = action_steps controls it applied, u'[j] = u[j+k] for j < N-k and
   * u'[j] = u[N-1] otherwise, if that solve's exit status was TTMPC_CONVERGED, and from zeros
   * otherwise (run_step's initial_guess).
   * The previous step's outputs are read from res->u and res->exit_status, which must therefore
   * hold zeros before the first step.  Multipliers still follow use_y0.                         */
  TTMPC_FLEET_WARM_START = 1,
  /* Solve only the robots that are RUNNING (get_action returns None before the solver is called
   * once the goal test holds).  The result rows of the other robots -- every member of res --
   * keep the values of the last step in which they were solved.                               */
  TTMPC_FLEET_SKIP_STOPPED = 2
};
typedef struct ttmpc_fleet {
  int n;            /* robots                                                         */
  int ref_stride;   /* rows per robot in ref_traj                                     */
  double *state;    /* [n][3] x y theta, in/out                                       */
  const double *goal;     /* [n][3]  (written by ttmpc_fleet_step_tasks_device)        */
  double *last_u;   /* [n][2] last applied action, in/out (zeros before the first)    */
  int *idx_ref;     /* [n] index into the global reference trajectory, in/out         */
  int *status;      /* [n] TTMPC_FLEET_*, in/out (robots not RUNNING are left alone)  */
  const double *ref_traj; /* [n][ref_stride][3] get_global_ref_traj output; written by
                             ttmpc_fleet_step_tasks_device when a robot takes a task  */
  const int *ref_len;     /* [n] valid rows (written by ttmpc_fleet_step_tasks_device) */
  const double *stc;      /* static half-space rows: [n][Nstcobs*nstcobs], or one
                             shared row block when stc_shared != 0                   */
  int stc_shared;
  int n_dyn_live;   /* moving obstacles described by dyn_cur / dyn_last (<= Ndynobs)  */
  /* config.action_steps = k: controls of one solution a robot applies before the next solve.
   * 1 everywhere; 1..N_hor in ttmpc_fleet_step_device (out of range -> TTMPC_ERR_BAD_ARG; the
   * pack and advance entry points return TTMPC_ERR_UNSUPPORTED for k != 1).  With k > 1:
   *  - run_solver computes each of its k taken states from the state the step started in, with
   *    u[0] .. u[k-1], and continues from the last one; advance therefore takes one RK4 step with
   *    u[k-1], and last_u becomes u[k-1] (past_actions[-1]), which pack puts into p.  The other
   *    taken states are not an output: rebuild them from p[0:3] (that state) and res->u.
   *  - the goal test reads the FIRST control u[0] of the previous solution
   *    (InterfaceMpc._last_action = actions[0]) from res->u, which must therefore hold zeros
   *    before the first step, as for TTMPC_FLEET_WARM_START.
   *  - moving obstacles still move by dyn_disp once per control step, and the dynamic-obstacle
   *    rows still extrapolate from the positions of two consecutive control steps (main.py:80-89).
   *  - res->pred_states stays the rollout of u* from p.s.                                       */
  int action_steps;
  int options;      /* TTMPC_FLEET_* bit mask of the step; C callers must zero it         */
  const double *other;    /* [n][ns*N*Nother] other-robot predictions or NULL (zeros) */
  const double *dyn;      /* [n][Ndynobs*ndynobs*N] ready-made rows or NULL           */
  double *dyn_cur;  /* [n][n_dyn_live][2] current obstacle positions (in/out) or NULL */
  double *dyn_last; /* [n][n_dyn_live][2] positions one step earlier (in/out)         */
  const double *dyn_disp; /* [n][n_dyn_live][2] displacement per step (advance)       */
  double dyn_size;  /* rx = ry of the extrapolated rows (main.py:32 DYN_OBS_SIZE)     */
  double tuning[10];      /* q block (set_work_mode, trajectory_generator.py:117-131) */
  double base_speed, low_speed;
  double stc_weight, dyn_weight;
  /* hybrid mode (main.py:194-201): where use_hint[e] != 0 the N reference positions are the
   * DQN hint hint[e] (rl_ref) and the headings stay those of the original local reference
   * (InterfaceMpc.get_local_ref_traj(rl_ref) + ref_traj_filter(decay = 1)).  NULL = never. */
  const double *hint;     /* [n][N][2] */
  int *use_hint;          /* [n] input -- or OUTPUT when sw_state != NULL             */
  /* HintSwitcher.switch (main_pre.py:27-52), evaluated by the pack kernel when sw_state != NULL
   * with the robot position, the ORIGINAL local reference and the obstacle list
   * "processed static polygons + circle_to_rect(moving obstacle)" (main.py:91-95,200):
   * shapely Polygon.contains / distance restated (interior strictly, 0 inside).      */
  int *sw_state;            /* [n][2] switch_on, detach_cnt (in/out) or NULL           */
  const double *sw_poly_xy; /* [n or 1][sw_max_poly][sw_max_pv][2] static polygons      */
  const int *sw_poly_nv;    /* [n or 1][sw_max_poly] vertex counts (0 = unused slot)    */
  int sw_max_poly, sw_max_pv, sw_poly_shared, sw_detach_steps;
  double sw_switch_distance, sw_detach_distance; /* HintSwitcher(10, 2, 10) in main.py:129 */
  double sw_dyn_radius;     /* circle_to_rect radius (main.py:91: DYN_OBS_SIZE)         */
} ttmpc_fleet;

/* d_p [n][np] is written for every robot (robots that are not RUNNING keep packing from
 * their frozen state, so the batch stays dense). */
int ttmpc_fleet_pack_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet, double *d_p,
                            void *stream);
/* d_u [n][nu*N] solutions, d_exit_status [n] of the solve that used d_p. */
int ttmpc_fleet_advance_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet,
                               const double *d_u, const int *d_exit_status, void *stream);
/* pack + solve + advance, on `stream`.  The solve starts from zeros (run_step with
 * initial_guess=None) unless fleet->options has TTMPC_FLEET_WARM_START, and runs every robot
 * unless it has TTMPC_FLEET_SKIP_STOPPED.  Multipliers are carried in res->y when use_y0 != 0,
 * like the reference's Solver object.  The only entry point that takes action_steps > 1. */
int ttmpc_fleet_step_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet, double *d_p,
                            int use_y0, const ttmpc_result *res, void *stream);

/* Task queues of ttmpc_fleet_step_tasks_device: robot e has count[e] tasks, a goal [3] and a
 * polyline path of path_n (1..max_nodes) nodes each; next[e] of them have been taken.  All device
 * pointers.
 *
 * In the pack kernel, after the goal test, a robot that is TTMPC_FLEET_REACHED and has a task left
 * takes the next one -- a robot that arrived in this step as well as one that was parked before
 * its tasks were queued -- and does what InterfaceMpc.initialization(state, goal, path, mode)
 * does with it:
 *   - goal <- the task's goal; ref_traj / ref_len <- get_global_ref_traj(ts, path, state,
 *     base_speed) (trajectory_generator.py:160-201), sampled from the robot's current state with
 *     the device's arithmetic (sqrt(fma(dx,dx,dy*dy)), IEEE division, a 1-ulp atan2): within ulps of
 *     the Python sampler, not bit for bit;
 *   - idx_ref <- 0 and last_u <- 0 (past_actions is reset); status <- RUNNING; next[e] += 1;
 *   - the closest-point search and the goal test run again on the new task, so a robot whose
 *     consecutive goals lie within the 5 cm goal box takes several tasks in one step.  With
 *     action_steps = k > 1 the goal test still reads u[0] of the previous solution from res->u
 *     (InterfaceMpc._last_action, which initialization keeps).
 * The rest of the step is unchanged: the robot is packed and solved in this step, its multipliers
 * carry over in res->y (the reference keeps its Solver object), and with TTMPC_FLEET_WARM_START a
 * robot that took a task in this step starts from zeros (its previous solution tracked another
 * trajectory).  With the HintSwitcher on, a robot that took a task is switched once, if it is
 * RUNNING afterwards, on the new task's original local reference.  TTMPC_FLEET_REACHED thus means
 * that the last queued task is done.
 *
 * A task that cannot be driven -- no node, a walk the reference would index past the last node in
 * (a node it lands on within 1e-9 of the last one), no row or more than ref_stride rows -- sets
 * status TTMPC_FLEET_BAD_TASK and advances next[e] past it; goal, ref_traj, ref_len, idx_ref and
 * last_u keep the previous task's values.                                                       */
typedef struct ttmpc_fleet_tasks {
  int max_tasks, max_nodes;
  const int *count;      /* [n] queued tasks, 0..max_tasks                          */
  int *next;             /* [n] in/out: queued tasks taken so far (zeros at first)  */
  const double *goal;    /* [n][max_tasks][3]                                       */
  const double *path_xy; /* [n][max_tasks][max_nodes][2]                            */
  const int *path_n;     /* [n][max_tasks]                                          */
  double *path_out;      /* [n][max_nodes][2] or NULL: current path, in the layout  */
  int *path_out_n;       /* [n]                   ttdqn_internal_obs_device reads   */
} ttmpc_fleet_tasks;
/* ttmpc_fleet_step_device with task queues: writes fleet->goal, fleet->ref_traj and fleet->ref_len
 * of the robots that take a task (and their path_out rows when path_out != NULL).  With every count
 * zero it computes exactly what ttmpc_fleet_step_device computes.  tasks == NULL, max_tasks < 0,
 * max_nodes < 1, a NULL array other than path_out / path_out_n with max_tasks > 0, or path_out
 * without path_out_n -> TTMPC_ERR_BAD_ARG before any device work.  The pack and advance entry
 * points take no tasks. */
int ttmpc_fleet_step_tasks_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet,
                                  const ttmpc_fleet_tasks *tasks, double *d_p, int use_y0,
                                  const ttmpc_result *res, void *stream);

/* Obstacle-contact and tracking monitor of ttmpc_fleet_monitor_device: what the closed loop did in
 * the step that just ran, per robot, on the device.  All arrays are device pointers.
 *
 * Swept clearance.  The monitor runs after the step's advance, so robot e moved on the chord from
 * prev_xy[e] to state[e][0:2] and each moving obstacle j moved from dyn_last[e][j] to
 * dyn_cur[e][j].  clearance[e] is the minimum over the step of
 *   - per static polygon (a slot with nv < 3 is unused): the distance of the chord to the polygon
 *     minus robot_radius.  The polygon is a vertex ring, possibly non-convex (even-odd rule, strict
 *     interior as shapely's Polygon.contains); the distance is 0 if an endpoint is inside or the
 *     chord properly crosses an edge, else the least of the endpoint-to-edge and vertex-to-chord
 *     distances.  A zero-length chord gives shapely's Polygon.distance(Point);
 *   - per moving obstacle (when fleet->dyn_cur != NULL): the disc of radius moving_radius centred
 *     on the obstacle; both move linearly in time, so the distance is that of the origin to the
 *     segment from prev_xy - dyn_last to state - dyn_cur, minus (moving_radius + robot_radius);
 * and +inf for a robot without obstacles.  The chord stands in for the RK4 arc: with |w| <= 0.5
 * rad/s, v <= 1.5 m/s and ts = 0.2 s the arc leaves its chord by at most v ts (|w| ts) / 8, about
 * 4 mm.  Every robot is monitored, a parked one too (a moving obstacle may run into it).
 * Contact: clearance <= 0.  Then contact_steps[e] += 1, and first_contact[e] <- step if it is < 0.
 * min_clearance[e] <- min(min_clearance[e], clearance[e]).
 *
 * Tracking.  For a robot that is TTMPC_FLEET_RUNNING when the monitor runs (exactly the robots
 * that moved in this step): the distance of state[e][0:2] to the polyline through ref_traj rows
 * max(idx_ref - k, 0) .. min(idx_ref + 5k, ref_len) - 1 (k = action_steps), the window the next
 * pack's closest-point search scans; with one row the point distance.  deviation_max[e] <- max,
 * deviation_sum[e] += it, moved_steps[e] += 1.
 *
 * stop_on_contact != 0: a robot that is RUNNING and in contact gets status TTMPC_FLEET_COLLIDED
 * (after its deviation is taken).  It then stays where it is: pack and advance leave robots that
 * are not RUNNING alone, TTMPC_FLEET_SKIP_STOPPED skips its solve, and only REACHED robots take
 * queued tasks.  With stop_on_contact == 0 the monitor writes only the arrays of this struct.
 *
 * Arithmetic: plain IEEE mul / add in a fixed order (no contraction), so a C restatement compiled
 * with -ffp-contract=off matches it bit for bit.  Start values: prev_xy = the states before the
 * first step, min_clearance = +inf, first_contact = -1, the other in/out arrays 0.             */
typedef struct ttmpc_fleet_monitor {
  const double *poly_xy;  /* [n or 1][max_poly][max_pv][2] static polygons or NULL (none)     */
  const int *poly_nv;     /* [n or 1][max_poly] vertex counts (< 3: unused slot)              */
  int max_poly, max_pv;   /* max_poly >= 0; max_pv >= 3 when poly_xy != NULL                  */
  int poly_shared;        /* != 0: one polygon block for every robot                          */
  int stop_on_contact;
  double robot_radius;    /* >= 0: the robot is a disc of this radius                         */
  double moving_radius;   /* >= 0: radius of the moving obstacles' discs                      */
  int step;               /* written to first_contact                                        */
  int _pad;
  double *prev_xy;        /* [n][2] in/out: position at the previous call (set to state[0:2]) */
  double *clearance;      /* [n] out: this step's swept clearance                            */
  double *min_clearance;  /* [n] in/out: running minimum                                     */
  int *contact_steps;     /* [n] in/out: steps with clearance <= 0                           */
  int *first_contact;     /* [n] in/out: step of the first contact, -1 before it             */
  double *deviation_max;  /* [n] in/out: largest tracking deviation over the moved steps     */
  double *deviation_sum;  /* [n] in/out: summed tracking deviation over the moved steps      */
  int *moved_steps;       /* [n] in/out: steps in which the robot was RUNNING                 */
} ttmpc_fleet_monitor;
/* Run the monitor on `stream` after ttmpc_fleet_step_device or ttmpc_fleet_step_tasks_device (one
 * thread per robot).  mon == NULL, a NULL in/out array, poly_xy without poly_nv, max_poly < 0,
 * max_pv < 3 with polygons, a negative or non-finite radius, action_steps outside 1..N_hor or a
 * fleet the step would reject -> TTMPC_ERR_BAD_ARG before any device work. */
int ttmpc_fleet_monitor_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet,
                               const ttmpc_fleet_monitor *mon, void *stream);

/* Shared obstacle map of ttmpc_fleet_world_select_device: M >= 0 convex polygons that every robot
 * shares, of which each robot's K = Nstcobs static slots get the nearest ones before a step.  All
 * arrays are device pointers.
 *
 * The map.  Polygon o has a vertex ring poly_xy[o] (the convex hull the MPC sees), its half-space
 * row rows[o] of nstcobs doubles b[ne] a0[ne] a1[ne] (what polygon_halfspace_representation gives
 * for that hull; the kernel copies it and does not read it otherwise) and its axis-aligned bounding
 * box bbox[o] = (xmin, ymin, xmax, ymax).  reach R (finite, > 0) is the farthest obstacle that
 * matters; N_hor * ts * max(|lin_vel_min|, lin_vel_max), the farthest a feasible rollout gets, is
 * the natural choice.
 *
 * Selection for robot e, from p = state[e][0:2] (the state the pack kernel packs; a robot that
 * takes a task does not move, so task queues do not change it):
 *   - d_o = the distance of p to polygon o: 0 inside (even-odd rule), else the least distance to an
 *     edge; plain IEEE operations in a fixed order (the ring distance of the monitor's zero-length
 *     chord).  A polygon with poly_nv < 3 has no distance and is never selected; poly_nv > max_pv
 *     reads max_pv vertices.
 *   - eligible: d_o <= R.  n_reach[e] = the number of eligible polygons.
 *   - the eligible polygons ranked by (d_o, o) ascending (ties to the lower map index); the first
 *     k = min(K, n_reach) are taken and their rows written in ASCENDING MAP INDEX into slots
 *     0..k-1 of stc_out[e], zeros into the other slots; slot_poly[e][s] = the map index of slot s,
 *     -1 for an empty slot.  A map of M <= K polygons all within reach thus gives exactly the rows
 *     of the same polygons given as one shared block in map order, and a set that stays chosen keeps
 *     its rows from step to step.  n_reach[e] > K: an obstacle within reach got no slot.
 *   - every robot is selected, whatever its status (the pack kernel packs every robot).
 *
 * The grid.  A uniform grid over the map: cell (cx, cy), 0 <= cx < nx, 0 <= cy < ny, covers
 * [origin_x + cx cell, origin_x + (cx+1) cell) x [...y...]; its polygons are
 * cell_items[cell_start[c] .. cell_start[c+1]) with c = cy nx + cx, ascending within a cell.  It
 * must list polygon o in exactly the cells bx0..bx1 x by0..by1 with
 * bx0 = clamp(floor((xmin - origin_x) / cell), 0, nx-1), bx1 the same of xmax, by0 / by1 of
 * ymin / ymax (IEEE subtraction and division), and every polygon must lie inside the grid.  A query
 * visits cells floor((x - R - origin_x) / cell) - 1 .. floor((x + R - origin_x) / cell) + 1
 * (likewise in y), clamped to the grid, so no polygon within reach is missed to rounding, and
 * handles a polygon only in the lowest visited cell of its range, (max(qx0, bx0), max(qy0, by0)).
 * A robot outside the grid is exact too.  Map indices outside [0, M) in cell_items are skipped and
 * cell_start is clamped to [0, cell_start[nx ny]]: another grid cannot make the kernel read or write
 * out of bounds, but only a grid built by the rule above gives the selection above.  The kernel's
 * work per robot is the visited cells' items, independent of M at a fixed map density.
 *
 * Use: before each step call ttmpc_fleet_world_select_device on the step's stream and point
 * fleet.stc at d_stc_out with stc_shared = 0 (d_stc_out may be the buffer the step reads).     */
typedef struct ttmpc_fleet_world {
  int M;                   /* polygons, >= 0                                                  */
  int max_pv;              /* >= 3: vertex slots per polygon in poly_xy                       */
  const double *poly_xy;   /* [M][max_pv][2] vertex rings                                     */
  const int *poly_nv;      /* [M] vertex counts                                               */
  const double *rows;      /* [M][nstcobs] half-space rows                                    */
  const double *bbox;      /* [M][4] xmin ymin xmax ymax                                      */
  double reach;            /* R: finite, > 0                                                  */
  double origin_x, origin_y;
  double cell;             /* grid cell size: finite, > 0                                     */
  int nx, ny;              /* cells, >= 1 each                                                */
  const int *cell_start;   /* [nx*ny + 1] CSR offsets into cell_items                         */
  const int *cell_items;   /* [cell_start[nx*ny]] map indices                                 */
} ttmpc_fleet_world;
/* Write each robot's nearest map polygons (see ttmpc_fleet_world) on `stream`: d_stc_out
 * [n][Nstcobs*nstcobs], d_slot_poly [n][Nstcobs] or NULL, d_n_reach [n] or NULL.  Reads fleet->n
 * and fleet->state only.  world == NULL, M < 0, max_pv < 3, a non-finite or non-positive reach or
 * cell, nx or ny < 1 (or nx*ny too large for an int), a NULL map or grid array while M > 0, a NULL
 * d_stc_out or a fleet the step would reject -> TTMPC_ERR_BAD_ARG before any device work. */
int ttmpc_fleet_world_select_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet,
                                    const ttmpc_fleet_world *world, double *d_stc_out,
                                    int *d_slot_poly, int *d_n_reach, void *stream);

/* ------------------------------------------------------------------------
 * DQN side of the hybrid loop (src/main.py:174-193), device-resident.
 *
 * ttdqn_internal_obs_device: the `internal` observation of the ray model
 *   (variants/rays_reward1.py:27-31): SpeedObservation, AngularVelocityObservation,
 *   ReferencePathSampleObservation(1, 0, sample_offset), ReferencePathCornerObservation(
 *   corner_samples) -- components/int_obsv_*.py -- with path_progress =
 *   path.project(agent) (environment.py:115).
 *     d_agent5   [n][5]  x y theta v w
 *     d_path_xy  [n][max_nodes][2] reference-path polyline, d_path_n [n] node counts
 *                (1..max_nodes; one node is a path of length 0 at that point)
 *     d_internal [n][5 + 3*corner_samples] fp32 out, d_progress [n] out (may be NULL)
 * ttdqn_rl_ref_device: the DQN "hint" trajectory: MobileRobot.step(action, ts) followed by
 *   steps-1 x step_with_ref_speed(ts, ref_speed) on a copy of the agent
 *   (environment/agent.py:86-145); d_rl_ref [n][steps][2] positions.
 * ------------------------------------------------------------------------ */
int ttdqn_internal_obs_device(int n_envs, int max_nodes, int corner_samples, double sample_offset,
                              double max_distance, const double *d_agent5, const double *d_path_xy,
                              const int *d_path_n, float *d_internal, double *d_progress, void *stream);
int ttdqn_rl_ref_device(int n_envs, int steps, double ts, double ref_speed, const double *d_agent5,
                        const int *d_action, double *d_rl_ref, void *stream);

/* Cumulative device-side counters since the last reset: [0] cost-only
 * evaluations, [1] cost+gradient evaluations, [2] dynamic-obstacle bodies that
 * passed the bounding test, [3] PANOC iterations.  Synchronises the device.   */
int ttmpc_read_stats(unsigned long long out[4], int reset);
/* Launch geometry the solve kernel uses for n_scenes (reporting only). */
int ttmpc_launch_info(const ttmpc_config *cfg, int n_scenes, int *grid, int *block,
                      int *smem_bytes, int *blocks_per_sm, int *sm_count);

/* FP64 FMA-pipe peak probe: runs a dependent-chain-free DFMA kernel on every
 * SM and returns achieved TFLOP/s (used by bench.py as the roofline
 * denominator for the FP64-bound solve kernel).                            */
int ttmpc_measure_fp64_peak(double *tflops, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TTMPC_H */
