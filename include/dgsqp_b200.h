/* dgsqp_b200 -- C ABI of the batched Dynamic-Game SQP engine for NVIDIA B200 (sm_100a).
 *
 * The reference (zhu-edward/DGSQP) is pure Python and has no C ABI of its own; the seam its
 * Monte-Carlo drivers call is the solver class
 *     DGSQP(joint_dynamics, costs, agent_constraints, shared_constraints, bounds, params)
 *     .set_warm_start(u_ws) / .solve(states) / .step(states)        DGSQP/solvers/DGSQP.py:26-34,271-507
 * one game instance at a time.  This library is the batched replacement of that seam: the Python class
 * dgsqp_b200.DGSQP binds these entry points with ctypes.  Plain pointers and sizes only.
 *
 * Every function returns 0 on success or a negative DGSQP_E* code; dgsqp_last_error() gives the text.
 * No exceptions cross the ABI.  Buffers are owned by the caller.  A handle may be used from one host
 * thread at a time; different handles are independent.
 */
#ifndef DGSQP_B200_H
#define DGSQP_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DGSQP_MAX_AGENTS 4
#define DGSQP_MAX_TRACK_SEGS 8

enum {
  DGSQP_OK = 0,
  DGSQP_EINVAL = -1,      /* bad argument / unsupported game size */
  DGSQP_ECUDA = -2,       /* CUDA runtime error (no device, launch failure, ...) */
  DGSQP_ENOMEM = -3
};

/* Solve status per instance; maps 1:1 onto the reference's msg strings (DGSQP.py:383-474). */
enum {
  DGSQP_CONV_ABS_TOL = 0, /* 'conv_abs_tol' */
  DGSQP_CONV_REL_TOL = 1, /* 'conv_rel_tol' */
  DGSQP_MAX_IT = 2,       /* 'max_it'       */
  DGSQP_DIVERGED = 3,     /* 'diverged'     */
  DGSQP_QP_FAIL = 4,      /* 'qp_fail'      */
  DGSQP_TIME_LIMIT = 5    /* 'time_limit': the instance ran longer than params.time_limit (device clock, see dgsqp_params) */
};

/* Racing game of M kinematic bicycles on a constant-curvature-segment track.
 * Replaces the CasADi objects the reference scripts build and hand to DGSQP.__init__:
 *   vehicle  CasadiKinematicBicycleCombined            DGSQP/dynamics/dynamics_models.py:997-1079
 *   track    RadiusArclengthTrack (Chicane/CurveTrack) DGSQP/tracks/radius_arclength_track.py:199-225,361-408
 *   costs / constraints / bounds                       scripts/DGSQP_ALGAMES_monte_carlo_chicane.py:80-127,222-330
 *                                                      scripts/DGSQP_monte_carlo_agents.py:64-231               */
typedef struct {
  int32_t M;                 /* agents, 2..4 */
  int32_t N;                 /* horizon */
  double dt;
  double L_f, L_r;           /* wheel_dist_front / rear */
  double c_dr, c_da, c_s;    /* drag, damping, slip coefficients */
  double mass;
  double input_weight[2];    /* stage cost 1/2*w*u^2            (u = [u_a, u_steer]) */
  double rate_weight[2];     /* stage cost 1/2*w*(u_k-u_{k-1})^2 */
  double comp_weights[2];    /* terminal: -c0*s_i + sum_j c1*atan(s_j - s_i) */
  double u_ub[2], u_lb[2];   /* input box */
  double rate_ub[2], rate_lb[2]; /* input-rate limits per second (constraint is dt*rate) */
  double half_width;         /* |x_tran| <= half_width for k >= 1 */
  double obs_r[DGSQP_MAX_AGENTS]; /* collision radii: (r_i+r_j)^2 - |p_i-p_j|^2 <= 0, k >= 1 */
  int32_t track_nseg;
  double track_seg_len[DGSQP_MAX_TRACK_SEGS];
  double track_seg_curv[DGSQP_MAX_TRACK_SEGS];  /* signed curvature 1/r (0 = straight) */
} dgsqp_racing_game;

/* Highway-merge game of M kinematic unicycles (BASELINE config 5).  Replaces the CasADi objects
 * scripts/DGSQP_merge_monte_carlo.py builds and hands to DGSQP.__init__:
 *   vehicle  CasadiKinematicUnicycle, q = [x, y, v, psi], u = [F_x, w_z]   DGSQP/dynamics/dynamics_models.py:306-345
 *            discretised by rk3 with one sub-step                         DGSQP/dynamics/dynamics_models.py:202-212
 *   costs    stage 1/2 w_u.u^2 + 1/2 (q-goal)'diag(w_q)(q-goal), terminal term_scale * state term   merge.py:253-304
 *   lanes    two rows per agent and stage k = 0..N:  n(x)'(p - (pt - lane_r n(x))) <= 0 with the normal switched by
 *            ca.pw_const at x = brk (n_lo for x < brk, n_hi otherwise; brk = +inf for a straight lane)  merge.py:40-74,316-318
 *   bounds   input box (k < N), v bounds (k >= 1), pairwise collision rows (k >= 1)                    merge.py:130-169,306-314 */
typedef struct {
  double brk;
  double n_lo[2], n_hi[2];
  double pt[2];
} dgsqp_lane_row;

typedef struct {
  int32_t M;                 /* agents, 2..4 */
  int32_t N;                 /* horizon */
  double dt;
  double mass;
  double input_weight[2];
  double state_weight[4];
  double term_scale;
  double goal[DGSQP_MAX_AGENTS][4];
  double u_ub[2], u_lb[2];
  double v_ub, v_lb;
  double obs_r[DGSQP_MAX_AGENTS];
  double lane_r;
  dgsqp_lane_row lane[DGSQP_MAX_AGENTS][2];
} dgsqp_merge_game;

/* Mirrors DGSQPParams (DGSQP/solvers/solver_types.py:92-127); fields that only steer Python-side
 * behaviour (verbose, code_gen, debug_plot, ...) stay in the Python dataclass. */
typedef struct {
  double reg;
  double p_tol, d_tol;
  double beta, tau;
  int32_t line_search_iters;
  int32_t sqp_iters;
  int32_t nonmono_ls;
  int32_t merit_function;    /* 0 = 'stat_l1', 1 = 'stat' */
  int32_t conv_approx;
  /* `thresh` of DGSQP._get_mu (DGSQP.py:560): the l1 penalty weight mu is |d phi|/((1-rho)*viol) when the
   * summed constraint violation exceeds thresh, else 0.  The reference hard-codes 0 and that is what the Python class
   * passes for unchanged reference parameters; with 0, mu jumps between 0 and ~1e18 on rounding noise at active linear
   * constraints, 1e-10 (dgsqp_b200.DGSQP(..., mu_vio_thresh=1e-10), the setting of the golden fixtures) makes the choice
   * deterministic.  DESIGN.md deviation D2. */
  double mu_vio_thresh;
  /* DGSQPParams.time_limit (DGSQP.py:470-474) in seconds, measured per instance on the device's global timer from the
   * moment a CTA picks the instance up; <= 0 = no limit (the reference's default None). */
  double time_limit;
  /* 1 (default of the Python class): every QP starts from the active set of the instance's previous QP (qp_gi.cuh);
   * 0: cold start of every QP like the reference (DGSQP.py:240-241).  Same solution, fewer active-set iterations. */
  int32_t qp_warm_start;
  /* 1: keep (p_feas, comp, stat, qp_solves) of every SQP iteration for dgsqp_last_iter_data -- the `cond` and
   * `qp_solves` entries of the reference's iter_data (DGSQP.py:445-452, save_iter_data). */
  int32_t iter_log;
} dgsqp_params;

/* Mirrors DGSQPV2Params (DGSQP/solvers/solver_types.py:130-174): the v2 step policy of DGSQP/solvers/DGSQP_v2.py
 * (decaying regularisation, relaxed d-steps inside a shrinking radius, m-steps against a merit memory with
 * checkpoint reload, max_it counted in m-steps).  Constants the reference hard-codes (rel_tol_req = 10,
 * initial radius factor 20, eigenvalue floor 1e-9, divergence at 1e10) are hard-coded here too. */
typedef struct {
  double reg, reg_decay;
  double p_tol, d_tol;
  double beta, tau;
  int32_t line_search_iters;
  int32_t sqp_iters;                /* counted in m-steps (DGSQP_v2.py:407) */
  int32_t nms, nms_frequency, nms_memory_size;   /* memory size 1..16 */
  int32_t merit_function;           /* 0 = 'stat_l1', 1 = 'sum_obj_l1' (DGSQP_v2.py:1157-1164) */
  int32_t has_merit_parameter;      /* 0: mu from _get_mu (:683-707), 1: constant merit_parameter */
  double merit_parameter;
  double merit_decrease;            /* sigma */
  int32_t merit_decrease_condition; /* 0 = 'armijo', 1 = 'max' */
  double delta_decay;               /* gamma */
  double mu_vio_thresh;             /* see dgsqp_params */
  double time_limit;                /* DGSQPV2Params.time_limit (DGSQP_v2.py:412), see dgsqp_params */
  int32_t qp_warm_start;            /* see dgsqp_params */
  int32_t iter_log;                 /* see dgsqp_params; IterationData of DGSQP_v2.py:31-52: cond, qp_solves */
} dgsqp_v2_params;

typedef struct dgsqp_handle dgsqp_handle;

/* Builds the device-side solver for one game (the analogue of DGSQP.__init__/_build_solver,
 * DGSQP.py:26-230,587-979).  device = CUDA ordinal.  Fails with DGSQP_ECUDA when no GPU is usable:
 * there is no CPU fallback. */
int dgsqp_create(const dgsqp_racing_game* game, const dgsqp_params* params, int device, dgsqp_handle** out);
/* Same for the v2 solver class (DGSQP_v2.py:55-230); dgsqp_solve_batch then runs the v2 policy.  v2 keeps u_prev
 * between calls (:328); the batched entry point uses u_prev = 0 like the Monte-Carlo drivers do. */
int dgsqp_create_v2(const dgsqp_racing_game* game, const dgsqp_v2_params* params, int device, dgsqp_handle** out);
/* Same two constructors for the merge game; every other entry point takes the handle of either game.
 * dims for this game: n_q = 4M, n_u = 2M, n = N*n_u, m = 6M + (N-1)(P+8M) + (P+4M), P = M(M-1)/2. */
int dgsqp_create_merge(const dgsqp_merge_game* game, const dgsqp_params* params, int device, dgsqp_handle** out);
int dgsqp_create_merge_v2(const dgsqp_merge_game* game, const dgsqp_v2_params* params, int device, dgsqp_handle** out);
int dgsqp_destroy(dgsqp_handle* h);

/* dims[0..3] = n_q (joint state), n_u (joint input), n = N*n_u, m = number of constraint rows */
int dgsqp_dims(const dgsqp_handle* h, int32_t dims[4]);

/* Solves B independent instances (the loop body of the Monte-Carlo drivers,
 * scripts/DGSQP_ALGAMES_monte_carlo_chicane.py:485-488: set_warm_start + solve).
 *   x0      [B, n_q]          joint initial state (state2q order)
 *   u_ws    [B, n]            warm start, agent-major (DGSQP.set_warm_start, DGSQP.py:271-281)
 *   l_ws    [B, m] or NULL    dual warm start; NULL = the reference's behaviour, l0 = max(0,-lsqr(GG',Gq))
 *                             (DGSQP.py:312-326; set_warm_start accepts l_ws but v1 never uses it)
 *   u_out   [B, n]            solution inputs, agent-major
 *   l_out   [B, m]            multipliers (l_pred)
 *   x_out   [B, (N+1)*n_q]    state trajectory (q_pred)
 *   cost_out[B, M]  cond_out[B, 3] = (p_feas, comp, stat)
 *   num_iters/status/qp_solves [B]
 * memspace: 0 = host pointers (copies are done inside, on `stream`), 1 = device pointers.
 * stream: a cudaStream_t (NULL = default stream).  The call returns after the work has completed. */
int dgsqp_solve_batch(dgsqp_handle* h, int32_t B, const double* x0, const double* u_ws, const double* l_ws,
                      double* u_out, double* l_out,
                      double* x_out, double* cost_out, double* cond_out, int32_t* num_iters, int32_t* status,
                      int32_t* qp_solves, int32_t memspace, void* stream);

/* dgsqp_solve_batch with the previous input u_{-1} of every instance (u_prev [B, n_u] or NULL = zeros; same memory space
 * as the other buffers): the receding-horizon use of the v2 class, whose solve() keeps u_prev between calls
 * (DGSQP_v2.py:311,328) -- it enters the input-rate costs and rate constraints of stage 0.  Handles created with
 * DGSQPParams (v1) ignore it: v1's solve() zeroes u_prev on entry (DGSQP.py:305). */
int dgsqp_solve_batch_up(dgsqp_handle* h, int32_t B, const double* x0, const double* u_ws, const double* l_ws, const double* u_prev,
                         double* u_out, double* l_out, double* x_out, double* cost_out, double* cond_out, int32_t* num_iters,
                         int32_t* status, int32_t* qp_solves, int32_t memspace, void* stream);

/* Same as dgsqp_solve_batch with device pointers but only enqueues (no synchronisation). */
int dgsqp_solve_batch_async(dgsqp_handle* h, int32_t B, const double* x0, const double* u_ws, const double* l_ws,
                            double* u_out,
                            double* l_out, double* x_out, double* cost_out, double* cond_out, int32_t* num_iters,
                            int32_t* status, int32_t* qp_solves, void* stream);

/* Warm-start generation on the device: the PID lane-follower roll-out the Monte-Carlo drivers run for every sampled agent
 * before a solve (scripts/DGSQP_ALGAMES_monte_carlo_chicane.py:411-467, DGSQP/solvers/PID.py:74-138,187-238, one-step
 * simulation DGSQP/dynamics/dynamics_models.py:161-186 with classical RK4 x 4 sub-steps, local_to_global
 * DGSQP/tracks/radius_arclength_track.py:752-807).  K agents start at (s0, x_tran0, v0), e_psi = 0.
 *   key_pts  HOST [(track_nseg+1) * 6]  x, y, psi, cumulative s, segment length, curvature (get_track_key_pts, :361-408)
 *   q0 [K, 6]  state2q of the initial states;  xy [K, N+1, 2] global positions of the roll-out (collision pre-check);
 *   u_ws [K, N, 2] inputs = the warm start of that agent.        memspace: 0 host pointers, 1 device pointers. */
int dgsqp_pid_rollout(const dgsqp_racing_game* game, const double* key_pts, int device, int32_t K, const double* s0,
                      const double* xt0, const double* v0, double* q0, double* xy, double* u_ws, int32_t memspace, void* stream);

/* Monte-Carlo instance generation on the device (the sampling half of the Monte-Carlo drivers,
 * scripts/DGSQP_ALGAMES_monte_carlo_chicane.py:384-467, DGSQP_monte_carlo_agents.py:257-308, DGSQP_merge_monte_carlo.py:424-495;
 * host statement dgsqp_b200/montecarlo.py).  The stream is numpy.random.PCG64, started from the state of
 * np.random.default_rng(seed).bit_generator.state.  Trial t consumes draws D*t .. D*t+D-1 (head-to-head D = 5:
 * ego_s, ego_xt, ego_v, d, tar_v; M agents D = 3M: s, x_tran, v per agent; merge D = 12 in sample_merge's order) and
 * instance i is the i-th accepted trial, so the output does not depend on the batch size: the first B/2 instances of a
 * B-instance call are those of a B/2-instance call.  A trial is rejected when the PID roll-outs of its agents (see
 * dgsqp_pid_rollout) come closer than r_i + r_j at any stage k = 0..N (head-to-head: also when the target starts behind
 * s = 0 or off the track); merge: when the zero-input RK3 roll-outs do, car 3 rolled out from the zero state.
 *   key_pts      HOST, as in dgsqp_pid_rollout
 *   x0 [B, n_q]  DEVICE, state2q of the agents;  u_ws [B, n] DEVICE, PID warm start, agent-major (racing only; the merge
 *                scenario starts from a zero warm start);  trial [B] DEVICE or NULL: trial id of every instance
 *   accepted, trials_used  HOST: instances written, trials consumed (id of the last accepted trial + 1)
 * Stops after max_trials trials: then returns DGSQP_EINVAL and the first *accepted rows are valid.  The call returns after
 * the work on `stream` has completed.  Racing: M = 2..4 (head-to-head: M = 2); merge: the 3-car scenario. */
typedef struct { uint64_t state_hi, state_lo, inc_hi, inc_lo; } dgsqp_pcg64;   /* numpy.random.PCG64 state */
enum { DGSQP_SAMPLE_HEAD_TO_HEAD = 0, DGSQP_SAMPLE_AGENTS = 1 };
int dgsqp_sample_racing(const dgsqp_racing_game* game, const double* key_pts, int32_t kind, const dgsqp_pcg64* rng,
                        int device, int32_t B, int64_t max_trials, double* x0, double* u_ws, int64_t* trial,
                        int32_t* accepted, int64_t* trials_used, void* stream);
int dgsqp_sample_merge(const dgsqp_merge_game* game, const dgsqp_pcg64* rng, int device, int32_t B, int64_t max_trials,
                       double* x0, int64_t* trial, int32_t* accepted, int64_t* trials_used, void* stream);

/* Statistics of a solved batch reduced on the device, so that a Monte-Carlo sweep that only wants the summary table of
 * scripts/process_data_curve.py:98-110 / process_data_merge.py:58-67 does not have to copy B x (n + m) doubles back.
 * status / num_iters / qp_solves / cond are DEVICE pointers as written by dgsqp_solve_batch(memspace = 1) (cond may be
 * NULL); out16 is a HOST array: count, #conv_abs_tol, #conv_rel_tol, #max_it, #diverged, #qp_fail, #time_limit,
 * sum iters, sum iters^2, sum qp_solves, the same three sums over converged instances, max p_feas and max stat over
 * converged instances, reserved.  The additive layout is what the per-GPU shards all_gather at the end of a run. */
int dgsqp_batch_stats(int device, int32_t B, const int32_t* status, const int32_t* num_iters, const int32_t* qp_solves,
                      const double* cond, double* out16, void* stream);

/* The same 16 statistics for the LAST solve_batch[_async] on this handle, accumulated by the solve kernel itself as its
 * instances finish (one atomic per entry and instance in the kernel's epilogue: no second pass over the outputs, no extra
 * launch).  Waits for that launch; out16 is a HOST array.  Counts and iteration sums are integer-valued doubles, so the
 * result does not depend on the order in which the instances finish. */
int dgsqp_last_stats(dgsqp_handle* h, double* out16);

/* Per-instance work counters of the LAST solve_batch on this handle (device->host copy), DGSQP_NDIAG = 8 ints each:
 * full evaluations, gradient-only evaluations, QP active-set iterations, max #negative eigenvalues of a Hessian,
 * QPs whose Hessian was indefinite, sum of #negative eigenvalues, sum of final active-set sizes, line-search trials. */
#define DGSQP_NDIAG 8
int dgsqp_last_diag(dgsqp_handle* h, int32_t B, int32_t* diag);

/* Per-iteration record of the LAST solve_batch on a handle created with params.iter_log = 1: out is a HOST array
 * [B, dgsqp_iter_log_capacity(h), 4] of (p_feas, comp, stat, qp_solves of that iteration); rows past an instance's
 * num_iters + 1 are zero.  What the reference keeps as iter_data[i]['cond' | 'qp_solves'] (DGSQP.py:445-452). */
int dgsqp_iter_log_capacity(const dgsqp_handle* h);
int dgsqp_last_iter_data(dgsqp_handle* h, int32_t B, double* out);

/* Per-instance phase profile of the LAST solve_batch: dgsqp_phase_count() SM-clock cycle counters per
 * instance (order: rollout+derivatives [full], adjoints/sensitivities [full], Hessian DP, tridiagonalisation,
 * negative eigenpairs, Cholesky, triangular inverse, active-set loop, LSQR, rollout+Jacobians [gradient-only],
 * adjoints [gradient-only], merit, other).  Replaces the reference's verbose per-phase wall-clock prints
 * (DGSQP.py:233,261,349,443,510,525). */
int dgsqp_phase_count(void);
int dgsqp_last_phase_cycles(dgsqp_handle* h, int32_t B, int64_t* cycles);

/* Measures the device's sustained FP64 FMA throughput (TFLOP/s, 2 flops per FMA) with a register-only
 * probe kernel: the roofline denominator for this FP64-bound path. */
int dgsqp_measure_fp64_peak(int device, double* tflops);

/* Number of kernels launched by this library since load (for bench accounting). */
int64_t dgsqp_kernel_launches(void);

/* Memory placement of one CTA (one game instance in flight): out[0] = dynamic shared memory bytes, out[1] = global
 * workspace bytes, out[2] = 1 when the two n x n work matrices are shared-memory resident, out[3] = bit 0: the packed
 * sensitivity rows are, bit 1: every hot buffer is, bit 2: the first work matrix (factors) is.  dgsqp_set_smem_limit caps the shared memory the planner may use (0 = device maximum);
 * with a small cap everything falls back to the global workspace (used by the tests to cover both placements). */
int dgsqp_memory_plan(const dgsqp_handle* h, int64_t out[4]);
int dgsqp_set_smem_limit(dgsqp_handle* h, int64_t bytes);

/* Grid configuration: CTAs per SM (0 = as many as fit) and threads per CTA (0 = default 256, at most 512). */
int dgsqp_configure(dgsqp_handle* h, int32_t ctas_per_sm, int32_t threads);

const char* dgsqp_last_error(void);
const char* dgsqp_version(void);

#ifdef __cplusplus
}
#endif
#endif
