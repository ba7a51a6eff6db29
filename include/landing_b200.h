/*
 * landing_b200.h -- C ABI of the B200-native batched solver for the SRB landing NLP of
 * se-hwan/landing-controller.  Plain pointers and sizes only; every entry point either runs on
 * the GPU or fails (there is no CPU fallback).
 *
 * Two groups of symbols are exported by liblanding_b200.so (= drop-in landingCtrller_IPOPT.so):
 *
 * (1) The CasADi-generated-C function ABI that the reference's solver object binds by name
 *     (reference: optimizations/landing/codegen_casadi/landingCtrller_IPOPT.c:10916-10992 for the
 *     per-function template; callers external.cpp:63-111,325-362, nlpsol.cpp:100-109):
 *     for F in {nlp, nlp_f, nlp_g, nlp_grad, nlp_grad_f, nlp_hess_l, nlp_jac_g}
 *       F, F_alloc_mem, F_init_mem, F_free_mem, F_checkout, F_release, F_incref, F_decref,
 *       F_n_in, F_n_out, F_default_in, F_name_in, F_name_out, F_sparsity_in, F_sparsity_out, F_work
 *     declared in casadi_symbols.h.  One scenario per call (latency bound; for drop-in and parity).
 *
 * (2) The batched entry points below (new; SURVEY 8b "Batched extension"): thousands of scenarios
 *     per call, host or device buffers, AoS (CasADi vector per scenario) or SoA layout.
 */
#ifndef LANDING_B200_H
#define LANDING_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct landing_ctx landing_ctx;

enum { LANDING_OK = 0, LANDING_ERR_ARG = 1, LANDING_ERR_CUDA = 2, LANDING_ERR_NOGPU = 3 };
enum { LANDING_HOST = 0, LANDING_DEVICE = 1 }; /* where the caller's buffers live */
enum { LANDING_AOS = 0, LANDING_SOA = 1 };     /* [B][n] (one CasADi vector per scenario) | [n][B] */

/* per-scenario solve status (replaces IPOPT's return status, which the reference drops:
 * generate_landingCtrller_IPOPT.m:269 solve_limited) */
enum {
  LANDING_ST_CONVERGED = 0,
  LANDING_ST_MAX_ITER = 1,
  LANDING_ST_LINESEARCH_FAIL = 2,
  LANDING_ST_NAN = 3,
  LANDING_ST_FACTOR_FAIL = 4,
  LANDING_ST_NOT_INTERIOR = 5, /* landing_kino_step_batch: a slack or bound multiplier not strictly interior */
  LANDING_ST_RUNNING = 9
};

/* Create a context for the N-knot problem on CUDA device `device`.
 * Sizes: n_x = 36N-24, n_p = 13N+81, m = 104N-92, nnz(J) = 385N-421, nnz(H) = 189(N-1). */
int landing_create(int n_knots, int device, landing_ctx **ctx);
void landing_destroy(landing_ctx *ctx);
const char *landing_last_error(void);

/* dims = {N, n_x, n_p, m, nnzJ, nnzH} */
int landing_dims(const landing_ctx *ctx, long long dims[6]);
/* host-only size query (no GPU needed) */
int landing_dims_for(int n_knots, long long dims[6]);
/* CasADi CCS pattern {nrow, ncol, colind[ncol+1], row[nnz]} (mem.h:73-92) of
 * which = 0: jac_g_x (casadi_s5, landingCtrller_IPOPT.c:64), 1: hess_gamma_x_x upper triangle
 * (casadi_s4, :63); 2: dense x (casadi_s0), 3: dense p (s1), 4: scalar (s2), 5: dense g (s3).
 * Host pointers owned by the library; no GPU needed. */
const long long *landing_sparsity(const landing_ctx *ctx, int which);
const long long *landing_sparsity_for(int n_knots, int which);

/* Batched evaluation of the generated functions (replaces nlp_f :10995, nlp_g :11161,
 * nlp_grad_f :52602, nlp_jac_g :94014, nlp_hess_l :53527, nlp_grad :22015).
 * Inputs x[B x n_x], p[B x n_p]; lam_f[B], lam_g[B x m] needed for hess / grad_x / grad_p.
 * NULL inputs are all-zero (as `arg[i]==0` in the generated C); NULL outputs are skipped.
 * status[B] (optional, int32): 0 ok, -1 a NaN/Inf was produced (oracle_function.cpp:218-266). */
typedef struct landing_eval_io {
  const double *x, *p, *lam_f, *lam_g;
  double *f;      /* [B]        */
  double *g;      /* [B x m]    */
  double *grad_f; /* [B x n_x]  */
  double *jac;    /* [B x nnzJ] */
  double *hess;   /* [B x nnzH] */
  double *grad_x; /* [B x n_x]  grad_gamma_x */
  double *grad_p; /* [B x n_p]  grad_gamma_p */
  int *status;    /* [B]        */
} landing_eval_io;

int landing_eval_batch(landing_ctx *ctx, long long B, int memspace, int layout,
                       const landing_eval_io *io);

/* lbg(p), ubg(p): the bounds the reference's .casadi wrapper computes from the parameters
 * (generate_landingCtrller_IPOPT.m:319-321; optistack_internal.cpp:742-870). +-inf one-sided. */
int landing_bounds_batch(landing_ctx *ctx, long long B, int memspace, int layout, const double *p,
                         double *lbg, double *ubg);

/* Shared numeric data of a sweep (generate_landingCtrller_IPOPT.m:173-196). */
typedef struct landing_problem {
  double T; /* horizon, dt = T/(N-1) */
  double q_min[6], q_max[6], qd_min[6], qd_max[6];
  double q_term_min[6], q_term_max[6], qd_term_min[6], qd_term_max[6];
  double q_term_ref[6], qd_term_ref[6];
  double c_ref[12];
  double QN[12];
  double mu, l_leg_max, f_max, mass, Ib[3], Ib_inv[3];
  /* Variant data used by the SOLVER only (the generated-function ABI above is the landingCtrller_IPOPT problem):
   * running GRF cost sum_k sum_legs (Qf . f^2) dt_k and kinematic box half-widths (x, y, z) -- the "CCC" landing
   * problem whose IPOPT solutions the reference stores (generate_quadruped_SRBM_CCC.m:80-91,169-176 with
   * analysis/eval_SRBM_CCC.m:49-52: QX = Qc = 0, Qf = (1e-4, 1e-4, 1e-3), box 0.05/0.05/0.27).
   * Defaults {0,0,0} and {0.15, 0.15, 0.30} = generate_landingCtrller_IPOPT.m:83-85,150-155. */
  double Qf[3], kin_box[3];
  /* Knot spacings dt[0..N-2] (HOST pointer, read during the call), or NULL for the uniform T/(N-1).  The reference's
   * callers pass dt as a vector: uniform in the generator's own test call (generate_landingCtrller_IPOPT.m:195,319-327),
   * NON-uniform in the sweep / MPC callers: dt_val = [0.05 0.02x15 0.05 0.05 0.1 0.2] for N = 21
   * (generate_data/generate_training_data_automated.m:28,130-136; main_scripts/landing_optimization.m:28,305-311). */
  const double *dt;
  /* FORMULATION.  0 (default): the contact-implicit NLP of landingCtrller_IPOPT (generate_landingCtrller_IPOPT.m:90-169).
   * 1: the fixed-contact-schedule NLP of quadruped_SRBM_NLP.m:84-176 (BASELINE configs[0]) -- solver only:
   *    f_z <= cs f_max (:148), cs c_z = 0 (:154), cs (c+ - c) = 0 (:155-158) instead of the complementarity / no-slip
   *    inequalities; no terminal rows (:105-108 are commented out); running cost sum_k dt_k ((X_k - Xref_k)' QX (X_k -
   *    Xref_k) + f_k' Qf f_k) (:85-92; Qc = 0 in the reference's parameter set :213 and is not implemented) next to the
   *    terminal cost QN.  cs: HOST pointer to 4 (N-1) ints, cs[4 k + leg] in {0, 1}.  The extra equality rows vanish
   *    identically where cs = 0 (rank-deficient Jacobian); they are handled the way IPOPT handles that case, by the dual
   *    regularisation delta_c: sigma = 1 / delta_c in the condensed stage matrix, y+ = y + (J dx + c) / delta_c.
   *    lam_g is returned in the row layout of formulation 0 (unused rows carry 0). */
  int formulation;
  const int *cs;
  double QX[12];
  double delta_c; /* 1e-7 */
} landing_problem;

void landing_problem_default(landing_problem *pb);

/* p[B x n_p] and x0[B x n_x] from drop conditions drops[B x 12] = (q_init[6], qd_init[6]),
 * generated on the device (generate_landingCtrller_IPOPT.m:199-208, 336: Xref linspace,
 * Uref feet = Xref_pos + c_ref, forces 0, x0 = [Xref(:);Uref(:)]).  drops is always AoS. */
int landing_build_batch(landing_ctx *ctx, long long B, int memspace, int layout,
                        const landing_problem *pb, const double *drops, double *p, double *x0);

/* Interior-point options; names follow the IPOPT options the reference sets
 * (generate_landingCtrller_IPOPT.m:232-263). */
typedef struct landing_options {
  int max_iter;              /* 3000 */
  double tol;                /* 1e-4 */
  double constr_viol_tol;    /* 1e-3 */
  double dual_inf_tol;       /* 1 (IPOPT default) */
  double compl_inf_tol;      /* 1e-4 (IPOPT default) */
  double mu_init;            /* 0.1 */
  double bound_push;         /* 0.5 */
  double bound_frac;         /* 0.5 */
  double bound_relax_factor; /* 1e-6 */
  int max_soc;               /* 4 -- ACCEPTED BUT UNUSED: no second-order correction is implemented (see below) */
  /* Jamming watchdog (this library's substitute for IPOPT's restoration phase, which the restatement does not
   * have): when the accepted primal step length stays below jam_alpha for jam_iters consecutive iterations the
   * iterate is re-centred exactly as after a failed line search (slacks pushed back inside their bounds,
   * multipliers reset, mu = mu_init or restart_mu).  jam_iters = 0 switches it off. */
  int jam_iters;             /* 5 */
  double jam_alpha;          /* 0.02 */
  /* Re-centrings allowed per scenario (failed line searches + watchdog).  On the grid and random sweeps 99.7 % of the
   * scenarios that converge need at most 8; the ones that exhaust the budget sit at a point of local infeasibility
   * and return LANDING_ST_LINESEARCH_FAIL.  (The reference's IPOPT would enter its restoration phase there.) */
  int max_restarts;          /* 8 */
  int reserved[5];
  /* Barrier parameter a re-centring restarts from; <= 0 (the default) means mu_init.  Measured with the CPU
   * restatement (DESIGN.md 3): on the GRID sweeps of BASELINE configs[1] / [2] 0.01 saves 13 % / 16 % of the iterations
   * with as many scenarios converged, on the reference's RANDOM sweeps with the sweep callers' parameters it loses
   * converged scenarios (85.6 % instead of 89.6 % of 1024 drops) -- so it is an option, not the default. */
  double restart_mu;         /* 0 = mu_init */
} landing_options;

/* IPOPT options the reference sets (generate_landingCtrller_IPOPT.m:232-263) that this solver does NOT implement:
 * mu_strategy = adaptive / mu_oracle = probing (monotone Fiacco-McCormick update instead), max_soc (no second-order
 * correction), min/max_refinement_steps (no iterative refinement of the Riccati solve), nlp_scaling_method =
 * gradient-based (never triggers at the reference's initial guesses: max |J(x0)| <= 50), acceptable_tol /
 * acceptable_iter (only the strict tolerances terminate; with acceptable_tol = tol the acceptable test was measured
 * never to fire on the sweeps, DESIGN.md section 3), and IPOPT's restoration phase (replaced by re-centring with
 * the watchdog above).  DESIGN.md section 3 lists the measured consequences. */
void landing_options_default(landing_options *opt);

/* Solve B independent landing NLPs, one per drop condition (replaces one call of the
 * serialized solver function per scenario: main_scripts/landing_optimization.m:305-311,
 * generate_data/generate_training_data_automated.m:130-136).
 * Outputs (host or device per memspace, AoS): x_star[B x n_x], f_star[B], status[B] (int32),
 * iters[B] (int32); optional lam_g[B x m]. x0 may be NULL (reference initial guess). */
typedef struct landing_solve_io {
  const double *drops; /* [B x 12] */
  const double *x0;    /* [B x n_x] or NULL */
  double *x_star, *f_star, *lam_g;
  double *viol; /* [B] final max constraint violation, optional */
  int *status, *iters;
} landing_solve_io;

int landing_solve_batch(landing_ctx *ctx, long long B, int memspace, const landing_problem *pb,
                        const landing_options *opt, const landing_solve_io *io);

/* One sweep on SEVERAL GPUs of this process (SURVEY 8e: the scenario batch shards naturally, no data-path collective):
 * scenario b is solved on devices[b % n_devices] (interleaved shards: the iteration count grows along the axes of a grid
 * sweep), one host thread and one context per device, and the result records [x*, f*, status, iters, viol, lam_g] of the
 * WHOLE sweep are gathered into the caller's HOST arrays in global scenario order -- the library-level counterpart of
 * the NCCL all-gather a process-per-GPU launch does (bench.py).  A device index may be listed more than once (several
 * contexts, i.e. several independent work queues, on one GPU).  io: HOST pointers, same meaning as above. */
typedef struct landing_multi landing_multi;
int landing_multi_create(int n_knots, int n_devices, const int *devices, landing_multi **m);
void landing_multi_destroy(landing_multi *m);
int landing_solve_batch_multi(landing_multi *m, long long B, const landing_problem *pb,
                              const landing_options *opt, const landing_solve_io *io);

/* Time-varying LQR pass along solved trajectories (replaces, for a batch, quadruped_SRBM_NLP.m:428-497 with
 * srbm-utilities/generateVariationalDynamics.m:9-62 and generateRiccatiIntegrator.m:24,49-53): P(t_k), k = 0..n_steps-1,
 * t_k = k dt, from P(t_{n_steps-1}) = F by explicit Euler steps of Pdot = A'P + PA - P B R^-1 B'P + Q, and the gains
 * K_k = R^-1 B(t_k)' P(t_k).  State (p, rpy, omega, v, feet[12]), control = GRFs[12].  Matrices row-major. */
typedef struct landing_tvlqr {
  double T;        /* horizon of the trajectories (knot spacing T/(N-1)) */
  double dt;       /* Riccati step, 0.022 in the reference */
  int n_steps;     /* time points */
  double Q[576], F[576], R[12]; /* running weight, terminal weight, diagonal of the control weight (90); Q and F must
                                   be symmetric: P stays symmetric and A'P + PA is formed as W + W' with W = A'P */
  double Ib[9];    /* full 3x3 body inertia, get_mass_matrix(model, zeros(18,1), 0) */
  double mass;
} landing_tvlqr;
void landing_tvlqr_default(landing_tvlqr *par);
/* x_star [B x n_x] (AoS, as landing_solve_batch returns it); P_out [B x n_steps x 576], K_out [B x n_steps x 288]
 * (12 x 24 row-major); either output may be NULL. */
int landing_tvlqr_batch(landing_ctx *ctx, long long B, int memspace, const landing_tvlqr *par,
                        const double *x_star, double *P_out, double *K_out);

/* Kino-dynamic ("full-body") landing NLP, the reference's KNITRO variant (SURVEY 8 f-2;
 * generate_solver/generate_landingCtrller_KNITRO.m:34-193): +12 joint angles per knot, foot positions tied to the forward
 * kinematics of the legs (get_forward_kin_foot.m:4-25), joint-torque limits tau = J_f' (-R' f) (get_foot_jacobians_mc.m:12-24),
 * joint limits, XYZ rotation convention (rpyToRotMat_xyz.m:2).  Batched constraint values and sparse Jacobian (CCS value
 * array, pattern from landing_kino_sparsity) and, below, the Lagrangian Hessian (landing_kino_hess_batch), gradient and
 * KKT residuals (landing_kino_kkt_batch) -- the functions an NLP solver iterates on --, the primal-dual Newton step of
 * one interior-point iteration (landing_kino_step_batch) and the interior-point solve over them (landing_kino_solve_batch).  x[B x n_x] = [X(:); jpos(:); U(:)] per scenario (Opti variable order :45-51),
 * g[B x m], jac[B x nnz]; dims = {N, n_x = 12N + 36(N-1), m = 48 + 141(N-2) + 117, nnz}.  The row map and the bounds
 * lbg / ubg are restated in oracle/kino_ref.py (pinned to the stored solution generate_solver/prevSoln.mat). */
typedef struct landing_kino_problem {
  double mu, mass, Ib[3], Ib_inv[3];
  const double *dt; /* HOST pointer to N-1 knot spacings */
} landing_kino_problem;
int landing_kino_dims(int n_knots, long long dims[4]);
const long long *landing_kino_sparsity(int n_knots); /* CCS {nrow, ncol, colind[ncol+1], row[nnz]}, host, library-owned */
int landing_kino_eval_batch(landing_ctx *ctx, long long B, int memspace, int layout, const landing_kino_problem *pb,
                            const double *x, double *g, double *jac);

/* The rest of what a solver of the kino-dynamic NLP needs per drop condition -- what generate_landingCtrller_KNITRO.m
 * :198-262,300-327 computes before it calls the solver: the bounds lbg / ubg [B x m] (Opti canonical form of :93-193
 * with q_init / qd_init / c_init of the drop, the velocity-dependent kinematic box kin_box_limits.m of the body-frame
 * velocity :246-248, initial feet c_init :232-236), the initial guess x0 [B x n_x] = [X; jpos_guess; U] assembled
 * from an SRB solution x_srb [B x (36N-24)] as landing_solve_batch returns it (:302-323; NULL: the reference
 * trajectories Xref / Uref of :272-286, which are also the SRB stage's own initial guess), and the terminal cost
 * f = (X_N - Xref_N)' QN (X_N - Xref_N) with its gradient (:86-88).  drops [B x 12] = (q_init, qd_init) as for
 * landing_solve_batch.  Any output may be NULL.  Defaults = the values of :214-262. */
typedef struct landing_kino_setup {
  double q_term_min[6], q_term_max[6], qd_term_min[6], qd_term_max[6]; /* :214-217 */
  double z_min;        /* q_min(3) = 0.075 (:219; only the z bound is enforced, :184) */
  double l_leg_max;    /* 0.4 */
  double jpos_min[12], jpos_max[12]; /* (-pi/3, -pi/2, 0), (pi/3, pi/2, 3 pi/4) per leg */
  double tau_max[3];   /* gear ratio x 3 Nm: 18, 18, 27.99 (get_robot_model.m:237-241) */
  double QN[12];       /* 0 0 100 10 10 0 10 10 10 10 10 10 */
  double q_term_ref[6], qd_term_ref[6]; /* (0 0 0.25 0 0 0), 0 */
  double jpos_guess[3]; /* 0, -pi/4, pi/2 (:325) */
} landing_kino_setup;
void landing_kino_setup_default(landing_kino_setup *ks);
int landing_kino_setup_batch(landing_ctx *ctx, long long B, int memspace, int layout, const landing_kino_setup *ks,
                             const double *drops, const double *x_srb, double *lbg, double *ubg, double *x0);
int landing_kino_cost_batch(landing_ctx *ctx, long long B, int memspace, int layout, const landing_kino_setup *ks,
                            const double *x, double *f, double *grad_f);

/* Lagrangian Hessian of the kino-dynamic NLP: H = d2/dx2 (lam_f f(x) + lam_g' g(x)), f the terminal cost of
 * landing_kino_cost_batch, g the constraint function of landing_kino_eval_batch (the signs of CasADi's nlp_hess_l), as
 * the CCS value array of its UPPER triangle (row <= col; the convention of landing_sparsity(ctx, 1)).  Exact
 * second derivatives of the same knot function.  Every entry of hess is written on every call. */
/* upper-triangle CCS {nrow, ncol, colind[ncol+1], row[nnz]} of the Lagrangian Hessian; host, library-owned, no GPU */
const long long *landing_kino_hess_sparsity(int n_knots);
/* hess[B x nnzH]; x [B x n_x]; lam_f [B] and lam_g [B x m]: NULL = all zero; ks (QN, q/qd_term_ref) required when lam_f != NULL */
int landing_kino_hess_batch(landing_ctx *ctx, long long B, int memspace, int layout, const landing_kino_problem *pb,
                            const landing_kino_setup *ks, const double *x, const double *lam_f,
                            const double *lam_g, double *hess);

/* Lagrangian gradient and KKT residuals of the kino-dynamic NLP at a primal-dual point (x, lam_f, lam_g), with CasADi's
 * sign convention L = lam_f f + lam_g' g (f the terminal cost of landing_kino_cost_batch, g the rows of
 * landing_kino_eval_batch), per scenario:
 *   grad_x    = lam_f grad f + J' lam_g                                     (CasADi nlp_grad: grad_gamma_x)
 *   viol      = max_i max(lbg_i - g_i, g_i - ubg_i, 0); an infinite bound never counts
 *   dual_inf  = max_j |grad_x_j|, unscaled.  The NLP has no variable bounds, so lam_x = -grad_x
 *   compl_inf = max_i c_i over the inequality rows (lbg_i < ubg_i; equality rows are excluded),
 *               c_i = max(lam_g_i, 0) |ubg_i - g_i| + max(-lam_g_i, 0) |g_i - lbg_i|; a multiplier of the wrong sign
 *               for an infinite bound gives +inf (lam_g_i = 0 gives 0)
 * A NaN in any input of a scenario (x, lam_f, lam_g, lbg, ubg), or in the g or grad_x computed from them, makes each of
 * that scenario's viol / dual_inf / compl_inf NaN, and no other scenario's.  Results are deterministic: the same bits from
 * run to run, in both layouts and both memory spaces.  grad_x is computed without forming J, and every entry is written
 * on every call.  Every output may be NULL; B = 0 launches nothing. */
typedef struct landing_kino_kkt_io {
  const double *x;         /* [B x n_x], required */
  const double *lam_f;     /* [B] in both layouts, NULL = 0 (needs ks) */
  const double *lam_g;     /* [B x m], NULL = 0 */
  const double *lbg, *ubg; /* [B x m], both or neither (landing_kino_setup_batch gives them) */
  double *grad_x;          /* [B x n_x] */
  double *viol;            /* [B]: needs lbg / ubg */
  double *dual_inf;        /* [B] */
  double *compl_inf;       /* [B]: needs lbg / ubg */
} landing_kino_kkt_io;
/* ks (QN, q/qd_term_ref of the cost) is required only when lam_f != NULL.  LANDING_ERR_ARG, with the context left
 * usable: a NULL ctx / pb / pb->dt / io / x, B < 0, lam_f without ks, only one of lbg / ubg, viol or compl_inf without
 * the bounds. */
int landing_kino_kkt_batch(landing_ctx *ctx, long long B, int memspace, int layout, const landing_kino_problem *pb,
                           const landing_kino_setup *ks, const landing_kino_kkt_io *io);

/* Primal-dual Newton step of one interior-point iteration of the kino-dynamic NLP, with IPOPT's inertia correction, per
 * scenario.  IPOPT's form (oracle/ip_ref.c): every inequality row i has a slack s_i and bound multipliers zL_i (finite
 * lbg_i) and zU_i (finite ubg_i); y has CasADi's sign, L = f + y'(g - s); W = the hess of landing_kino_hess_batch with
 * lam_f = 1, lam_g = y.  The step solves
 *   (W + delta_w I) dx + J' dy       = -(grad_f + J' y)
 *   -dy_i - dzL_i + dzU_i            = y_i + zL_i - zU_i         inequality rows
 *   J_E dx                           = -(g_E - lbg_E)            equality rows
 *   J_I dx - ds                      = -(g_I - s)
 *   zL ds + (s - lbg) dzL            = mu - zL (s - lbg)         finite lbg
 *   -zU ds + (ubg - s) dzU           = mu - zU (ubg - s)         finite ubg
 * The row kinds are structural: the equality rows are rows 0..23 (X_0, c_0) and the 12 dynamics rows of each knot, every
 * other row is an inequality row (one with both bounds infinite has y + dy = 0).  delta_w follows IPOPT's schedule from
 * dw_last: the first trial is dw_last / 3 (0 if that is below 1e-7, or if dw_last = 0); after a failed factorisation
 * 1e-4 (dw_last = 0) or max(1e-20, dw_last / 3), then x100 (at most 8 times while dw_last = 0) or x8; above 1e40 the
 * scenario fails.  A factorisation fails when a Cholesky pivot of a stage's control block is <= 1e-14, which is exactly
 * "the reduced Hessian on the null space of J_E is not positive definite".  Per scenario: status 0 (step found),
 * LANDING_ST_FACTOR_FAIL or LANDING_ST_NOT_INTERIOR (a slack not strictly inside a finite bound of its row, or a
 * multiplier of a finite bound <= 0): then every output vector of that scenario is NaN, and no other scenario is touched.
 * delta_w: the value used (NaN for a non-interior iterate); n_factor: factorisations tried.  With tau in (0, 1) and the
 * alpha outputs: the fraction-to-boundary step lengths alpha_pr = max a <= 1 with (s - lbg) + a ds >= (1 - tau)(s - lbg)
 * and (ubg - s) - a ds >= (1 - tau)(ubg - s), alpha_du the same for zL + a dzL and zU + a dzU.  ds, dzL, dzU are 0 on
 * equality rows and dzL / dzU on infinite bounds; s, zL, zU are not read there.  Results are the same bits in both
 * layouts, both memory spaces and from run to run; every output entry is written on every call; B = 0 launches nothing. */
typedef struct landing_kino_step_io {
  const double *g, *jac, *hess, *grad_f; /* [B x m], [B x nnzJ], [B x nnzH], [B x n_x] at the iterate */
  const double *s, *y, *zL, *zU;         /* [B x m] */
  const double *lbg, *ubg;               /* [B x m] */
  const double *mu, *dw_last;            /* [B] in both layouts */
  double *dx;                            /* [B x n_x] */
  double *ds, *dy, *dzL, *dzU;           /* [B x m] */
  double *delta_w;                       /* [B] */
  int *n_factor, *status;                /* [B] */
  double tau;                            /* fraction-to-boundary parameter, needed with alpha_pr / alpha_du */
  double *alpha_pr, *alpha_du;           /* [B], both or neither (optional) */
} landing_kino_step_io;
/* LANDING_ERR_ARG, with the context left usable: a NULL ctx / io / required pointer, B < 0, only one alpha output, or
 * tau outside (0, 1) with the alpha outputs. */
int landing_kino_step_batch(landing_ctx *ctx, long long B, int memspace, int layout, const landing_kino_step_io *io);

/* Interior-point solve of the kino-dynamic NLP, one per drop condition: the second half of the reference's pipeline
 * (main_scripts/landing_optimization.m:300-377: SRB solve, then the KNITRO kino-dynamic solve from its solution).  The
 * method is IPOPT's primal-dual filter line search as oracle/ip_ref.c restates it for the SRB solver (DESIGN.md 3, 3.2):
 * relaxed bounds, slacks on the inequality rows (the structural row kinds of landing_kino_step_batch), the monotone
 * barrier update, the filter with switching condition and Armijo test, IPOPT's inertia correction, and the jamming
 * watchdog with re-centring instead of a restoration phase.  The landing_options fields used keep their meanings
 * (max_iter, tol, constr_viol_tol, dual_inf_tol, compl_inf_tol, mu_init, bound_push, bound_frac, bound_relax_factor,
 * jam_iters, jam_alpha, max_restarts, restart_mu).  The bounds and, without x0, the initial guess are those of
 * landing_kino_setup_batch for the drop (from x_srb, or from the reference trajectories when x_srb is NULL); the cost is
 * the terminal cost of landing_kino_cost_batch.  Buffers are AoS, host or device per memspace.  Per scenario: status
 * (CONVERGED, MAX_ITER, LINESEARCH_FAIL, NAN -- a NaN in the drop, the guess or any measured quantity --, FACTOR_FAIL),
 * iters, x_star, f_star = f(x_star), and optionally lam_g (y, CasADi's sign), restarts and the final viol / dual_inf /
 * compl_inf with the definitions of landing_kino_kkt_batch at (x_star, lam_f = 1, lam_g) and the bounds of the drop.
 * A scenario's result is the same bits whether it is solved alone or in any batch, in any order, from host or device
 * buffers.  The host synchronises the context's stream once per outer round and once per line-search round to read
 * back a count; otherwise, with device buffers, the call only enqueues.  stats (HOST pointer, optional): outer rounds,
 * line-search rounds and compactions of the call; the launch count is documented beside the call in capi.cu.
 * MEMORY: the call keeps the state of all B scenarios on the device at once (two copies of the persistent state, the
 * round's Jacobian, Hessian and direction, the trial point): about 0.73 MB per scenario at N = 21 and 1.41 MB at N = 40,
 * in one allocation that grows with B.  There is no chunking: a batch whose scratch does not fit the device fails with
 * LANDING_ERR_CUDA (the context stays usable); split such a batch into several calls. */
typedef struct landing_kino_solve_io {
  const double *drops; /* [B x 12] (q_init, qd_init), required */
  const double *x_srb; /* [B x (36N-24)] SRB solutions (landing_solve_batch's x_star) or NULL */
  const double *x0;    /* [B x n_x] initial guess or NULL: then the guess of landing_kino_setup_batch from x_srb */
  double *x_star;      /* [B x n_x] */
  double *f_star;      /* [B]      terminal cost at x_star */
  double *lam_g;       /* [B x m]  y with CasADi's sign (L = f + lam_g' g), optional */
  double *viol, *dual_inf, *compl_inf; /* [B] final measures (the definitions of landing_kino_kkt_batch), optional */
  int *status, *iters; /* [B] */
  int *restarts;       /* [B] re-centrings used, optional */
  long long *stats;    /* [3] HOST: outer rounds, line-search rounds, compactions; optional */
} landing_kino_solve_io;
/* LANDING_ERR_ARG, with the context left usable: a NULL ctx / pb / pb->dt / ks / opt / io / drops / x_star / f_star /
 * status / iters, B < 0, or options out of range (max_iter < 0, a tolerance, mu_init or bound_push <= 0, bound_frac
 * outside (0, 0.5], bound_relax_factor < 0, jam_iters < 0, jam_alpha < 0, max_restarts < 0, restart_mu NaN).  B = 0
 * launches nothing. */
int landing_kino_solve_batch(landing_ctx *ctx, long long B, int memspace, const landing_kino_problem *pb,
                             const landing_kino_setup *ks, const landing_options *opt, const landing_kino_solve_io *io);

/* Measured FP64 FMA throughput of the context's device in TFLOP/s (a DFMA micro-kernel timed with CUDA
 * events): the roofline denominator of the interior-point kernel, which is FP64-pipe bound by design. */
int landing_fp64_peak(landing_ctx *ctx, double *tflops);

/* STREAM CONTRACT.  Every context owns one non-blocking CUDA stream (landing_stream).  Calls with LANDING_HOST buffers
 * copy in, run and copy out on it and return after synchronising it.  Calls with LANDING_DEVICE buffers only ENQUEUE work
 * on it and return immediately: the caller orders its own streams against landing_stream(ctx) -- inputs produced on
 * another stream need an event wait before the call, consumers an event wait after it (cudaStreamWaitEvent), or call
 * landing_synchronize().  A context is not thread-safe (one host thread at a time per context); different contexts,
 * also on the same device, may be used concurrently from different threads.  Every call leaves the calling thread's
 * current CUDA device as it found it. */
int landing_synchronize(landing_ctx *ctx);

/* number of kernel launches issued by this context so far (bench accounting) */
long long landing_launch_count(const landing_ctx *ctx);
/* CUDA stream (cudaStream_t) the context launches on; for event timing by the caller */
void *landing_stream(const landing_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif
