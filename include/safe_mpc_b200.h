/*
 * safe_mpc_b200.h -- C ABI of the B200-native batched RTI-MPC engine.
 *
 * This is the drop-in boundary for the hot path of idra-lab/safe-mpc: everything the
 * reference delegates to `acados_template.AcadosOcpSolver` + CasADi/adam/L4CasADi generated
 * code (reference call sites: src/safe_mpc/controller.py:141-164,193,208-209,247) plus the
 * per-problem control logic wrapped around it (controller.py:169-184,226-231,274-284,
 * 375-388,448-498; env_model.py:192-206; scripts/mpc.py:102-291), batched over B
 * independent problems that live on one GPU.
 *
 * Conventions
 *   - plain C, no torch types; every array argument is a caller-owned pointer.
 *   - `mem` says where the caller's arrays live: SMPC_HOST (pageable or pinned host memory;
 *     the library does the H2D/D2H copies on its own stream and returns after they complete)
 *     or SMPC_DEVICE (device pointers, e.g. torch tensor .data_ptr(); no copies, no sync).
 *   - caller-side layout is batch-major row-major: x[B][nx], xg[B][N+1][nx], ug[B][N][nu].
 *   - every function returns 0 on success, <0 on API/CUDA error (text via smpc_last_error).
 *     Per-problem solver status uses the acados codes the reference consumes
 *     (controller.py:166,279,379,489): 0 ok, 1 NaN, 2 max-iter, 3 min-step, 4 QP failure.
 *   - one handle per (GPU, controller type, N, batch); not re-entrant; no global state.
 *   - there is NO CPU fallback: without a CUDA device smpc_create fails with SMPC_ERR_CUDA.
 */
#ifndef SAFE_MPC_B200_H
#define SAFE_MPC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMPC_NQ 5            /* config.yaml:10 n_dofs (compile-time in this build)     */
#define SMPC_NX (2 * SMPC_NQ)
#define SMPC_NU SMPC_NQ
#define SMPC_NZ (SMPC_NX + SMPC_NU)
#define SMPC_NPAIR 6         /* config.yaml:205-216 collision_pairs (capsule-capsule)  */
#define SMPC_MAX_POINTS 8    /* moving points: [0]=EE, then capsule end points          */
#define SMPC_HID 256         /* config.yaml:66 network_size hidden width                */
#define SMPC_NN_NPARAM (SMPC_HID * SMPC_NX + SMPC_HID + 2 * (SMPC_HID * SMPC_HID + SMPC_HID) + SMPC_HID + 1)
#define SMPC_MAX_N 128       /* longest supported horizon                               */

/* memory space of caller arrays */
#define SMPC_HOST 0
#define SMPC_DEVICE 1

/* error codes */
#define SMPC_OK 0
#define SMPC_ERR_ARG (-1)
#define SMPC_ERR_CUDA (-2)
#define SMPC_ERR_UNSUPPORTED (-3)

/* controller state machines (reference utils.py:64-75 + classes in controller.py) */
enum {
  SMPC_CTRL_NAIVE = 0,          /* NaiveController            controller.py:251-284 */
  SMPC_CTRL_ZEROVEL = 1,        /* TerminalZeroVelocity       controller.py:295-317 */
  SMPC_CTRL_ST = 2,             /* STController               controller.py:319-361 */
  SMPC_CTRL_STWA = 3,           /* STWAController             controller.py:364-393 */
  SMPC_CTRL_HTWA = 4,           /* HTWAController             controller.py:396-401 */
  SMPC_CTRL_RECEDING = 5,       /* RecedingController         controller.py:404-502 */
  SMPC_CTRL_REAL_RECEDING = 6,  /* RealReceding               controller.py:504-565 */
  SMPC_CTRL_EVERYWHERE = 7,     /* ControllerSafeSetEverywhere controller.py:646-689 */
  SMPC_CTRL_BACKUP = 8,         /* SafeBackupController       controller.py:692-712 */
  SMPC_CTRL_PARALLEL = 9        /* ParallelController         controller.py:567-644 (N solves per step, one per candidate node) */
};

/* which stages carry the viability-network row (safe_set.py:82-104) */
enum {
  SMPC_NN_NONE = 0,
  SMPC_NN_TERMINAL = 1,         /* ST / STWA / HTWA / RealReceding                  */
  SMPC_NN_RECEDING = 2,         /* stages 1..N-1 gated by p[4], terminal always on */
  SMPC_NN_EVERYWHERE = 3,       /* stages 1..N, never gated                        */
  SMPC_NN_PARALLEL = 4          /* stages 1..N, all hard, only the candidate node of the running solve is on (controller.py:578-588) */
};

enum { SMPC_NN_STRICT = 0, SMPC_NN_TF32X3 = 1 };

enum { SMPC_PREC_F64 = 0, SMPC_PREC_F32 = 1 };

enum { SMPC_COST_ZERO = 0, SMPC_COST_EXT = 1, SMPC_COST_NLS = 2 };

/*
 * Stage record: the linearisation of one stage of one problem, SMPC_REC doubles.
 * Written by the linearisation kernel, consumed by the QP kernel, readable through
 * smpc_get_lin() for parity tests.  QP variable order is z = [du(5); dq(5); dv(5)].
 */
#define SMPC_REC 192
#define SMPC_REC_U 0        /* 5   u_guess[k] (zeros at k=N)                                     */
#define SMPC_REC_X 5        /* 10  x_guess[k]                                                    */
#define SMPC_REC_G 15       /* 15  cost gradient, [u q v], scaled by the stage weight            */
#define SMPC_REC_HQQ 30     /* 15  q-block of the cost Hessian, lower triangle row-major, scaled */
#define SMPC_REC_TAU 45     /* 5   tau(x,u)                                                      */
#define SMPC_REC_JTAU 50    /* 75  d tau / d [u q v], row-major 5x15                             */
#define SMPC_REC_DIST 125   /* 6   squared capsule distances                                     */
#define SMPC_REC_JDIST 131  /* 30  d dist / dq, row-major 6x5                                    */
#define SMPC_REC_NN 161     /* 1   viability row value (5e5 when gated off)                      */
#define SMPC_REC_JNN 162    /* 10  d c / d [q v]                                                 */
#define SMPC_REC_B 172      /* 10  dynamics offset  A x_k + B u_k - x_{k+1}  (zeros at k=N)      */
#define SMPC_REC_HU 182     /* 1   diagonal of the u-block of the Hessian incl. Levenberg-Marquardt */
#define SMPC_REC_HV 183     /* 1   diagonal of the v-block incl. LM                              */
#define SMPC_REC_HQ 184     /* 1   LM term added to the diagonal of the q-block                  */
#define SMPC_REC_NNROW 185  /* 1   1.0 if the stage has a viability row                          */
#define SMPC_REC_SOFT 186   /* 1   L1 penalty of the soft viability row, <0: hard                */
#define SMPC_REC_NTAU 187   /* 1   number of torque rows (5, or 0 at k=N)                        */
#define SMPC_REC_NDIST 188  /* 1   number of capsule rows (6, or 0 at stage 0 when noise>0)      */

/* QP constraint slots of one stage (lam/t layout of smpc_get_qp): rows are
 * [box x (10)] [tau (5)] [dist (6)] [nn (1)], slot = side*SMPC_QP_NR + row, then the two slacks */
#define SMPC_QP_NR 22
#define SMPC_QP_NC (2 * SMPC_QP_NR + 2)

/*
 * Static description of one OCP family (shared by all B problems of a handle).
 * Filled by the host layer from config.yaml + URDF exactly as the reference's
 * Parameters / AdamModel / AbstractController.__init__ do (parser.py:60-221,
 * env_model.py:18-165, controller.py:12-125).
 */
typedef struct smpc_problem {
  /* ---- dimensions and modes ---- */
  int32_t nq;                    /* must equal SMPC_NQ                                            */
  int32_t N;                     /* horizon (config.yaml:5, --horizon)                            */
  int32_t n_pairs;               /* must equal SMPC_NPAIR                                         */
  int32_t n_points;              /* <= SMPC_MAX_POINTS                                            */
  int32_t controller;            /* SMPC_CTRL_*                                                   */
  int32_t nn_rows;               /* SMPC_NN_*                                                     */
  int32_t nn_terminal_soft;      /* terminal NN row has an L1 slack (controller.py:348-354)       */
  int32_t stage0_collision_rows; /* 0 when --noise > 0 (controller.py:68-75), else 1              */
  int32_t cost_type;             /* SMPC_COST_*                                                   */
  int32_t abort_flag;            /* config.yaml:58                                                */
  int32_t qp_iter_max;           /* config.yaml:18 qp_max_iter                                    */
  int32_t lm_scale_dt;           /* 1: LM term is scaled by the stage time step for k<N (acados
                                    ocp_nlp_approximate_qp_matrices convention, see DESIGN.md)    */
  int32_t qp_cond_pred_corr;     /* HPIPM BALANCE: 1                                              */
  int32_t nn_precision;          /* SMPC_NN_STRICT: fp32 weights, fp64 accumulation (FP64 pipe);
                                    SMPC_NN_TF32X3: fp32-class evaluation on the tensor cores (the precision of the
                                    reference's libtorch call, safe_set.py:76-94), see csrc/mlp_tc.cu              */
  int32_t qp_keep_slots;         /* 1: never compact the solver's slots during a solve, so that smpc_get_lin / smpc_get_qp stay
                                    available for every batch size (tests, the merit line search of the guess generator); 0: default */
  int32_t precision;             /* SMPC_PREC_F64 (default): the QP solver state is stored in fp64, results agree with the fp64 reference path
                                    to 1e-6; SMPC_PREC_F32: everything a solve streams from HBM (stage records, search directions, condensed
                                    matrices, Riccati factors) is stored in fp32, the iterate and all arithmetic stay fp64 -- 40 % less HBM
                                    traffic per interior-point iteration, trajectories within 1e-3 relative (BASELINE.json north_star, fp32
                                    mode); pair it with qp_tol_* = 1e-5 / 1e-6 (the fp32 search direction bottoms the residuals out near 1e-5) */
  /* ---- scalars ---- */
  double dt;                     /* config.yaml:7                                                 */
  double q_weight, r_weight;     /* config.yaml:35,39                                             */
  double lm;                     /* levenberg_marquardt, config.yaml:21                           */
  double alpha;                  /* safety margin in percent, p[3]                                */
  double eps;                    /* config.yaml:48                                                */
  double slack_penalty_e;        /* zl_e = zu_e of the soft terminal row (ws_r for ST, ws_t for receding) */
  double tol_x, tol_tau, tol_obs, tol_safe, tol_conv; /* config.yaml:42-49                       */
  double qp_mu0, qp_tol_stat, qp_tol_eq, qp_tol_ineq, qp_tol_comp, qp_alpha_min, qp_reg_prim;
  double gravity[3];             /* world-frame gravity acceleration, (0,0,-9.80665)              */
  double qp_maxiter_accept;      /* acados' SQP_RTI takes the step of a QP that ran into qp_iter_max (controller.py:166 sees status 0).
                                    Whether an INFEASIBLE QP ends at qp_iter_max or at the minimum step length is decided by rounding
                                    (its multipliers diverge; DESIGN.md section 4), so a max-iter exit only counts as solved when every
                                    residual is within this factor of its tolerance (default 1e3); <= 0: every max-iter exit is accepted */
  double reserved_d[7];
  /* ---- serial chain (lumped over locked/fixed joints, see host/robot_model.py) ---- */
  double joint_R[SMPC_NQ][9];    /* row-major rotation parent-body <- joint frame at q=0          */
  double joint_p[SMPC_NQ][3];    /* joint-frame origin in the parent body frame                   */
  double joint_axis[SMPC_NQ][3]; /* unit axis in the joint's own frame                            */
  double inertial[SMPC_NQ][10];  /* nominal: m, c[3], Ixx,Iyy,Izz,Ixy,Iyz,Ixz about the CoM       */
  /* ---- bounds ---- */
  double x_min[SMPC_NX], x_max[SMPC_NX];     /* model bounds widened by q_margin (env_model.py:115-121) */
  double lbx[SMPC_NX], ubx[SMPC_NX];         /* OCP box, stages 1..N-1 (controller.py:49-51)            */
  double lbx_e[SMPC_NX], ubx_e[SMPC_NX];     /* OCP box, stage N (controller.py:53-55,300-306,701-707)  */
  double tau_min[SMPC_NU], tau_max[SMPC_NU]; /* env_model.py:113-114                                    */
  double ee_ref[3];                          /* config.yaml:73                                          */
  /* ---- points rigidly attached to bodies; point 0 is the end effector ---- */
  int32_t point_body[SMPC_MAX_POINTS];
  double point_local[SMPC_MAX_POINTS][3];
  /* ---- capsule-capsule pairs: moving segment (points pa,pb) vs fixed world segment (C,D) ---- */
  int32_t pair_pa[SMPC_NPAIR], pair_pb[SMPC_NPAIR];
  double pair_C[SMPC_NPAIR][3], pair_D[SMPC_NPAIR][3];
  double pair_lo_ocp[SMPC_NPAIR];  /* (r1+r2+2*margin)^2            env_model.py:266 */
  double pair_lo_chk[SMPC_NPAIR];  /* (r1+r2)^2 - tol_obs           env_model.py:268 */
  double pair_hi;                  /* 1e6                           env_model.py:266 */
  /* ---- viability network (safe_set.py:26-43,82-87) ---- */
  double nn_mean[SMPC_NQ], nn_std[SMPC_NQ];
  const float* nn_weights;         /* host pointer, SMPC_NN_NPARAM floats:
                                      W1[HID][NX] b1[HID] W2[HID][HID] b2[HID] W3[HID][HID] b3[HID] W4[HID] b4[1]
                                      (row-major, torch nn.Linear convention y = W x + b); may be NULL if nn_rows==0 */
} smpc_problem_t;

typedef struct smpc_handle smpc_handle_t;
typedef struct smpc_sim smpc_sim_t;

/* --- life cycle (replaces AcadosOcpSolver(ocp, json_file, generate, build), controller.py:247) --- */
int smpc_create(const smpc_problem_t* prob, int32_t batch, int32_t device, smpc_handle_t** out);
void smpc_destroy(smpc_handle_t* h);
/* text of the last error of this handle (h may be NULL: last error of smpc_create on this thread) */
const char* smpc_last_error(const smpc_handle_t* h);
const char* smpc_version(void);

/* --- per-problem plant data --- */
/* perturbed inertial parameters of the simulated plant, [B][NQ][10]
 * (replaces update_randomized_dynamics + the z1_randomized*.urdf files, env_model.py:321-328) */
int smpc_set_plant_inertial(smpc_handle_t* h, const double* inertial, int32_t mem);
/* additive torque noise drawn by the host with default_rng(seed=i) (mpc.py:126, env_model.py:196), [B][NU] */
int smpc_set_torque_noise(smpc_handle_t* h, const double* tau_noise, int32_t mem);

/* --- stage parameters of the cost: the end-effector reference per stage ---
 * The reference sets p = [cost.traj[:, current_step + i], alpha, gate] on every stage of every solve (controller.py:153-156); for the
 * reach costs cost.traj is ee_ref repeated (cost_definition.py:29-31,67,89), for the tracking costs a time-indexed path (Tracking8*,
 * TrackingMovingCircle*, cost_definition.py:102-288).  traj[n][3] is that array (one row per control step, shared by the batch like
 * the reference's cost object); stage k of problem b is linearised around traj[min(current_step[b] + k, n - 1)], current_step being
 * the per-problem counter that smpc_controller_step advances and smpc_reset_controller clears.  n = 0: back to the constant
 * smpc_problem_t::ee_ref.  (alpha and the gate are per handle / per problem state: smpc_problem_t::alpha, SMPC_STATE_R.) */
int smpc_set_ee_trajectory(smpc_handle_t* h, const double* traj, int32_t n, int32_t mem);

/* --- warm start (controller.py:195-200,390-393) --- */
int smpc_set_guess(smpc_handle_t* h, const double* xg, const double* ug, int32_t mem);
int smpc_get_guess(smpc_handle_t* h, double* xg, double* ug, int32_t mem);
int smpc_get_temp(smpc_handle_t* h, double* x_temp, double* u_temp, int32_t mem);
/* reset_controller(): fails=0, r=N, current_step=0 (controller.py:234-238,359-361,444-446) */
int smpc_reset_controller(smpc_handle_t* h);

/* --- one RTI iteration = AbstractController.solve(x0) (controller.py:136-167) ---
 * uses the stored guess; writes x_temp/u_temp (fetch with smpc_get_temp) and status[B].
 * active[B] (may be NULL = all): problems with active==0 are skipped and keep their state;
 * status may be NULL. */
int smpc_rti_solve(smpc_handle_t* h, const double* x0, const uint8_t* active, int32_t* status, int32_t mem);

/* --- controller.step(x) -> (u, abort_flag) for every problem (controller.py:274-284 etc.) --- */
int smpc_controller_step(smpc_handle_t* h, const double* x, const uint8_t* active,
                         double* u, uint8_t* abort_flag, int32_t mem);

/* --- plant step = AdamModel.integrate(x,u) (env_model.py:192-206) --- */
int smpc_plant_step(smpc_handle_t* h, const double* x, const double* u,
                    double* x_next, double* a_applied, int32_t mem);

/* --- pieces exposed for parity tests and for the host-side mirror of AdamModel --- */
/* tau_fun(x,u) (env_model.py:80-83), n rows */
int smpc_tau(smpc_handle_t* h, int32_t n, const double* x, const double* u, double* tau, int32_t mem);
/* Torque-input dynamics with sensitivities -- extension row (f)4 of SURVEY.md section 8 (north_star: "RNEA/ABA inside an explicit RK4
   integrator that emits state/control sensitivities"); the reference has no counterpart call: its OCP dynamics are the constant
   double integrator f_fun (env_model.py:58-71).  x' = [v; M(q)^-1 (tau - h(q, v))] with the reference's mass_matrix_fun /
   bias_force_fun (env_model.py:42-43) on the controller model; one explicit RK4 step of length dt for n rows:
   x_next [n][10], A = d x_next / d x [n][10][10], B = d x_next / d tau [n][10][5] (row-major; A and / or B may be NULL). */
int smpc_rk4_sens(smpc_handle_t* h, int32_t n, const double* x, const double* tau, double dt,
                  double* x_next, double* A, double* B, int32_t mem);
/* ee_fun(x) (env_model.py:91-95) [n][3] and the 6 collision-constraint values (env_model.py:263-271) [n][6] */
int smpc_kinematics(smpc_handle_t* h, int32_t n, const double* x, double* ee, double* dist, int32_t mem);
/* nn_func_x(x): c(x) with the handle's alpha (safe_set.py:100-102) and its gradient [n][NX] (grad may be NULL) */
int smpc_nn_constraint(smpc_handle_t* h, int32_t n, const double* x, double* c, double* grad, int32_t mem);
/* stage records of the last smpc_rti_solve, [B][N+1][SMPC_REC] */
int smpc_get_lin(smpc_handle_t* h, double* lin, int32_t mem);
/* QP solution of the last smpc_rti_solve: dz[B][N+1][15] ([du;dx]; terminal stage: dx in the first 10),
 * pi[B][N][10], lam/t[B][N+1][SMPC_QP_NC]; any pointer may be NULL */
int smpc_get_qp(smpc_handle_t* h, double* dz, double* pi, double* lam, double* t, int32_t mem);

/* --- per-problem controller state (controller.py attrs fails, r, last_status, x_viable) --- */
enum { SMPC_STATE_FAILS = 0, SMPC_STATE_R = 1, SMPC_STATE_STATUS = 2, SMPC_STATE_QP_ITER = 3, SMPC_STATE_QP_STATUS = 4 };
int smpc_get_state_i32(smpc_handle_t* h, int32_t field, int32_t* out, int32_t mem);
int smpc_set_state_i32(smpc_handle_t* h, int32_t field, const int32_t* in, int32_t mem);
int smpc_get_x_viable(smpc_handle_t* h, double* x_viable, int32_t mem);
/* max-norm residuals of the last QP of every problem [B][5]: stationarity, dynamics, inequality, complementarity, mu (what acados'
 * get_stats('qp_res..') / HPIPM's get_max_res_* report; controller.py:192-193 only reads the timing fields) */
int smpc_get_qp_residuals(smpc_handle_t* h, double* res5, int32_t mem);

/* --- closed loop = the per-test body of scripts/mpc.py:102-291, batched ---
 * `backup` is a handle created with controller = SMPC_CTRL_BACKUP and N = back_hor (mpc.py:54-73),
 * same batch.  One smpc_sim_step advances every live problem by one control step: abort following /
 * PD hold / controller.step, backup solve on abort, plant step, bounds and collision checks.
 * Asynchronous towards the caller (nothing is copied back), but not free of host synchronisation: the QP solver reads one pair of
 * counters per interior-point iteration (csrc/qp.cu) unless the batch is small enough for the solo kernel. */
int smpc_sim_create(smpc_handle_t* main_ctrl, smpc_handle_t* backup, int32_t n_steps, smpc_sim_t** out);
void smpc_sim_destroy(smpc_sim_t* s);
int smpc_sim_reset(smpc_sim_t* s, const double* x_init, int32_t mem);
int smpc_sim_step(smpc_sim_t* s);
int smpc_sim_run(smpc_sim_t* s, int32_t n_steps);
/* outcome bits after n_steps: see SMPC_OUT_*; runs the convergence test of mpc.py:273 first */
#define SMPC_OUT_CONVERGED 1  /* conv_idx        */
#define SMPC_OUT_COLLIDED 2   /* collisions_idx  */
#define SMPC_OUT_ABORTED 4    /* was added to viable_idx at least once (before the final filtering) */
int smpc_sim_get_outcome(smpc_sim_t* s, int32_t* outcome, int32_t mem);
/* logs: x[B][n_steps+1][NX], u[B][n_steps][NU], NaN after termination (mpc.py:114-116) */
int smpc_sim_get_log(smpc_sim_t* s, double* x, double* u, int32_t mem);
/* x_viable of the first abort of each problem [B][NX] (NaN if none) */
int smpc_sim_get_x_viable(smpc_sim_t* s, double* xv, int32_t mem);
/* out[0] = RTI solves of the main controller, out[1] = backup solves, out[2] = problem-steps simulated,
 * out[3] = total IPM iterations */
int smpc_sim_get_counters(smpc_sim_t* s, int64_t* out4);

/* --- timing of the last rti_solve/controller_step, milliseconds, CUDA events (replaces get_stats, controller.py:192-193) ---
 * out[0]=time_lin out[1]=time_sim out[2]=time_qp out[3]=time_qp_solver_call out[4]=time_glob out[5]=time_reg out[6]=time_tot */
int smpc_get_times(smpc_handle_t* h, double* out7);
/* per-kernel timing of the QP solver (the split interior-point kernels of csrc/qp.cu), CUDA events on the streams the
 * kernels are launched on.  smpc_set_profiling(h, 1) makes every following solve record one event pair per kernel (and
 * synchronise at its end); smpc_get_profile returns, for the last solve, the summed duration [ms] and the launch count per
 * kernel kind (index = SMPC_PROF_*), the span of the whole solve [ms] and the IPM iterations the host sequenced (those of the slowest
 * problem; iterations that SMPC_PROF_SOLO -- one launch that runs whole iterations on the device -- performed are not counted). */
enum { SMPC_PROF_INIT = 0, SMPC_PROF_PREP = 1, SMPC_PROF_CTL = 2, SMPC_PROF_RIC1 = 3, SMPC_PROF_STEP0 = 4, SMPC_PROF_RIC2 = 5,
       SMPC_PROF_STEP1 = 6, SMPC_PROF_RED = 7, SMPC_PROF_COMPACT = 8, SMPC_PROF_STEP2 = 9, SMPC_PROF_FINAL = 10, SMPC_PROF_SOLO = 11, SMPC_PROF_N = 12 };
int smpc_set_profiling(smpc_handle_t* h, int32_t enable);
int smpc_get_profile(smpc_handle_t* h, double* ms /*[SMPC_PROF_N]*/, int32_t* count /*[SMPC_PROF_N]*/, double* span_ms, int32_t* iterations);
/* number of kernels this handle has launched so far (bench.py "gpu_launches") */
int64_t smpc_launch_count(const smpc_handle_t* h);
/* the CUDA stream the handle launches on (cudaStream_t as void*) */
void* smpc_stream(smpc_handle_t* h);
/* make the handle launch on the caller's stream (cudaStream_t as void*; it must belong to the handle's device and outlive the
 * handle or the next smpc_set_stream) -- what a per-call cudaStream_t argument would do (SURVEY.md section 8(b)), set once instead of
 * passed to every function.  NULL: back to a private non-blocking stream.  Returns after the work queued so far has finished.
 * The legacy default stream is not supported (the QP solver orders its internal streams with events against this one).
 * CUDA graphs: while this stream is being captured, smpc_rti_solve, smpc_controller_step, smpc_plant_step and smpc_sim_step are captured
 * with their whole QP loop (a conditional WHILE node; the backup solve of smpc_sim_step in a conditional IF node; device pointers only,
 * not the parallel controller, no profiling; INTEGRATION.md section 3). */
int smpc_set_stream(smpc_handle_t* h, void* stream);
int smpc_sync(smpc_handle_t* h);

/* --- measured machine peaks for the roofline of bench.py (SURVEY.md section 8(d): the dynamics / QP kernels are charged to the
 * FP64 FMA pipe; MEASURED_PEAKS.json has no FP64 number): dense FMA rate of the FP64 and FP32 pipes, TFLOP/s, CUDA events --- */
int smpc_measure_peaks(int32_t device, double* fp64_tflops, double* fp32_tflops);

#ifdef __cplusplus
}
#endif
#endif /* SAFE_MPC_B200_H */
