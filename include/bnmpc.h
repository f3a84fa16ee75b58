/* bnmpc - B200-native batched NMPC solver: C-ABI of the drop-in boundary.
 *
 * This header is the whole boundary between the reference-facing host code (Python, ctypes) and the CUDA
 * implementation (libbnmpc.so, sm_100a).  Plain C types only.  Each entry point names the reference interface it
 * replaces (paths relative to the reference repo BroilerCompiler/drone-attitude-control); the arithmetic behind
 * those reference calls lives in acados / HPIPM / BLASFEO / CasADi-generated C, reached through
 * acados_template.AcadosOcpSolver / AcadosSimSolver (ctypes) - this library replaces that stack for this path.
 *
 * One handle <-> one device <-> one CUDA stream <-> `batch` independent OCP instances.  Not thread-safe.
 * All calls are asynchronous on the handle's stream except those that copy to host memory (they synchronise).
 * The handle owns every workspace; the caller owns every buffer it passes; no pointer is retained after a call
 * returns.  Return value: 0 on success, negative BNMPC_E_* on API errors (message via bnmpc_last_error()).
 * Per-instance solver outcomes use the acados status codes (reference src/Readme.md:14-20).
 *
 * Layouts.  "AoS" buffers are [batch][dim] row-major doubles (one acados-style vector per instance).
 * "Batch-minor" buffers are [...][dim][batch] doubles with the batch index contiguous (coalesced in HBM).
 * `on_device` != 0 means the pointer is device memory of the handle's device; 0 means host memory (pinned host
 * memory makes the copy asynchronous).  All API arrays are FP64 regardless of the compute precision.
 */
#ifndef BNMPC_H
#define BNMPC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNMPC_VERSION 210

/* models (reference src/force_model/dynamics.py:12-47, src/jerk_model/dynamics.py:12-52).  FORCE_DENSE solves the
 * force-model OCP without exploiting the x/z block structure (the generic coupled path; in-product cross-check). */
#define BNMPC_MODEL_FORCE 0
#define BNMPC_MODEL_JERK 1
#define BNMPC_MODEL_FORCE_DENSE 2
/* NOT in the reference: the plant model (src/plant.py:27-33, u = (theta, Fd)) as controller model - a nonlinear OCP that
 * exercises the general path (sensitivities per stage and SQP iteration, several SQP iterations per solve). */
#define BNMPC_MODEL_THRUST 3
/* NOT in the reference: the 3-D attitude-and-total-thrust model of the north-star (SURVEY 8f rank 2): states position (3),
 * velocity (3), attitude quaternion body->world (w, x, y, z); inputs total thrust T and body rates (wx, wy, wz):
 *   pdot = v,  vdot = (T / m) R(q) e3 - g e3,  qdot = 1/2 q (x) (0, w)       nx = 10, nu = 4, ny = 14, p = (mass, g).
 * Box constraints on thrust and body rates (all stages) and on position / velocity (stages 1..N-1), LINEAR_LS cost, ERK4.
 * The planar plant of src/plant.py:27-33 is its restriction to the x-z plane (theta = pitch about y, Fd = T).  It is served by
 * the acados-style surface - set / get / solve / solve_for_x0 / step_for_x0 / sim_step (x [batch][10], u [batch][substeps][4])
 * - and has no fused closed loop (bnmpc_closed_loop_run returns BNMPC_E_UNSUPPORTED). */
#define BNMPC_MODEL_ATT 4

#define BNMPC_FP64 0
#define BNMPC_FP32 1

/* acados return values, reference src/Readme.md:14-20 */
#define BNMPC_SUCCESS 0
#define BNMPC_FAILURE 1      /* NaN/Inf in x0, yref or p */
#define BNMPC_MAXITER 2      /* SQP iteration cap (or, in RTI mode, QP iteration cap) */
#define BNMPC_MINSTEP 3
#define BNMPC_QP_FAILURE 4   /* QP solver: minimum step / NaN */

/* API error codes */
#define BNMPC_E_ARG (-1)
#define BNMPC_E_FIELD (-2)
#define BNMPC_E_STAGE (-3)
#define BNMPC_E_CUDA (-4)
#define BNMPC_E_UNSUPPORTED (-5)

/* fields of set/get: reference `ocp_solver.set(stage, name, vec)` / `.get(stage, name)`
 * (src/force_model/controller.py:30-39, src/force_model/ocp.py:120-122) */
#define BNMPC_F_X 0      /* 'x'    stage 0..N,   dim nx   (get/set) */
#define BNMPC_F_U 1      /* 'u'    stage 0..N-1, dim nu   (get/set) */
#define BNMPC_F_YREF 2   /* 'yref' stage 0..N-1 dim nx+nu, stage N dim nx (set/get) */
#define BNMPC_F_LBX 3    /* 'lbx'  stage 0: x0 embedding (controller.py:30); stages 1..N-1: lower state bound of that stage */
#define BNMPC_F_UBX 4    /* 'ubx'  stage 0: x0 embedding (controller.py:31), must equal lbx; stages 1..N-1: upper state bound */
#define BNMPC_F_P 5      /* 'p'    stage ignored, dim 2 = (mass, g) of the controller model (north-star extension) */
#define BNMPC_F_PI 6     /* 'pi'   stage 0..N-1, dim nx   (get) */
#define BNMPC_F_LAM 7    /* 'lam'  stage 0..N-1, dim 2*(nu[+nx]) = [lbu, lbx, ubu, ubx] multipliers (get) */
#define BNMPC_F_LBU 8    /* 'lbu'  stage 0..N-1, dim nu: lower input bound of that stage (get/set) */
#define BNMPC_F_UBU 9    /* 'ubu'  stage 0..N-1, dim nu: upper input bound of that stage (get/set) */
/* Per-stage bounds ('lbu'/'ubu', and 'lbx'/'ubx' at stages >= 1): acados' ocp_solver.set accepts them at any stage; the
 * reference fixes its boxes once in create_ocp (src/force_model/ocp.py:62-76) and never sets them per stage.  Until the first
 * such set() every stage of every instance uses the boxes of bnmpc_config (lbu/ubu/lbx/ubx) and no kernel looks anything
 * up; the first set() allocates per-instance storage ([batch][N][2][nu+nx] doubles, initialised with those boxes) and
 * bnmpc_solve / bnmpc_solve_for_x0 switch to a second instantiation of the solve kernel that reads the bounds per stage.
 * bnmpc_closed_loop_run refuses (BNMPC_E_UNSUPPORTED) on such a handle. */

/* per-instance int32 statistics: reference `ocp_solver.get_stats(name)` */
#define BNMPC_STAT_STATUS 0
#define BNMPC_STAT_SQP_ITER 1
#define BNMPC_STAT_QP_ITER 2

typedef struct bnmpc_config {
    int32_t model;          /* BNMPC_MODEL_* */
    int32_t horizon;        /* N_horizon (reference src/params.py:121) */
    int32_t precision;      /* BNMPC_FP64 | BNMPC_FP32 */
    int32_t erk_stages;     /* OCP integrator, one step per interval.  1..4: explicit Runge-Kutta with that many stages (acados
                               ERK + sim_method_num_stages; jerk 1, src/jerk_model/ocp.py:86-87).  0: acados IRK with its
                               defaults - Gauss-Legendre collocation, 4 stages, 3 Newton iterations, sensitivities by the
                               implicit function theorem - the integrator_type of the force OCP (src/force_model/ocp.py:85).
                               The default of the force model is 4: for its affine dynamics ERK4 and the collocation both
                               return the exact discretisation (tests: equal to 1e-14), at a fraction of the work */
    int32_t sqp_max_iter;   /* acados nlp_solver_max_iter default 100 (nlp_solver_type SQP, src/force_model/ocp.py:86) */
    int32_t qp_max_iter;    /* acados qp_solver_iter_max default 50 */
    int32_t rti;            /* 1: one QP per solve, no NLP residual test (SQP_RTI of the north-star) */
    int32_t threads_per_block; /* reserved (ignored): the launch shape follows from the model and the horizon - one persistent
                               CTA per SM with as many warps (= instances in flight) as the on-chip memories hold */
    double dt;              /* interval length, tf / N (src/params.py:116, src/force_model/ocp.py:93) */
    double W[16];           /* diag of cost.W, order [x; u] (src/force_model/ocp.py:38-47) */
    double W_e[12];         /* diag of cost.W_e */
    double lbx[12], ubx[12]; /* state box, stages 1..N-1 (src/force_model/ocp.py:72-76) */
    double lbu[4], ubu[4];  /* input box, stages 0..N-1 (src/force_model/ocp.py:62-67) */
    double tol[4];          /* NLP tolerances stat, eq, ineq, comp (acados default 1e-6) */
    double qp_tol[4];       /* QP tolerances (acados passes the NLP tolerances on to HPIPM) */
    double mu0, thr0, alpha_min, lam_min, t_min; /* HPIPM arguments as acados sets them */
    /* plant integrator = AcadosSim of src/plant.py (src/force_model/ocp.py:98-104, src/jerk_model/ocp.py:97-104) */
    int32_t sim_erk_stages; /* force path 4, jerk path 1 */
    int32_t sim_substeps;   /* force path 1, jerk path ctrls_per_sample = 10 */
    double sim_dt;          /* force path dt, jerk path dt_conv */
} bnmpc_config;

/* Fills *cfg with the reference's configuration of `model` (OCP.create_ocp + create_ocp_solver + create_simulator). */
int bnmpc_config_default(int model, bnmpc_config* cfg);

/* AcadosOcpSolver(ocp) + AcadosSimSolver(sim)  (src/force_model/ocp.py:95-96,104): allocates everything. */
int bnmpc_create(const bnmpc_config* cfg, int batch, int device, void** handle);
int bnmpc_destroy(void* handle);
/* cudaStream_t to run on (default: a stream created by the handle). */
int bnmpc_set_stream(void* handle, void* cuda_stream);
int bnmpc_synchronize(void* handle);
/* dimensions of the configured model: nx, nu, ny (=nx+nu), ny_e (=nx), N, np, number of blocks */
int bnmpc_dims(void* handle, int32_t dims[7]);
/* workspace bytes held by the handle */
int64_t bnmpc_workspace_bytes(void* handle);

/* ocp_solver.set(stage, field, value) for all instances at once; value is AoS [batch][dim]. */
int bnmpc_set(void* handle, int stage, int field, const double* value, int on_device);
/* ocp_solver.get(stage, field); out is AoS [batch][dim]. */
int bnmpc_get(void* handle, int stage, int field, double* out, int on_device);
/* OCP.set_up_ocp in one call (src/force_model/ocp.py:117-122): AoS [batch][N*ny + ny_e] = yref_0 .. yref_{N-1}, yref_N.
 * Makes this stored yref the source of the solves again (after bnmpc_set_yref_row). */
int bnmpc_set_yref_all(void* handle, const double* value, int on_device);
/* The reference as the reference hands it to OCP.set_up_ocp (src/force_model/ocp.py:117-122): the whole trajectory, bound
 * once, plus a row index per control step (bnmpc_set_yref_row) instead of a window upload per step.
 *
 * bnmpc_set_ref_table copies `table` into memory the handle owns (cudaMemcpyAsync on the handle's stream; the call returns
 * when the copy is done, no pointer is retained) and counts it in bnmpc_workspace_bytes.  layout 1 = one [rows][cols] table
 * shared by all instances, 2 = [batch][rows][cols] (instance-major) - the numbering of bnmpc_closed_loop_args.ref_shared.
 * Row r = [xref_r (nx) | uref_r (nu) | ignored], cols >= nx + nu (the 8-column gen_circle_traj table of force / jerk, the
 * 14-column helix table of the 3-D model), rows >= N + 1.  The table stays FP64 in FP32 mode: the solve rounds what it
 * reads exactly as bnmpc_set_yref_all rounds the uploaded window, so both ways give bit-identical results.
 * table == NULL releases the binding.  Binding does not change the yref source; binding a new table or releasing it while
 * the old one is selected first stores the current window as the yref (one gather kernel), so the next solve sees the
 * same yref either way.  BNMPC_E_ARG for a layout other than 1 or 2, cols < nx + nu or rows < N + 1. */
int bnmpc_set_ref_table(void* handle, const double* table, int rows, int cols, int layout, int on_device);
/* OCP.set_up_ocp(row, xref, uref) for all instances: yref_k = [xref[row+k], uref[row+k]] (k < N), yref_N = xref[row+N],
 * read by bnmpc_solve / bnmpc_solve_for_x0 / bnmpc_step_for_x0 straight from the bound table - no copy, no kernel - until
 * bnmpc_set_yref_all or bnmpc_set(k, 'yref', v) is called.  bnmpc_set(k, 'yref', v) while the table is selected first
 * stores the current window as the yref (one gather kernel), then writes stage k: the same as bnmpc_set_yref_all(window)
 * followed by that set.  bnmpc_get(k, 'yref') while the table is selected returns the window's stage k (the values the
 * solve reads: rounded to float in FP32) and changes no handle state.  BNMPC_E_ARG with no table bound, or unless
 * 0 <= row and row + N < rows. */
int bnmpc_set_yref_row(void* handle, int row);
/* zero the primal iterate and multipliers (state of a freshly created acados solver) */
int bnmpc_reset(void* handle);
/* ocp_solver.solve() (src/force_model/controller.py:32): one acados-style SQP run per instance from the stored
 * iterate with the stored x0 / yref / p.  Per-instance status via bnmpc_get_stats. */
int bnmpc_solve(void* handle);
/* ocp_solver.solve_for_x0(x0_bar) of acados_template (used by the reference's dev scripts, src/force_model/ocp.py:162-164)
 * = set(0,'lbx',x0); set(0,'ubx',x0); solve(); get(0,'u'), for all instances in ONE call: x0 AoS [batch][nx] in,
 * u0 AoS [batch][nu] and status int32 [batch] out (either may be NULL).  In FP64 the inputs are copied straight into the
 * solver state and the outputs straight out of it: one kernel launch per call.
 * on_device: 0 = host buffers, returns when u0 / status are in host memory; 1 = device buffers, asynchronous on the handle's
 * stream; BNMPC_HOST_ASYNC (2) = PINNED host buffers, asynchronous - the copies and the solve are enqueued on the handle's
 * stream and the caller calls bnmpc_synchronize() before reading u0 / status (lets the caller enqueue the upload of the
 * next step's reference window behind this step's x0 instead of in front of it). */
#define BNMPC_HOST_ASYNC 2
int bnmpc_solve_for_x0(void* handle, const double* x0, double* u0, int32_t* status, int on_device);
/* One iteration of follow_trajectory (src/force_model/controller.py:26-48, src/jerk_model/controller.py:27-50) for all
 * instances in ONE call, with the yref set before (bnmpc_set_yref_all): x0 embedding + solve() + get(0,'u') + Converter.convert
 * + OCP.simulate_next_x including the noise draw.  x0 AoS [batch][nx] (plant state, + the carried acceleration a_i for the
 * jerk model); eps [batch] or NULL (the np.random.normal(0, noise) draw of each instance); p_plant AoS [batch][2] or NULL
 * (nominal).  Out: u0 [batch][nu], u_plant [batch][2] = (theta, Fd) of the last sub-step, status [batch], x_next
 * [batch][nx] = the next step's x0 (any of u0 / u_plant / status may be NULL).  Two kernel launches; on_device as for
 * bnmpc_solve_for_x0. */
int bnmpc_step_for_x0(void* handle, const double* x0, const double* eps, const double* p_plant, double* u0, double* u_plant,
                      int32_t* status, double* x_next, int on_device);
/* Parametric solution sensitivities at the stored solution of every instance (acados' eval_solution_sensitivity), for the
 * models whose Gauss-Newton Hessian is the exact Hessian of the Lagrangian (FORCE, JERK, FORCE_DENSE: affine dynamics,
 * LINEAR_LS cost); BNMPC_E_UNSUPPORTED for THRUST and ATT.  The KKT matrix is the x0-eliminated one of the converged QP with
 * Hessian diagonal dt W (W_e at stage N) + lam_lb / t_lb + lam_ub / t_ub: the stored multipliers, slacks recomputed from the
 * stored iterate as t_lb = max(v - lb, t_min), t_ub = max(ub - v, t_min), the instance's boxes (per-stage bounds when set).
 * With no bound active this is the exact derivative of the solution; with strict complementarity it tends to the
 * active-set derivative.  An instance whose last status is not BNMPC_SUCCESS, or that has no multipliers yet, gets NaN rows.
 * Computed in the handle's precision, FP64 in and out.  One kernel launch per call; the handle's state (iterate,
 * multipliers, statistics, yref source) is not changed.  on_device: 0 = host buffers, returns with the results in host
 * memory (staged through handle-owned device memory, allocated on first use, counted by bnmpc_workspace_bytes); 1 = device
 * buffers, asynchronous on the handle's stream.
 * d x_k / d x0 and d u_k / d x0 at the stored solution, stages 0 .. stages-1 (1 <= stages <= N+1, else BNMPC_E_ARG):
 * sens_x [batch][stages][nx][nx], sens_u [batch][min(stages, N)][nu][nx]; either may be NULL.  sens_x[0] = I. */
int bnmpc_eval_sens_x0(void* handle, int stages, double* sens_x, double* sens_u, int on_device);
/* The adjoint (vector-Jacobian product) of the same derivative, one solve with the KKT matrix for any seed:
 * seed_x [batch][N+1][nx], seed_u [batch][N][nu] (NULL = zero, not both: BNMPC_E_ARG); grad_x0 [batch][nx] =
 * sum_k (d x_k / d x0)' seed_x[k] + (d u_k / d x0)' seed_u[k], grad_yref [batch][N*ny + ny_e] (bnmpc_set_yref_all layout)
 * the same with respect to the cost reference (0 for the x-part of stage 0: x_0 is fixed by x0); either output may be NULL.
 * This is bnmpc_eval_adjoint_sens_p with grad_p = NULL. */
int bnmpc_eval_adjoint_sens(void* handle, const double* seed_x, const double* seed_u, double* grad_x0, double* grad_yref, int on_device);
/* d x_k / d p and d u_k / d p at the stored solution, p = (mass, g) of the controller model (BNMPC_F_P, np = 2), stages
 * 0 .. stages-1 (1 <= stages <= N+1, else BNMPC_E_ARG): sens_x [batch][stages][nx][np], sens_u [batch][min(stages, N)][nu][np];
 * either may be NULL.  sens_x[0] = 0 (x_0 is fixed by x0).  With the same KKT matrix and c_k = phi_k(x_k, u_k; p) - x_{k+1}:
 * d(z, pi) / d p_j = -K^{-1} [dR_j; dc_j], dc_j = d phi_k / d p_j, dR_j = (d B_k / d p_j)' pi_k (u-part),
 * (d A_k / d p_j)' pi_k (x-part, stages >= 1), where phi_k, A_k, B_k are the configured integrator (erk_stages) and its
 * sensitivities, differentiated exactly.  One factorisation and np solves per instance. */
int bnmpc_eval_sens_p(void* handle, int stages, double* sens_x, double* sens_u, int on_device);
/* bnmpc_eval_adjoint_sens plus grad_p [batch][np] = sum_k (d x_k / d p)' seed_x[k] + (d u_k / d p)' seed_u[k], all from one
 * solve with the KKT matrix; any output may be NULL.  With grad_p = NULL this is bnmpc_eval_adjoint_sens, bit for bit; with
 * grad_p, grad_x0 and grad_yref agree with it to rounding (the evaluation of grad_p is a separate kernel instantiation). */
int bnmpc_eval_adjoint_sens_p(void* handle, const double* seed_x, const double* seed_u, double* grad_x0, double* grad_yref,
                              double* grad_p, int on_device);
/* ocp_solver.get_stats / status: int32 [batch] */
int bnmpc_get_stats(void* handle, int which, int32_t* out, int on_device);

/* AcadosSimSolver set('x')/set('u')/solve()/get('x') of the plant (src/force_model/ocp.py:106-112), `substeps` times
 * in a row as OCP.simulate_next_x of the jerk path does (src/jerk_model/ocp.py:106-113): each sub-step is one ERK step
 * (sim_erk_stages stages) of length sim_dt with its own input.
 * x AoS [batch][4], u AoS [batch][substeps][2] = (theta, Fd) per sub-step, p_plant AoS [batch][2] or NULL (nominal),
 * eps [batch] or NULL added to all states of an instance at the end (the np.random.normal draw, :114-115).
 * on_device as for bnmpc_solve_for_x0: 0 host buffers (returns with x_next in host memory), 1 device buffers (asynchronous),
 * BNMPC_HOST_ASYNC pinned host buffers, copies and kernel enqueued, the caller synchronises. */
int bnmpc_sim_step(void* handle, int substeps, const double* x, const double* u, const double* p_plant, const double* eps,
                   double* x_next, int on_device);

/* Fused closed loop = follow_trajectory (src/force_model/controller.py:8-56, src/jerk_model/controller.py:8-58) for
 * all instances, device-resident between steps.  All pointers are DEVICE pointers, batch-minor layout. */
typedef struct bnmpc_closed_loop_args {
    int32_t n_steps;        /* control steps to run in this call */
    int32_t first_step;     /* index of the first step (row offset into ref, noise and the logs) */
    int32_t ref_rows;       /* rows of ref; needs first_step + n_steps + N <= ref_rows */
    int32_t ref_shared;     /* layout of ref: 1 = one [rows][8] table shared by all instances, 0 = [rows][8][batch]
                               (batch-minor), 2 = [batch][rows][8] (instance-major: a warp reads its window as one
                               contiguous 2 KB segment - the layout to prefer for per-instance tables), 3 = no table:
                               ref is [batch][4] = (radius, centre_x, centre_z, phase) of gen_circle_traj and every row
                               is computed on the fly with n = ref_rows - horizon samples per revolution (T = 10 s) */
    int32_t log_stride;     /* number of steps the log arrays were allocated for (>= first_step + n_steps) */
    int32_t steps_per_launch; /* <= 1: one kernel launch per control step (the latency path: step i is complete when launch i
                               is).  k > 1: up to k control steps of every instance per launch - an instance keeps its working
                               set on chip for a chunk of consecutive steps and instances advance independently of each
                               other inside the launch (the Monte-Carlo throughput path; results are identical) */
    const double* ref;      /* gen_circle_traj layout, 8 columns [px pz vx vz ax az+g 0 0] (src/generate_trajectory.py:7-28) */
    const double* noise;    /* [log_stride][batch] or NULL: eps of step s for instance i (src/force_model/ocp.py:114) */
    /* optional logs (NULL to skip), [log_stride(+1)][dim][batch] */
    double* Xsim;           /* [log_stride+1][4][batch]; row first_step must hold the current state on entry if non-NULL */
    double* U_plant;        /* [log_stride][2][batch]  (theta, Fd) of the last sub-step (controller.py:44 / jerk :46) */
    double* U_ctrl;         /* [log_stride][2][batch]  u0 of the OCP */
    double* a_log;          /* [log_stride][2][batch]  force: u0/m (controller.py:38), jerk: a_i (jerk controller.py:45) */
    int32_t* status;        /* [log_stride][batch] */
    int32_t* qp_iter;       /* [log_stride][batch] */
    /* Plant noise drawn on the device instead of read from `noise` (which must then be NULL): eps of (instance i, step s) =
     * noise_std * N(0,1) from Philox4x32-10 with key = noise_seed and counter = (first_instance + i, s), Box-Muller on the
     * first two 53-bit uniforms - one scalar per instance and step like np.random.normal(0, noise) at
     * src/force_model/ocp.py:114-115, independent of batch size, sharding and launch shape (bnmpc_philox_noise gives the
     * same numbers as an array). */
    int32_t noise_philox;   /* 0 = off */
    int32_t reserved;
    uint64_t noise_seed;
    double noise_std;       /* params.py:122 noise = 0.01 */
    int64_t first_instance; /* global id of instance 0 of this handle (its rank's offset into the sharded batch) */
} bnmpc_closed_loop_args;

/* start of follow_trajectory: Xsim[0] = x0, a_i = [0, g], closedLoopCost = 0, zero iterate.
 * x0 [4][batch]; p_ctrl, p_plant [2][batch] (NULL = nominal mass 0.03277, g 9.81).  Device pointers. */
int bnmpc_closed_loop_init(void* handle, const double* x0, const double* p_ctrl, const double* p_plant);
int bnmpc_closed_loop_run(void* handle, const bnmpc_closed_loop_args* args);
/* gen_circle_traj (src/generate_trajectory.py:7-28) for every instance from (radius, centre_x, centre_z, phase)
 * [batch][4] with the device arithmetic of ref_shared = 3: table [batch][rows][8] (instance-major), rows = n + horizon.
 * Device pointers. */
int bnmpc_gen_circle_table(void* handle, const double* params, int rows, double* table);
/* results so far: cost [batch] (closedLoopCost), abs_err [batch] (sum over steps of |pref-psim| over both position
 * coordinates = calc_aed numerator, src/store_results.py:233-236), x [4][batch] current plant state, acc [2][batch]
 * (jerk a_i).  Any pointer may be NULL.  Device pointers. */
int bnmpc_closed_loop_state(void* handle, double* cost, double* abs_err, double* x, double* acc);
/* int32 [batch]: control steps since bnmpc_closed_loop_init whose solve returned a non-zero status.  The reference raises
 * on the first one (src/force_model/controller.py:33-36); the fused loop keeps stepping - it applies u0 of the iterate the
 * solver left, logs the status of the step - and counts, so that a run without per-step logs still reports failures. */
int bnmpc_closed_loop_failures(void* handle, int32_t* out, int on_device);
/* The draws of noise_philox as an array: out [n_steps][batch] (device pointer) = noise_std * N(0,1) of instances
 * first_instance .. first_instance + batch - 1 at steps first_step .. first_step + n_steps - 1. */
int bnmpc_philox_noise(void* handle, uint64_t seed, double noise_std, int64_t first_instance, int first_step, int n_steps, double* out);

/* Measured FMA throughput of `device` in TFLOP/s for BNMPC_FP64 / BNMPC_FP32 (saturating kernel, 8 independent chains
 * per thread, best of 5): the denominator of the roofline fraction bench.py reports (MEASURED_PEAKS.json has no
 * vector-pipe figure). */
int bnmpc_measure_fma_peak(int device, int precision, double* tflops);

/* Device self-test of the reciprocal the solver passes use (bnmpc_core.cuh: rcp_vec, six operands with one range guard):
 * evaluates it on `count` x 6 pseudo-random operands - solver_range != 0: positive, 1e-14 .. 1e6 (what slacks look like);
 * 0: all bit patterns, including zeros, subnormals, infinities and NaNs - and counts the results whose bits differ from
 * the IEEE division 1.0 / t (NaN == NaN).  The solver's parity claim needs *mismatches == 0.  No reference counterpart:
 * acados divides on the CPU. */
int bnmpc_selftest_rcp(int device, int64_t count, int solver_range, int64_t* mismatches);

/* Debug aid (no reference counterpart): while buf != NULL, CTA 0 of every lockstep launch (steps_per_launch > 1) records
 * (clock64, tag << 56 | masks) pairs at the barriers of its schedule into the device buffer buf[1..cap), buf[0] = words used. */
int bnmpc_debug_profile(void* handle, long long* buf, int cap);
/* number of kernels this library has launched on the handle since creation */
int64_t bnmpc_launch_count(void* handle);
const char* bnmpc_last_error(void);
int bnmpc_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BNMPC_H */
