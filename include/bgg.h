/* bilevel-gait-gen_b200 -- C ABI of the B200-native RTI-MPC hot path.
 *
 * Plain pointers and sizes only; every pointer is HOST memory unless the name says device.  All arithmetic is FP64.
 * The reference has no FFI seam -- its hot path is a set of C++ classes linked statically into the callers
 * (SURVEY.md section 8b) -- so each entry point names the reference member function(s) it stands in for, for a
 * whole batch of independent MPC instances at once.  The C++ shim in bilevel-gait-gen_b200/host/ (mpc::MPC /
 * mpc::MPCSingleRigidBody with the reference's own signatures) and the ctypes binding used by the tests both sit on
 * top of exactly these functions.
 *
 * Return value: 0 on success, a negative BGG_E* code otherwise (never throws across the boundary);
 * bgg_last_error() gives the message of the last failure on the calling thread.
 */
#ifndef BGG_H_
#define BGG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BGG_OK 0
#define BGG_EINVAL (-1)
#define BGG_ECUDA (-2)
#define BGG_ENOMEM (-3)
#define BGG_ESTATE (-4)

#define BGG_NX 12        /* tangent states, mpc/models/single_rigid_body_model.cpp:30 */
#define BGG_NX_MAN 13    /* manifold states [p(3) l(3) quat xyzw(4) a(3)], single_rigid_body_model.h:87-92 */
#define BGG_NUM_EE 4

/* mpc::SolveQuality, mpc/include/qp/qp_interface.h:12-22 */
enum bgg_status {
    BGG_SOLVED = 0, BGG_SOLVED_INACC = 1, BGG_MAX_ITER = 2, BGG_PRIMAL_INFEASIBLE = 3, BGG_DUAL_INFEASIBLE = 4,
    BGG_PRIMAL_INFEASIBLE_INACC = 5, BGG_DUAL_INFEASIBLE_INACC = 6, BGG_UNSOLVED = 7, BGG_OTHER = 8
};

/* mpc::MPCInfo (mpc/include/mpc.h:39-62): the fields that act on the live path, plus solver settings
 * (ClarabelInterface ctor, mpc/qp/clarabel_interface.cpp:18-27). */
typedef struct bgg_config {
    int32_t num_nodes;        /* N, 4 < N <= 64 */
    int32_t max_spline_vars;  /* cap on force+position spline variables per instance: a multiple of 8, >= num_nodes + 1 and
                                 <= 160 (0 = default 160).  bgg_create refuses larger values: the condensing and KKT kernels
                                 keep per-block tables sized for 160.  The shipped configurations need at most 148. */
    int32_t device;           /* CUDA device ordinal */
    int32_t ipm_max_iter;     /* 0 = default 50 */
    int32_t ipm_refine;       /* iterative refinement of the late solves against the regularised matrix: 0 / positive = one step (default), negative = none */
    int32_t ipm_refine_after; /* refine the solves only once the complementarity gap mu has fallen below 10^-k of its first value, k = this field
                                 (0: library default 12, i.e. only solves run to tighter than default tolerances; negative: refine from the first
                                 iteration).  Independently of k, an instance still iterating at iteration 20 is refined from there on. */
    double integrator_dt;
    double friction_coef;
    double force_bound;
    double swing_height;
    double foot_offset;
    double ee_box_size[2];
    double force_cost;
    double ipm_tol_feas;      /* 0 = default 1e-8 */
    double ipm_tol_gap;       /* 0 = default 1e-8 */
    double ipm_eq_delta;      /* 0 = default 1e-10 (static regularisation of the equality rows) */
    double ipm_reg_eps;       /* 0 = default 1e-10 (static regularisation of the eliminated cone block and of H) */
    double ipm_tol_infeas;    /* 0 = default 1e-8 (primal infeasibility certificate, Clarabel tol_infeas_abs / _rel) */
} bgg_config;

/* What the reference reads out of pinocchio at construction: mpc/models/model.cpp:27 (mass),
 * mpc/models/single_rigid_body_model.cpp:33-37 (Ir_, Ir_inv_), :258-308 (GetCOMToHip offsets). Row-major 3x3. */
typedef struct bgg_robot {
    double mass;
    double Ir[9];
    double Ir_inv[9];
    double hip_xy[BGG_NUM_EE * 2];
    double gravity[3];
} bgg_robot;

/* Leg chains for the inverse kinematics (what mpc/models/single_rigid_body_model.cpp:314-455 reaches through pinocchio's
 * forwardKinematics / computeFrameJacobian): hip, thigh, calf revolute joint and the foot frame of each leg, every placement
 * given in the frame of the movable joint before it (the hip in the floating base), rotations row-major, axes in the joint frame.
 * Leg order FL, FR, RL, RR = pinocchio's joint order for a1.urdf: q = [p, quat xyzw, 4 x (hip, thigh, calf)]. */
typedef struct bgg_leg_chain {
    double t[4][3];
    double R[4][9];
    double axis[3][3];
} bgg_leg_chain;
typedef struct bgg_kinematics {
    bgg_leg_chain leg[BGG_NUM_EE];
} bgg_kinematics;
#define BGG_NQ 19
#define BGG_NV 18

typedef struct bgg_handle bgg_handle;

const char* bgg_last_error(void);
int bgg_device_count(void);

/* Measured FP64 FMA throughput of `device` (register-resident FMA chains, best of 5): the ceiling bench.py reports
 * the solver kernels against.  No reference counterpart. */
int bgg_measure_fp64_peak(int device, double* tflops);

/* MPCSingleRigidBody::MPCSingleRigidBody (mpc/mpc_single_rigid_body.cpp:8-23) + MPC::MPC (mpc/mpc.cpp:38-76). */
int bgg_create(const bgg_config* cfg, const bgg_robot* robot, bgg_handle** out);
void bgg_destroy(bgg_handle* h);

/* MPC::AddQuadraticTrackingCost (mpc.cpp:533-540), SetQuadraticFinalCost / SetLinearFinalCost (:143-157).
 * Q and Phi are the diagonals (every shipped configuration is diagonal); x_des is a tangent state. */
int bgg_set_costs(bgg_handle* h, const double Q_diag[BGG_NX], const double x_des[BGG_NX], const double Phi_diag[BGG_NX],
                  const double Phi_w[BGG_NX]);

/* Create `batch` instances, each the trajectory the reference constructs by default: Trajectory ctor
 * (mpc/trajectory.cpp:11-48) over CreateDefaultSwitchingTimes (mpc.cpp:566-588) = {0,.3,.6,.9,1.2}, feet 1 and 2
 * starting in stance.  contact_times (optional, [4][num_contacts]) replaces the default switching times. */
int bgg_batch_reset(bgg_handle* h, int batch, const double* contact_times, int num_contacts);

/* MPC::SetStateTrajectoryWarmStart (mpc.cpp:660-666).  per_node != 0: states is [batch][N+1][13];
 * per_node == 0: states is [batch][13] and is replicated over the nodes (what every driver does, test/mpc_test.cpp:91). */
int bgg_set_warm_states(bgg_handle* h, const double* states, int per_node);

/* MPC::UpdateContactTimes (mpc.cpp:1085-1088) for instances [first, first+count): times is [count][4][num_contacts]. */
int bgg_set_contact_times(bgg_handle* h, int first, int count, const double* times, int num_contacts);

/* One RTI solve for every instance: MPC::GetRealTimeUpdate -> MPCSingleRigidBody::Solve
 * (mpc.cpp:92-108, mpc_single_rigid_body.cpp:25-216).  state [batch][13], t0 [batch], ee_start [batch][4][3].
 * Output arrays may be NULL.  status/iters are int32 [batch]; alpha/cost are double [batch]; z [batch][z_stride] receives what
 * the caller of the reference reads back, the decision vector after the line-search update (MPC::GetQPSolution, mpc.cpp:
 * 1071-1073: [x_0 .. x_N (12 each, tangent) | force spline variables | position spline variables], n <= z_stride entries
 * per instance, the rest of a row untouched; BGG_EINVAL if an instance has more than z_stride variables). */
int bgg_solve_batch(bgg_handle* h, const double* state, const double* t0, const double* ee_start, int32_t* status,
                    int32_t* iters, double* alpha, double* cost, double* z, int z_stride);

/* The solver seam on its own: QPInterface::SetupQP + Solve (mpc/include/qp/qp_interface.h:30-65) as ClarabelInterface implements
 * them (mpc/qp/clarabel_interface.cpp:29-155), for `count` independent QPs that share one sparsity pattern:
 *     min 1/2 x'Px + q'x   s.t.  A x + s = b ,  s = 0 on the rows with is_eq != 0 (Zero cone), s >= 0 on the others (Nonnegative cone).
 * P [n x n] and A [m x n] in compressed-sparse-column form as Eigen::SparseMatrix holds them (P: a triangle or the full symmetric
 * matrix); P_val [count][nnz(P)], A_val [count][nnz(A)], q [count][n], b [count][m].  Outputs x [count][n], y / s [count][m]
 * (multipliers and slacks in the caller's row order), status (mpc::SolveQuality) and iteration counts; y, s, status, iters may be
 * NULL.  Same interior-point iteration and tolerances as bgg_solve_batch, on dense data: n <= 128 (the reference's 3-variable
 * cross-solver QP, test/mpc_test.cpp:857-1005; the 42-variable whole-body QP of controllers/qp_control.cpp).  The MPC QP itself
 * goes through bgg_solve_batch, whose kernel exploits its structure. */
int bgg_qp_solve_batch(bgg_handle* h, int count, int n, int m, const int32_t* P_colptr, const int32_t* P_rowidx, const double* P_val,
                       const int32_t* A_colptr, const int32_t* A_rowidx, const double* A_val, const double* q, const double* b,
                       const uint8_t* is_eq, double* x, double* y, double* s, int32_t* status, int32_t* iters);

/* Derivative of the seam's QPs at a primal-dual point: ClarabelInterface::SetupDerivativeCalcs (mpc/qp/clarabel_interface.cpp:262-602)
 * and the vectors CalcDerivativeWrtVecs / CalcDerivativeWrtMats form from it (:182-260), for `count` QPs on one pattern (the same
 * conventions as bgg_qp_solve_batch).  With G the inequality rows of A, Ae the equality rows, lam = y on G's rows, nu = y on Ae's:
 *     [ P    G'D(lam)   Ae' ] [dz  ]      [dx]
 *     [ G    D(s)       0   ] [dlam]  = - [0 ]        (the reference's own +D(s) block)
 *     [ Ae   0          0   ] [dnu ]      [0 ]
 * x [count][n], y / s [count][m]: the point, in the caller's row order (normally what bgg_qp_solve_batch returned); dx [count][n]: the
 * gradient of the loss in x (the reference passes P x + q, ClarabelInterface::Computedx :604-612).  Outputs, each may be NULL:
 * dz [count][n] (= dq); dy [count][m] (dlam on inequality rows, dnu on equality rows); db [count][m] (-dnu on equality rows,
 * dh = -lam o dlam on inequality rows); dA [count][nnz(A)] on A's pattern (dnu_r x_j + nu_r dz_j on an equality row r,
 * lam_r dlam_r x_j + lam_r dz_j on an inequality row); status [count]: 0 ok, 1 a zero or non-finite pivot or a non-finite result,
 * 2 s <= 0 on a kept inequality row or a non-finite input.  A QP of status 1 or 2 gets zero outputs.  Inequality rows without a stored
 * entry are left out as in the solve (dlam = 0, dh = 0).  Limits: n <= 128 and n + (equality rows) <= 160, else BGG_EINVAL. */
int bgg_qp_adjoint_batch(bgg_handle* h, int count, int n, int m, const int32_t* P_colptr, const int32_t* P_rowidx, const double* P_val,
                         const int32_t* A_colptr, const int32_t* A_rowidx, const double* A_val, const uint8_t* is_eq, const double* x,
                         const double* y, const double* s, const double* dx, double* dz, double* dy, double* db, double* dA, int32_t* status);

/* The same solve split for measurement: copy inputs to HBM once, run the kernels on resident data, fetch results.
 * bgg_solve_resident returns with the solve enqueued on the handle's stream; it waits only for the step's first small kernel
 * (the per-instance set-up, whose sizes decide the shared-memory layout of the rest), not for the solve. */
int bgg_upload_inputs(bgg_handle* h, const double* state, const double* t0, const double* ee_start);
int bgg_solve_resident(bgg_handle* h);
/* z (optional): [batch][z_stride] decision vectors; a page-locked buffer whose z_stride is the full row length 12 (N + 1) + max_spline_vars
 * receives the device copy directly, any other buffer goes through the handle's pinned staging area */
int bgg_download_results(bgg_handle* h, int32_t* status, int32_t* iters, double* alpha, double* cost, double* z, int z_stride);
int bgg_synchronize(bgg_handle* h);
/* Closed-loop sweeps on resident data: replace every instance's inputs by the model's own next step -- state = node 1 of
 * the solved trajectory (the plant of apps/mpc_demo.cpp:185 and test/gait_opt_playground.cpp:128), t0 += dt, measured
 * feet = the trajectory's feet at the new time.  Follow with bgg_solve_resident. */
int bgg_advance_plant(bgg_handle* h, double dt);

/* MPCSingleRigidBody::ComputeParamPartialsClarabel (mpc/mpc_single_rigid_body.cpp:642-792) for instance b, foot `ee`, contact time
 * `contact_idx`: the partials of the QP's constraint matrices and equality right-hand side with respect to that contact time, as
 * triplets in the reference's numbering -- dA (num_eq x n: dynamics | touch-down | foot start), dG (num_ineq x n: force box |
 * friction pyramid | foot box), db [num_eq]; exact zeros are not listed (utils/sparse_matrix_builder.cpp:25).  The gait-gradient
 * path (bgg_gait_gradient_batch) never forms these; this is the export for callers that want the matrices (test/mpc_test.cpp:140-236).
 * counts = [nnz dA, nnz dG, num_eq, num_ineq]; db must hold 12 (N + 1) + 16 entries (num_eq never exceeds that).  Returns BGG_OK; 1 when the instance's last solve is not Solved (the reference
 * returns false); a negative code otherwise (cap too small: counts holds the sizes needed). */
int bgg_param_partials(bgg_handle* h, int b, int ee, int contact_idx, int cap, int32_t* counts, int32_t* Ar, int32_t* Ac, double* Av, int32_t* Gr,
                       int32_t* Gc, double* Gv, double* db);

/* ---- joint-space targets (SURVEY 8f row 2) */
int bgg_set_kinematics(bgg_handle* h, const bgg_kinematics* kin);
/* SingleRigidBodyModel::InverseKinematics (single_rigid_body_model.cpp:314-425) for `count` independent problems: state [count][13]
 * (manifold SRB state), ee_des [count][4][3], joint_guess [count][12] (the tail of state_guess) -> q [count][19].
 * status: 0, or 1 where the reference throws "IK did not converge."; iters [count][4] (may be NULL): iterations per foot. */
int bgg_ik_batch(bgg_handle* h, int count, const double* state, const double* ee_des, const double* joint_guess, double* q, int32_t* status,
                 int32_t* iters);
/* MPCController::GetTargetsFromTraj (controllers/mpc_controller.cpp:414-511) for every instance, on the trajectories resident on
 * the device: time [batch]; q_des [batch][19] is q_des_ (in: the running IK guess, out: the configuration target); v_des [batch][18];
 * force_des [batch][4][3].  status: 0; 1 "IK did not converge."; 2 "bad interp."; 3 time beyond the trajectory. */
int bgg_targets_from_traj_batch(bgg_handle* h, const double* time, double* q_des, double* v_des, double* force_des, int32_t* status);
/* device milliseconds of the four kernels of the last bgg_solve_resident (prepare, condense, ipm, finish),
 * measured with CUDA events on the handle's stream; enable with bgg_set_profiling(h, 1). */
int bgg_set_profiling(bgg_handle* h, int enable);
int bgg_last_kernel_ms(bgg_handle* h, float ms[4]);
int bgg_kernel_launch_count(bgg_handle* h, int64_t* launches);
/* CUDA events on the handle's stream for whole-step timing: record event `slot` (0..7); elapsed ms between two slots
 * (synchronises on the later one). */
int bgg_event_record(bgg_handle* h, int slot);
int bgg_event_elapsed_ms(bgg_handle* h, int slot_start, int slot_end, float* ms);

/* --- parity taps and accessors (all sizes are per instance) ------------------------------------------------------ */
typedef struct bgg_sizes {
    int32_t n, nu, nf, np, n_samples, n_eebox, n_eq, n_td, m_ineq, status, iters, ls_iters, error;
    int32_t nfv[BGG_NUM_EE], npv[BGG_NUM_EE], fbase[BGG_NUM_EE], pbase[BGG_NUM_EE];
    double t0, alpha, cost, prim_res, dual_res, gap, eq_violation, step_norm, merit, merit_dd;
    double ee_box[2]; /* foot-box size the last QP was built with (the adapted size lives in the instance) */
    double qp_cost; /* objective of the QP optimum, 1/2 z'Pz + q'z */
    int32_t refined_iters; /* interior-point iterations of the last solve that ran with iterative refinement */
    int32_t no_iterate;    /* the solver stopped before its first finite residual evaluation (status Other, previous solution kept) */
} bgg_sizes;
int bgg_get_sizes(bgg_handle* h, int instance, bgg_sizes* out);

/* Discretised dynamics of the last solve, dense, as the reference holds them in A_, B_, C_
 * (mpc_single_rigid_body.cpp:236-262): Ad [count][N][12][12], Bd [count][N][12][nu_stride], cd [count][N][12]. */
int bgg_get_dynamics(bgg_handle* h, int first, int count, double* Ad, double* Bd, double* cd, int nu_stride);

/* Condensed QP of the last solve: H [nu][nu], g [nu], phipos [2(N-3)][nu] (position rows of the state map for the
 * foot-box rows, node-major from node 4), xoff [N+1][12] (state offsets).  Any pointer may be NULL. */
int bgg_get_condensed(bgg_handle* h, int instance, double* H, double* g, double* phipos, double* xoff);

/* The QP of the last solve exactly as the reference hands it to its solver (MPC::GetQPData, mpc.h; QPData::
 * ConstructSparseMats / ConstructVectors, mpc/qp/qp_data.cpp:169-289; utils/sparse_matrix_builder.cpp:11-42), for
 * instances [first, first+count): constraint matrix in compressed-sparse-column form with the reference's sparsity
 * (exact zeros dropped, rows ascending inside a column, constraint blocks stacked Dynamics | ForceBox | FrictionCone |
 * EndEffectorLocation | TDPosition | EndEffectorStart), the diagonal of P, q, and the Clarabel-form right-hand side ub.
 * dims [count][6] = {n, m, nnz, equality rows, inequality rows, error}; colptr [count][n_stride+1];
 * rowidx / val [count][nnz_cap]; p_diag / q [count][n_stride]; ub [count][m_stride].  error bit 3 = nnz > nnz_cap
 * (colptr is still valid, rowidx / val are not written). */
int bgg_export_qp_csc(bgg_handle* h, int first, int count, int32_t* dims, int32_t* colptr, int32_t* rowidx, double* val,
                      int nnz_cap, double* p_diag, double* q, double* ub, int n_stride, int m_stride);

/* Solution of the last solve.  qp_sol [n]: the QP optimum z* = [x_0..x_N | u] (MPC::Solve's `sol`);
 * z [n]: prev_qp_sol after the line-search update (MPC::GetQPSolution, mpc.cpp:1071-1073);
 * lam / slack [m_ineq] in the kernel's row order (see csrc/bgg_ipm.cu), nu_eq [n_eq]. */
int bgg_get_solution(bgg_handle* h, int instance, double* qp_sol, double* z, double* lam, double* slack, double* nu_eq);

/* --- gait optimiser: derivative of the cost with respect to the contact times ------------------------------------- */
#define BGG_MAX_CONTACTS 12   /* contact times (LiftOff / TouchDown knots) per foot */

/* MPCController::GaitOpt's derivative chain for every instance, after a solve (controllers/mpc_controller.cpp:518-552):
 * MPC::ComputeDerivativeTerms + GetQPPartials (mpc.cpp:1047-1069; clarabel_interface.cpp:182-260, 262-612),
 * MPCSingleRigidBody::ComputeParamPartialsClarabel for every contact time (mpc_single_rigid_body.cpp:642-792),
 * GaitOptimizer::ModifyQPPartials + ComputeCostFcnDerivWrtContactTimes (gait_optimizer.cpp:92-179, 536-539).
 * dHdtheta [batch][4][BGG_MAX_CONTACTS] (foot-major, unused entries 0); n_contacts [batch][4];
 * status [batch]: 0 ok, 1 the last solve was not `Solved` (the reference's calls return false), 2 singular system. */
int bgg_gait_gradient_batch(bgg_handle* h, int32_t* status, int32_t* n_contacts, double* dHdtheta);

/* GaitOptimizer::OptimizeContactTimes (mpc/gait_optimizer.cpp:185-364; constraint builders :410-534) for every
 * instance: the LP  min dH/dtheta . s  over the step of all contact times (polytope / start / trust-region / next-node
 * rows; BFGS is disabled in the reference).  time [batch] is the current time, trust the infinity-norm trust region
 * (the reference's Delta_ = 1), alpha scales the step (`step_ = alpha * step_`).  dHdtheta [batch][4][BGG_MAX_CONTACTS]
 * or NULL to use each instance's last bgg_gait_gradient_batch result.  Outputs, each [batch][4][BGG_MAX_CONTACTS]:
 * step, xk (the contact times the step applies to) and new_times = ConvertQPVecToContactTimes(xk + step);
 * status [batch][4]: 0 converged, 2 iteration limit.  The instances are not modified. */
int bgg_optimize_contact_times_batch(bgg_handle* h, const double* time, double trust, double alpha, const double* dHdtheta,
                                     double* step, double* xk, double* new_times, int32_t* status);

/* GaitOptimizer::LineSearch (mpc/gait_optimizer.cpp:671-753) for every instance: K copies, copy i with the contact times
 * ConvertQPVecToContactTimes(xk + (i / K) step) (GetContactTimes(alpha), :645-669), one RTI solve each from
 * (state, t0, ee_start) -- all batch x K solves run as one batch on the device -- then the arg-min of
 * cost / num_decision_vars over the copies that are not primal infeasible and SetWarmStartTrajectory(best).
 * The reference's LS_SIZE is 10.  best [batch] (-1: every copy infeasible, copy 0 is kept), costs / quality [batch][K]. */
int bgg_line_search_batch(bgg_handle* h, int K, const double* xk, const double* step, const double* state, const double* t0,
                          const double* ee_start, int32_t* best, double* costs, int32_t* quality);

/* One tick of controller::MPCController's MPC thread for the whole batch (controllers/mpc_controller.cpp:286-399, MPCUpdate, and
 * :518-573, GaitOpt), ONE call: everything the tick needs is enqueued on the handle's stream -- no intermediate wait for the
 * device, no allocation after the first tick -- and the call returns after a single read-back.  mode selects the branch the
 * reference takes for its robot (:323-345):
 *   BGG_TICK_SOLVE           GetRealTimeUpdate
 *   BGG_TICK_SOLVE_GAIT_OPT  GetRealTimeUpdate, then GaitOpt: ComputeDerivativeTerms, the QP and contact-time partials,
 *                            dH/dtheta, OptimizeContactTimes; the step stays on the device for the next line-search tick
 *   BGG_TICK_LINE_SEARCH     GaitOptimizer::LineSearch over K copies along that step, SetWarmStartTrajectory(best); instances
 *                            whose derivative was not ready (last solve not Solved) search along a zero step
 * Outputs (any may be NULL): status / iters / alpha / cost / z as bgg_solve_batch (of the parents; unchanged by a line-search
 * tick), deriv_ready [batch] (the reference's deriv_ready_ after this tick), dHdtheta [batch][4][BGG_MAX_CONTACTS] (GAIT_OPT
 * ticks), ls_best [batch] (LINE_SEARCH ticks: arg-min copy, -1 when every copy was infeasible; otherwise -1), ls_costs /
 * ls_quality [batch][K] (LINE_SEARCH ticks: cost / num_decision_vars and solve quality of every copy). */
#define BGG_TICK_SOLVE 0
#define BGG_TICK_SOLVE_GAIT_OPT 1
#define BGG_TICK_LINE_SEARCH 2
int bgg_controller_tick_batch(bgg_handle* h, int mode, int K, const double* state, const double* t0, const double* ee_start, int32_t* status,
                              int32_t* iters, double* alpha, double* cost, double* z, int z_stride, int32_t* deriv_ready, double* dHdtheta,
                              int32_t* ls_best, double* ls_costs, int32_t* ls_quality);
/* The contact-time step of the last GAIT_OPT tick (GaitOptimizer::OptimizeContactTimes: step, the times it applies to and the
 * times after a full step), each [batch][4][BGG_MAX_CONTACTS]; any pointer may be NULL. */
int bgg_controller_get_step(bgg_handle* h, double* step, double* xk, double* new_times);

/* Adjoint of the last bgg_gait_gradient_batch for one instance (parity tap): dz [n], dlam [m_ineq] (kernel row order),
 * dnu_dyn / nu_dyn [12 (N+1)] (differential and value of the dynamics-row multipliers), dnu_eq [n_eq]. */
int bgg_get_adjoint(bgg_handle* h, int instance, double* dz, double* dlam, double* dnu_dyn, double* dnu_eq, double* nu_dyn);

/* Trajectory::GetContactTimes (mpc/trajectory.cpp:339-346) of instances [first, first+count):
 * times / types [count][4][BGG_MAX_CONTACTS] (type 0 LiftOff, 1 TouchDown), counts [count][4]. */
int bgg_get_contact_times(bgg_handle* h, int first, int count, double* times, int32_t* types, int32_t* counts);

/* Parity tap: overwrite the stored solution of the last solve of one instance (any pointer may be NULL) so that the
 * derivative kernels can be checked on exactly the primal / dual point another solver produced.  Layouts as in
 * bgg_get_solution; the status of the instance is set to BGG_SOLVED. */
int bgg_set_solution(bgg_handle* h, int instance, const double* qp_sol, const double* z, const double* lam, const double* slack,
                     const double* nu_eq);

/* Raw trajectory of one instance (the POD bgg::Instance of csrc/bgg_types.cuh). */
size_t bgg_instance_bytes(void);
int bgg_get_instance(bgg_handle* h, int instance, void* out);
int bgg_set_instance(bgg_handle* h, int instance, const void* in);
/* Trajectory::GetState / GetForce / GetEndEffectorLocation (mpc/trajectory.cpp:267-269,395-411) */
int bgg_get_states(bgg_handle* h, int instance, double* states /* [N+1][13] */);
int bgg_eval_splines(bgg_handle* h, int instance, const double* times, int num_times, double* force /* [T][4][3] */,
                     double* position /* [T][4][3] */);

#ifdef __cplusplus
}
#endif
#endif /* BGG_H_ */
