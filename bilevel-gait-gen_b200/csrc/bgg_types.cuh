// bilevel-gait-gen_b200 -- device data model for the batched RTI MPC hot path.
//
// One MPC *instance* = one mpc::MPCSingleRigidBody of the reference (mpc/include/mpc_single_rigid_body.h:11-76)
// reduced to what its Solve() carries from one call to the next: the previous trajectory (states per node and the
// four feet's contact splines, mpc/include/trajectory.h:142-170) plus the adaptive foot-box size
// (mpc_single_rigid_body.cpp:929-937).  Instances are stored as an array of PODs in HBM; a CTA owns one instance
// at a time and stages it through shared memory with contiguous (coalesced) copies.
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define BGG_HD __host__ __device__ __forceinline__
#else
#define BGG_HD inline
#endif

namespace bgg {

constexpr int kNx = 12;              // tangent states (single_rigid_body_model.cpp:30)
constexpr int kNxMan = 13;           // manifold states (:31)
constexpr int kNumEE = 4;            // feet (trajectory.cpp:25-28 hard-codes the A1 pattern)
constexpr int kMaxKnots = 28;        // spline knots per foot (11 at construction; grows by <=3 per added segment)
constexpr int kMaxNodes = 64;        // MPC nodes N (reference cap is 100, trajectory.h:165; configs use 20 and 50)
constexpr int kSamplesPerStance = 10;   // FB_PER_FORCE, mpc.h:320
constexpr int kMaxStances = 4;       // stance segments per foot inside one horizon
constexpr int kEENodeStart = 4;      // EE_NODE_START, mpc_single_rigid_body.h:71
constexpr int kNumForcePolys = 3;    // trajectory.cpp:33-34
constexpr double kForceMult = 100.0; // end_effector_splines.h:152
// Largest max_spline_vars (bgg_config) a handle accepts, and its default.  The register accumulators of k_condense
// (kCondAcc), the KKT tile table (kTileTab) and the dense KKT work list (kMaxKktWork) are sized for it; bgg_create
// refuses more.
constexpr int kMaxSplineVars = 160;

// knot / time types, numerically identical to the reference enums (spline_node.h:14-18, end_effector_splines.h:11-15)
enum : uint8_t { kNoDeriv = 0, kFullDeriv = 1, kEmpty = 2 };
enum : uint8_t { kLiftOff = 0, kTouchDown = 1, kInter = 2 };

// One foot's contact splines (mpc::EndEffectorSplines).  Force knot types are shared by x,y,z; position knot types
// are shared by x,y (`ptype`) and separate for z (`ztype`), exactly the three patterns the reference builds
// (end_effector_splines.cpp:54-100).
struct FootSpline {
    int32_t n;                              // number of knots
    uint8_t ttype[kMaxKnots];               // LiftOff / TouchDown / Inter
    uint8_t ftype[kMaxKnots];               // force knot type
    uint8_t ptype[kMaxKnots];               // x,y position knot type
    uint8_t ztype[kMaxKnots];               // z position knot type
    double t[kMaxKnots];                    // knot times
    double f[3][kMaxKnots][2];              // force (value, stored derivative = derivative / FORCE_MULT)
    double p[3][kMaxKnots][2];              // position (value, derivative)
};

// What one instance carries between solves.
struct Instance {
    double states[kMaxNodes + 1][kNxMan];   // previous trajectory states, manifold form [p, l, quat xyzw, a]
    FootSpline foot[kNumEE];
    double ee_box[2];                       // current foot-box size (IncreaseEEBox / DecreaseEEBox)
    double init_time;
    int32_t run_count;
    int32_t pad_;
};

// Leg chains for the inverse kinematics (bgg_kinematics of include/bgg.h, same layout)
struct LegChain {
    double t[4][3];      // hip / thigh / calf joint and foot frame, each placed in the frame of the joint before it
    double R[4][9];
    double axis[3][3];
};
struct RobotKin {
    LegChain leg[kNumEE];
};

// Handle-wide constants (MPCInfo, mpc.h:39-62, plus what the reference reads out of pinocchio and its cost setters).
struct Params {
    int32_t N;                 // num_nodes
    int32_t max_nu;            // cap on spline decision variables per instance (shared-memory sizing)
    double dt;                 // integrator_dt
    double mass;
    double Ir[9], Ir_inv[9];   // row-major
    double gravity[3];
    double hip_xy[kNumEE][2];  // GetCOMToHip(ee).head<2>() (single_rigid_body_model.cpp:258-308)
    double friction_coef, force_bound, swing_height, foot_offset, force_cost;
    double ee_box_nominal[2];  // ee_bounds_ (mpc_single_rigid_body.cpp:22)
    double Q[kNx];             // diagonal of Q (every shipped config is diagonal)
    double w[kNx];             // -Q x_des
    double Phi[kNx];           // diagonal of the final cost
    double Phi_w[kNx];
    double merit_mu;           // 5000, mpc.cpp:65
    double td_fraction;        // 0.75, mpc.cpp:73
    // interior-point settings (the live reference solver is Clarabel, clarabel_interface.cpp:18-27)
    double ipm_tol_feas, ipm_tol_gap, ipm_eq_delta;
    double ipm_reg_eps;          // static regularisation of the eliminated cone block: W = 1 / (s/z + eps)
    double ipm_tol_infeas;       // infeasibility certificate tolerance (Clarabel tol_infeas_abs / _rel)
    int32_t ipm_max_iter, ipm_refine;
    double ipm_refine_mu_frac;   // iterative refinement starts once mu <= this fraction of the first iteration's mu ...
    int32_t ipm_refine_from_iter;   // ... or at this iteration, whichever comes first (an instance that needs this many is a hard one)
    int32_t pad_refine_;
};

enum SolveStatus : int32_t {    // mpc::SolveQuality, qp_interface.h:12-22
    kSolved = 0, kSolvedInacc = 1, kMaxIter = 2, kPrimalInfeasible = 3, kDualInfeasible = 4,
    kPrimalInfeasibleInacc = 5, kDualInfeasibleInacc = 6, kUnsolved = 7, kOther = 8
};

}  // namespace bgg
