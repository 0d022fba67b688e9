// bilevel-gait-gen_b200 -- C++ host shim: the reference's MPC call surface over the C ABI of include/bgg.h.
//
// Same namespace, class and member names as the reference so that its callers (controllers/mpc_controller.cpp,
// test/mpc_test.cpp, test/simulation_mpc.cpp, apps/mpc_demo.cpp) compile against this header instead of
// mpc/include/{mpc.h, mpc_single_rigid_body.h, trajectory.h, gait_optimizer.h, qp/qp_interface.h, qp/qp_data.h,
// qp/qp_partials.h} (SURVEY.md section 8b lists the members they use).  No CUDA in this header; every method body is
// one or two calls of the C ABI.  One shim object = one handle with batch 1; batch drivers use the ABI directly.
//
// Deliberate differences (INTEGRATION.md section 4): cost matrices are read by their diagonals (every shipped
// configuration is diagonal); on the gait-optimisation path QPPartialsDense / QPPartials are tokens, not 260 x 372 dense
// matrices -- the contraction they feed (GaitOptimizer::ComputeCostFcnDerivWrtContactTimes) runs on the device without forming
// them; QPPartials carries the real sparse dA / dG / db when the caller asks for them (MPC::SetExportParamPartials).
#pragma once
#include <array>
#include <fstream>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#if __has_include(<Eigen/Core>)
#include <Eigen/Core>
namespace mpc {
using vector_t = Eigen::VectorXd;
using matrix_t = Eigen::MatrixXd;
using vector_3t = Eigen::Vector3d;
using vector_2t = Eigen::Vector2d;
}  // namespace mpc
#else
#include "eigen_lite.h"
namespace mpc {
using vector_t = bgg_lite::VectorXd;
using matrix_t = bgg_lite::MatrixXd;
using vector_3t = bgg_lite::VectorNd<3>;
using vector_2t = bgg_lite::VectorNd<2>;
}  // namespace mpc
#endif

#include "../../include/bgg.h"
#include "../csrc/bgg_types.cuh"

namespace controller {
struct Contact {   // controllers/include/controller.h:15-24
    std::vector<bool> in_contact_;
    std::vector<int> contact_frames_;
    Contact() {}
    explicit Contact(int num_contacts) : in_contact_(num_contacts, false), contact_frames_(num_contacts, 0) {}
    int GetNumContacts() const { return static_cast<int>(in_contact_.size()); }
};
}  // namespace controller

namespace mpc {

enum SolveQuality {   // mpc/include/qp/qp_interface.h:12-22
    Solved, SolvedInacc, MaxIter, PrimalInfeasible, DualInfeasible, PrimalInfeasibleInacc, DualInfeasibleInacc, Unsolved, Other
};
enum MPCVerbosityLevel { Nothing = 0, Timing = 1, Optimization = 2, All = 3 };   // mpc.h:32-37
enum Gaits { Trot = 0, Amble = 1, Static_Walk = 2 };
enum TimeType { LiftOff = 0, TouchDown = 1, Inter = 2 };   // spline/end_effector_splines.h:11-15

class SplineTimes {   // spline/end_effector_splines.h:17-30
public:
    SplineTimes() {}
    SplineTimes(double time, TimeType type) : time_(time), type_(type) {}
    double GetTime() const { return time_; }
    TimeType GetType() const { return type_; }
    void SetTime(double time) { time_ = time; }

private:
    double time_ = 0;
    TimeType type_ = LiftOff;
};
using time_v = std::vector<SplineTimes>;

struct MPCInfo {   // mpc.h:39-62
    int num_nodes = 20;
    int num_qp_iterations = 1;
    int num_contacts = 4;
    double friction_coef = 0.5;
    vector_t vel_bounds, joint_bounds_lb, joint_bounds_ub;
    std::vector<std::string> ee_frames;
    int discretization_steps = 1;
    int num_switches = 4;
    double integrator_dt = 0.05;
    double force_bound = 150;
    double swing_height = 0.075;
    double foot_offset = 0.015;
    vector_t nom_state;
    vector_2t ee_box_size;
    int real_time_iters = 6000;
    MPCVerbosityLevel verbose = Nothing;
    double force_cost = 0;
};

// What the reference reads out of pinocchio at construction, computed from the URDF without it (urdf_consts.cpp):
// total mass (models/model.cpp:27), composite inertia about the CoM at the nominal configuration
// (single_rigid_body_model.cpp:33-37), hip offsets incl. the hard-coded shifts (:258-308).
bgg_robot RobotConstsFromURDF(const std::string& urdf_path);   // nominal A1 joint angles (apps/a1_configuration.yaml:init_config)
bgg_robot RobotConstsFromURDF(const std::string& urdf_path, const std::map<std::string, double>& joint_cfg);
bgg_kinematics LegKinematicsFromURDF(const std::string& urdf_path);   // leg chains for the inverse kinematics

// mpc::Trajectory (mpc/include/trajectory.h): a value type.  Here it is the instance POD fetched from the device plus
// the host build of the spline code the kernels use (csrc/bgg_spline.cuh).
class Trajectory {
public:
    Trajectory() {}
    Trajectory(const bgg::Instance& inst, int num_nodes, double node_dt) : inst_(inst), num_nodes_(num_nodes), node_dt_(node_dt) {}
    std::vector<vector_t> GetStates() const;
    vector_t GetState(int node) const;
    void SetState(int idx, const vector_t& state);
    double GetTime(int node) const { return inst_.init_time + node_dt_ * node; }
    int GetNode(double time) const;
    vector_3t GetForce(int end_effector, double time) const;
    vector_3t GetEndEffectorLocation(int end_effector, double time) const;
    std::vector<bool> GetContacts(double time) const;
    controller::Contact GetDesiredContacts(double time) const;
    int GetNumContactNodes(int ee) const;
    std::vector<time_v> GetContactTimes() const;
    void UpdateContactTimes(std::vector<time_v>& contact_times);
    bool IsForceMutable(int ee, double time) const;
    double GetNextContactTime(int ee, double time) const;
    void SetEEInContact(int ee, double time);
    double GetCurrentSwingTime(int ee) const;
    int GetTotalForceSplineVars() const;
    int GetTotalPosSplineVars() const;
    int GetTotalVariables() const { return GetTotalForceSplineVars() + GetTotalPosSplineVars() + 12 * (num_nodes_ + 1); }
    void SetInitTime(double time) { inst_.init_time = time; }
    const bgg::Instance& Raw() const { return inst_; }
    bgg::Instance& Raw() { return inst_; }

private:
    bgg::Instance inst_{};
    int num_nodes_ = 0;
    double node_dt_ = 0;
};

// mpc::QPData (mpc/include/qp/qp_data.h): the fields callers read (test/mpc_test.cpp:125,140-171).
struct SparseCsc {   // stands in for Eigen::SparseMatrix<double> (column-major compressed)
    int rows = 0, cols = 0;
    std::vector<int> outer, inner;
    std::vector<double> values;
    int nonZeros() const { return static_cast<int>(values.size()); }
    double coeff(int r, int c) const;
};
enum Constraints {   // mpc/include/qp/qp_data.h:17-27
    Dynamics, JointForwardKinematics, EndEffectorLocation, ForceBox, JointBox, FrictionCone, TDPosition, Raibert, EndEffectorStart
};
struct QPData {
    SparseCsc sparse_constraint_;
    SparseCsc sparse_cost_;              // P (diagonal on the MPC path); what ClarabelInterface::SetupQP hands to the solver
    std::vector<Constraints> constraints_;   // block order of the rows (single_rigid_body_model.cpp:22-29)
    vector_t cost_diag_, cost_linear, ub_;
    int num_decision_vars = 0, num_dynamics_constraints = 0, num_force_box_constraints_ = 0, num_cone_constraints_ = 0,
        num_ee_location_constraints_ = 0, num_td_pos_constraints_ = 0, num_start_ee_constraints_ = 0, num_raibert_constraints_ = 0;
    int num_equality_ = 0, num_inequality_ = 0;
    int GetTotalNumConstraints() const { return num_equality_ + num_inequality_; }
};

class MPC;
// On the MPC's gait-optimisation path QPPartialsDense is a token (see the header comment) that records which MPC the derivative
// terms belong to; ClarabelInterface::CalcDerivativeWrtVecs / WrtMats fill its matrices and vectors for a QP solved through the seam.
struct QPPartialsDense {
    const MPC* source = nullptr;
    matrix_t dA, dG;
    vector_t dq, db, dh;
    void SetZero() {
        dA.setZero();
        dG.setZero();
        dq.setZero();
        db.setZero();
        dh.setZero();
    }
};
// The solver seam (mpc/include/qp/qp_interface.h:30-65) and its live implementation (mpc/include/qp/clarabel_interface.h:43-106,
// mpc/qp/clarabel_interface.cpp:18-155), over bgg_qp_solve_batch: the interior-point kernel of the CUDA path on the QP it is handed.
class QPInterface {
public:
    explicit QPInterface(int num_decision_vars) : num_decision_vars_(num_decision_vars) {}
    virtual ~QPInterface() {}
    virtual void SetupQP(QPData& data, const vector_t& warm_start) = 0;
    virtual vector_t Solve(const QPData& data) = 0;
    virtual vector_t GetInfinity(int size) const { return vector_t::Constant(size, 1e30); }   // qp_interface.cpp:13-17
    virtual SolveQuality GetSolveQuality() const = 0;
    std::string GetSolveQualityAsString() const;
    virtual vector_t GetDualSolution() const = 0;
    virtual void ConfigureForInitialRun() = 0;
    virtual void ConfigureForRealTime(double run_time_iters) = 0;

protected:
    int num_decision_vars_;
    vector_t prev_qp_sol_;
};

class ClarabelInterface : public QPInterface {
public:
    ClarabelInterface(const QPData& data, bool verbose);
    ClarabelInterface(const ClarabelInterface& other);
    ClarabelInterface& operator=(const ClarabelInterface& other);
    ~ClarabelInterface() override;
    void SetupQP(QPData& data, const vector_t& warm_start) override;   // builds the cone list from data.constraints_ (:29-64)
    vector_t Solve(const QPData& data) override;                         // throws const std::string& "Primal infeasible." (:112-114)
    SolveQuality GetSolveQuality() const override { return solve_quality_; }
    vector_t GetDualSolution() const override { return dual_; }
    vector_t GetSlacks() const { return slacks_; }
    void ConfigureForInitialRun() override {}                            // the reference only moves tol_gap (:166-175); the kernel's are fixed
    void ConfigureForRealTime(double) override {}
    vector_t Computedx(const SparseCsc& P, const vector_t& q, const vector_t& xstar);   // dx = P x* + q (:604-612)
    vector_t Getdx() const { return dx_; }
    void SetVerbosity(bool verbose) { verbose_ = verbose; }
    // The derivative of the last Solve's optimum (:262-602) over bgg_qp_adjoint_batch: the differential system at its primal, dual and
    // slacks with right-hand side dx.  dl / du are OSQP's bound terms; on this path they must be zero, as the reference's call
    // SetupDerivativeCalcs(dx, 0, 0, data) passes them (mpc.cpp:1047-1056).  Throws std::runtime_error if no solution is held or the
    // system is singular; limits n <= 128 and n + (equality rows) <= 160.
    void SetupDerivativeCalcs(const vector_t& dx, double dl, double du, const QPData& data);
    // dq = dz, db = -dnu (equality rows), dh = -lam o dlam (inequality rows) (:182-196)
    void CalcDerivativeWrtVecs(QPPartialsDense& partials) const;
    // dA = dnu x' + nu dz' (equality rows x n), dG = D(lam) dlam x' + lam dz' (inequality rows x n), dense, on the pattern of the
    // constraint matrix and zero elsewhere (:198-260).  Rows as SetupDerivativeCalcs numbers them: the equality rows in order, the
    // inequality rows in order.
    void CalcDerivativeWrtMats(QPPartialsDense& partials) const;

private:
    bgg_handle* h_ = nullptr;
    bool verbose_ = false;
    std::vector<uint8_t> is_eq_;
    SolveQuality solve_quality_ = Unsolved;
    vector_t dual_, primal_, slacks_, dx_;
    bool have_solution_ = false, have_derivative_ = false;
    // set by SetupDerivativeCalcs: the point, dz and dy (dlam / dnu in the caller's row order), the constraint pattern
    vector_t d_x_, d_y_, d_dz_, d_dy_;
    SparseCsc d_pattern_;
    std::vector<uint8_t> d_is_eq_;
};

struct QPPartials {   // mpc/include/qp/qp_partials.h:15-35
    const MPC* source = nullptr;
    int ee = -1, idx = -1;
    // filled by ComputeParamPartialsClarabel when MPC::SetExportParamPartials(true) (bgg_param_partials); empty otherwise
    SparseCsc dA, dG, dP;
    vector_t db, dh, dq, dl, du;
    void SetZero() { dA = dG = dP = SparseCsc(); db = dh = dq = dl = du = vector_t(); }
};

class MPC {
public:
    MPC(const MPCInfo& info, const std::string& robot_urdf);
    MPC(const MPCInfo& info, const bgg_robot& robot);
    MPC(const MPC& other);
    MPC& operator=(const MPC& other);
    virtual ~MPC();

    Trajectory CreateInitialRun(const vector_t& state, const std::vector<vector_3t>& ee_start_locations);   // mpc.cpp:78-90
    Trajectory GetRealTimeUpdate(const vector_t& state, double init_time, const std::vector<vector_3t>& ee_start_locations,
                                 bool high_quality);                                                          // mpc.cpp:92-108
    virtual Trajectory Solve(const vector_t& state, double init_time, const std::vector<vector_3t>& ee_start_locations);
    void SetWarmStartTrajectory(const Trajectory& trajectory);                // mpc.cpp:110-119
    void SetQuadraticFinalCost(const matrix_t& Phi);                          // mpc.cpp:143-150
    void SetLinearFinalCost(const vector_t& w);                               // mpc.cpp:152-157
    void AddQuadraticTrackingCost(const vector_t& state_des, const matrix_t& Q);   // mpc.cpp:533-540
    void AddForceCost(double weight);
    static std::vector<std::vector<double>> CreateDefaultSwitchingTimes(int num_switches, int num_ee, double horizon);   // :566-588
    void SetDefaultGaitTrajectory(Gaits gait, int num_polys, const std::vector<vector_3t>& ee_pos);
    void SetStateTrajectoryWarmStart(const std::vector<vector_t>& states);    // mpc.cpp:660-666
    Trajectory GetTrajectory() const;
    controller::Contact GetDesiredContacts(double time) const { return GetTrajectory().GetDesiredContacts(time); }
    int GetNode(double time) const { return GetTrajectory().GetNode(time); }
    int GetNumDecisionVars() const;
    int GetNumConstraints() const;
    bool ComputeDerivativeTerms();                                            // mpc.cpp:1047-1057
    bool GetQPPartials(QPPartialsDense& partials) const;                      // mpc.cpp:1059-1069
    vector_t GetQPSolution() const;                                           // mpc.cpp:1071-1073
    void UpdateContactTimes(std::vector<time_v>& contact_times);              // mpc.cpp:1085-1088
    const QPData& GetQPData() const;
    void SetVerbosityLevel(MPCVerbosityLevel verbosity) { info_.verbose = verbosity; }
    void AdjustForCurrentContacts(double time, const controller::Contact& contact);   // mpc.cpp:1195-1203
    SolveQuality GetSolveQuality() const { return quality_; }
    // ComputeParamPartialsClarabel writes the sparse matrices into QPPartials as well (one small kernel and a read-back per call);
    // off by default: the gait optimiser's own path does not read them
    void SetExportParamPartials(bool on) { export_partials_ = on; }
    void PrintStats() const;
    void PrintStatLineToFile(std::ofstream& log_file) const;
    double GetAvgCost() const { return solves_ ? cost_sum_ / solves_ : 0.0; }
    double GetCost() const { return cost_; }
    // derivative of the cost with respect to every contact time (foot-major), filled by ComputeDerivativeTerms
    const std::vector<double>& CostDerivWrtContactTimes() const { return dHdtheta_; }
    bgg_handle* Handle() const { return h_; }
    const MPCInfo& Info() const { return info_; }

protected:
    void Create();
    void PushCosts();
    MPCInfo info_;
    bgg_robot robot_{};
    bgg_handle* h_ = nullptr;
    SolveQuality quality_ = Unsolved;
    bool export_partials_ = false;
    double cost_ = 0, cost_sum_ = 0, alpha_ = 0, last_solve_ms_ = 0;
    mutable bool used_log_file_ = false;
    int solves_ = 0, iters_ = 0;
    double Q_[12], xdes_[12], Phi_[12], Phi_w_[12];
    bool have_Q_ = false, have_Phi_ = false, have_Phi_w_ = false;
    mutable QPData data_;
    std::vector<double> dHdtheta_;
    bool deriv_ready_ = false;
};

class MPCSingleRigidBody : public MPC {   // mpc/include/mpc_single_rigid_body.h:11-76
public:
    using MPC::MPC;
    bool ComputeParamPartialsClarabel(const Trajectory& traj, QPPartials& partials, int ee, int idx);   // :642-792
    std::vector<vector_2t> GetEEBoxCenter();                                                             // :1060-1063
    double GetModifiedCost(int num_nodes) const { (void)num_nodes; return cost_; }
};

// mpc::MPCCentroidal (mpc/include/mpc_centroidal.h:15-221).  The reference declares this class and defines none of it
// (mpc/mpc_centroidal.cpp is commented out, SURVEY.md R1), so nothing can be in parity with it; the adapter gives code written
// against that header the live single-rigid-body MPC: feet at the nominal A1 stance where the header's signatures carry none.
class MPCCentroidal {
public:
    MPCCentroidal(const MPCInfo& info, const std::string& robot_urdf) : mpc_(info, robot_urdf) {}
    MPCCentroidal(const MPCInfo& info, const bgg_robot& robot) : mpc_(info, robot) {}
    Trajectory CreateInitialRun(const vector_t& state) { return mpc_.CreateInitialRun(state, ee_); }
    Trajectory GetRealTimeUpdate(double /*run_time_iters*/, const vector_t& state, double init_time) { return mpc_.GetRealTimeUpdate(state, init_time, ee_, false); }
    Trajectory Solve(const vector_t& state, double init_time) { return mpc_.Solve(state, init_time, ee_); }
    void SetWarmStartTrajectory(const Trajectory& trajectory) { mpc_.SetWarmStartTrajectory(trajectory); }
    void SetQuadraticFinalCost(const matrix_t& Phi) { mpc_.SetQuadraticFinalCost(Phi); }
    void SetLinearFinalCost(const vector_t& w) { mpc_.SetLinearFinalCost(w); }
    void AddQuadraticTrackingCost(const vector_t& state_des, const matrix_t& Q) { mpc_.AddQuadraticTrackingCost(state_des, Q); }
    static std::vector<std::vector<double>> CreateDefaultSwitchingTimes(int num_switches, int num_ee, double horizon) {
        return MPC::CreateDefaultSwitchingTimes(num_switches, num_ee, horizon);
    }
    void SetDefaultGaitTrajectory(Gaits gait, int num_polys, const std::array<std::array<double, 3>, 4>& ee_pos) {
        ee_.clear();
        for (const auto& p : ee_pos) ee_.emplace_back(p[0], p[1], p[2]);
        mpc_.SetDefaultGaitTrajectory(gait, num_polys, ee_);
    }
    void SetStateTrajectoryWarmStart(const std::vector<vector_t>& states) { mpc_.SetStateTrajectoryWarmStart(states); }
    void AddForceCost(double weight) { mpc_.AddForceCost(weight); }
    void PrintStats() { mpc_.PrintStats(); }
    controller::Contact GetDesiredContacts(double time) const { return mpc_.GetDesiredContacts(time); }
    Trajectory GetTrajectory() const { return mpc_.GetTrajectory(); }
    vector_t GetForceTarget(double time) const {
        vector_t f(12);
        const Trajectory t = mpc_.GetTrajectory();
        for (int e = 0; e < 4; ++e) { const vector_3t v = t.GetForce(e, time); for (int c = 0; c < 3; ++c) f(3 * e + c) = v(c); }
        return f;
    }
    int GetNode(double time) const { return mpc_.GetNode(time); }
    int GetNumDecisionVars() const { return mpc_.GetNumDecisionVars(); }
    int GetNumConstraints() const { return mpc_.GetNumConstraints(); }
    bool ComputeDerivativeTerms() { return mpc_.ComputeDerivativeTerms(); }
    bool GetQPPartials(QPPartials& partials) const { partials.source = &mpc_; return mpc_.GetSolveQuality() == Solved; }
    bool ComputeParamPartials(const Trajectory& traj, QPPartials& partials, int ee, int idx) { return mpc_.ComputeParamPartialsClarabel(traj, partials, ee, idx); }
    vector_t GetQPSolution() const { return mpc_.GetQPSolution(); }
    MPCSingleRigidBody& Live() { return mpc_; }

private:
    MPCSingleRigidBody mpc_;
    std::vector<vector_3t> ee_ = {vector_3t(0.1526, 0.12523, 0.011089), vector_3t(0.1526, -0.12523, 0.011089),
                                  vector_3t(-0.208321844, 0.1363286, 0.01444), vector_3t(-0.208321844, -0.1363286, 0.01444)};   // test/mpc_test.cpp:97-101
};

class GaitOptimizer {   // mpc/include/gait_optimizer.h:23-171
public:
    static constexpr int LS_SIZE = 10;
    GaitOptimizer(int num_ee, int num_contact_nodes, int num_decision_vars, int num_constraints, double contact_time_ub,
                  double min_time);
    void UpdateSizes(int num_decision_vars, int num_constraints);
    void SetContactTimes(const std::vector<time_v>& contact_times);
    void SetNumContactTimes(int ee, int num_times);
    QPPartialsDense& GetQPPartials() { return qp_partials_; }
    QPPartials& GetParameterPartials(int ee, int idx);
    void ModifyQPPartials(const vector_t& xstar) { (void)xstar; }   // dq += z*: folded into the device contraction
    void ComputeCostFcnDerivWrtContactTimes();                        // gait_optimizer.cpp:92-179
    void OptimizeContactTimes(double time, double actual_red_cost);   // :181-183
    void OptimizeContactTimes(double time, double actual_red_cost, double alpha, bool adapt_trust_region);   // :185-364
    std::vector<time_v>& GetContactTimes() { return contact_times_; }
    std::vector<time_v> GetContactTimes(double alpha) const;          // :645-649
    std::pair<std::vector<time_v>, double> LineSearch(MPCSingleRigidBody& mpc, double time, const std::vector<vector_3t>& ee_locations,
                                                      const vector_t& state);   // :671-753
    double GetStepNorm() const;
    const std::vector<double>& GetGradient() const { return dHdth; }
    const std::vector<double>& GetStep() const { return step_; }

private:
    std::vector<time_v> ConvertQPVecToContactTimes(const std::vector<double>& vec) const;   // :651-669
    int num_ee_;
    std::vector<time_v> contact_times_;
    std::vector<std::vector<QPPartials>> param_partials_;
    QPPartialsDense qp_partials_;
    std::vector<double> dHdth, step_, xk_, xkp1_;
    double Delta_ = 1;
    int run_num_ = 0;
};

}  // namespace mpc
