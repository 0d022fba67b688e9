// bilevel-gait-gen_b200 -- C++ host shim over the C ABI (see mpc_b200.h).  Every member names the reference member it
// stands in for; error behaviour follows the reference: std::runtime_error for misuse (e.g. mpc.cpp:122-124), solver
// outcomes through SolveQuality, derivative calls return false unless the last solve was `Solved` (mpc.cpp:1047-1069).
#include "mpc_b200.h"

#include <cmath>
#include <chrono>
#include <cstring>
#include <ctime>
#include <cstdio>

#include "../csrc/bgg_spline.cuh"

namespace mpc {

namespace {
void Check(int rc) {
    if (rc != BGG_OK) throw std::runtime_error(std::string("bgg: ") + bgg_last_error());
}
void FlattenEE(const std::vector<vector_3t>& ee, double out[12]) {
    if (ee.size() != 4) throw std::runtime_error("four end-effector locations expected");
    for (int e = 0; e < 4; ++e)
        for (int c = 0; c < 3; ++c) out[3 * e + c] = ee[e](c);
}
}  // namespace

// ------------------------------------------------------------------------------------------------------ Trajectory
vector_t Trajectory::GetState(int node) const {
    if (node < 0 || node > num_nodes_) throw std::runtime_error("Trajectory::GetState: node out of range");
    vector_t s(bgg::kNxMan);
    for (int i = 0; i < bgg::kNxMan; ++i) s(i) = inst_.states[node][i];
    return s;
}
std::vector<vector_t> Trajectory::GetStates() const {
    std::vector<vector_t> v;
    for (int k = 0; k <= num_nodes_; ++k) v.push_back(GetState(k));
    return v;
}
void Trajectory::SetState(int idx, const vector_t& state) {
    if (idx < 0 || idx > num_nodes_ || state.size() != bgg::kNxMan) throw std::runtime_error("Trajectory::SetState: bad argument");
    for (int i = 0; i < bgg::kNxMan; ++i) inst_.states[idx][i] = state(i);
}
int Trajectory::GetNode(double time) const { return static_cast<int>(std::ceil((time - inst_.init_time) / node_dt_)); }   // trajectory.cpp:479-481
vector_3t Trajectory::GetForce(int ee, double time) const {
    vector_3t f;
    for (int c = 0; c < 3; ++c) f(c) = bgg::value_at(inst_.foot[ee], true, c, time);
    return f;
}
vector_3t Trajectory::GetEndEffectorLocation(int ee, double time) const {
    vector_3t p;
    for (int c = 0; c < 3; ++c) p(c) = bgg::value_at(inst_.foot[ee], false, c, time);
    return p;
}
std::vector<bool> Trajectory::GetContacts(double time) const {
    std::vector<bool> c(4);
    for (int e = 0; e < 4; ++e) c[e] = bgg::is_in_contact(inst_.foot[e], time);
    return c;
}
controller::Contact Trajectory::GetDesiredContacts(double time) const {
    controller::Contact c(4);
    for (int e = 0; e < 4; ++e) c.in_contact_[e] = bgg::is_in_contact(inst_.foot[e], time);
    return c;
}
int Trajectory::GetNumContactNodes(int ee) const { return bgg::num_contacts(inst_.foot[ee]); }
std::vector<time_v> Trajectory::GetContactTimes() const {
    std::vector<time_v> out(4);
    for (int e = 0; e < 4; ++e) {
        const bgg::FootSpline& s = inst_.foot[e];
        for (int i = 0; i < s.n; ++i)
            if (s.ttype[i] != bgg::kInter) out[e].emplace_back(s.t[i], static_cast<TimeType>(s.ttype[i]));
    }
    return out;
}
void Trajectory::UpdateContactTimes(std::vector<time_v>& contact_times) {
    for (int e = 0; e < 4; ++e) {
        if (static_cast<int>(contact_times.at(e).size()) != GetNumContactNodes(e))
            throw std::runtime_error("UpdateContactTimes: wrong number of contact times");
        double t[bgg::kMaxKnots];
        for (size_t i = 0; i < contact_times[e].size(); ++i) {
            t[i] = contact_times[e][i].GetTime();
            if (t[i] < -1e-3) throw std::runtime_error("Invalid time: negative");   // end_effector_splines.cpp:865-869
        }
        bgg::set_contact_times(inst_.foot[e], t, static_cast<int>(contact_times[e].size()));
    }
}
bool Trajectory::IsForceMutable(int ee, double time) const { return bgg::is_force_mutable(inst_.foot[ee], time); }
double Trajectory::GetNextContactTime(int ee, double time) const { return bgg::next_touchdown_time(inst_.foot[ee], time); }
double Trajectory::GetCurrentSwingTime(int ee) const { return bgg::swing_time(inst_.foot[ee], inst_.init_time); }
void Trajectory::SetEEInContact(int ee, double time) {   // EndEffectorSplines::SetToTouchdown, end_effector_splines.cpp:1042-1060
    bgg::FootSpline& s = inst_.foot[ee];
    const int up = bgg::upper_idx(s, bgg::kPosXY, time);
    if (s.ttype[up] != bgg::kTouchDown) throw std::runtime_error("Attempting to change a lift off to a touchdown node.");
    if (std::abs(s.t[up] - time) > 1e-1) throw std::runtime_error("Attempting to change a touchdown node too far away from the current time.");
    const int up2 = bgg::upper_idx(s, bgg::kPosXY, s.t[up] + 0.001);
    const double time2 = s.t[up2];
    s.t[up] = time;
    for (int i = 1; i < bgg::kNumForcePolys; ++i)
        if (up + i < s.n) s.t[up + i] = i * (time2 - time) / bgg::kNumForcePolys + time;
}
int Trajectory::GetTotalForceSplineVars() const {
    int n = 0;
    for (int e = 0; e < 4; ++e) n += 3 * bgg::num_force_vars(inst_.foot[e]);
    return n;
}
int Trajectory::GetTotalPosSplineVars() const {
    int n = 0;
    for (int e = 0; e < 4; ++e) n += 2 * bgg::num_pos_vars(inst_.foot[e]);
    return n;
}

double SparseCsc::coeff(int r, int c) const {
    for (int k = outer[c]; k < outer[c + 1]; ++k)
        if (inner[k] == r) return values[k];
    return 0.0;
}

// ------------------------------------------------------------------------------------------------------ MPC
MPC::MPC(const MPCInfo& info, const std::string& robot_urdf) : info_(info), robot_(RobotConstsFromURDF(robot_urdf)) { Create(); }
MPC::MPC(const MPCInfo& info, const bgg_robot& robot) : info_(info), robot_(robot) { Create(); }

void MPC::Create() {
    bgg_config cfg{};
    cfg.num_nodes = info_.num_nodes;
    cfg.device = 0;
    cfg.integrator_dt = info_.integrator_dt;
    cfg.friction_coef = info_.friction_coef;
    cfg.force_bound = info_.force_bound;
    cfg.swing_height = info_.swing_height;
    cfg.foot_offset = info_.foot_offset;
    cfg.ee_box_size[0] = info_.ee_box_size(0);
    cfg.ee_box_size[1] = info_.ee_box_size(1);
    cfg.force_cost = info_.force_cost;
    Check(bgg_create(&cfg, &robot_, &h_));
    Check(bgg_batch_reset(h_, 1, nullptr, 0));   // Trajectory over CreateDefaultSwitchingTimes (mpc.cpp:38-76, 566-588)
    for (int i = 0; i < 12; ++i) Q_[i] = xdes_[i] = Phi_[i] = Phi_w_[i] = 0.0;
}

MPC::~MPC() {
    if (h_) bgg_destroy(h_);
}

MPC::MPC(const MPC& other) : info_(other.info_), robot_(other.robot_) {
    Create();
    *this = other;
}

MPC& MPC::operator=(const MPC& other) {   // deep copy incl. the solver state the next solve needs (mpc.cpp:1133-1181)
    if (this == &other) return *this;
    if (info_.num_nodes != other.info_.num_nodes) throw std::runtime_error("MPC::operator=: different horizon lengths");
    info_ = other.info_;
    robot_ = other.robot_;
    std::memcpy(Q_, other.Q_, sizeof Q_);
    std::memcpy(xdes_, other.xdes_, sizeof xdes_);
    std::memcpy(Phi_, other.Phi_, sizeof Phi_);
    std::memcpy(Phi_w_, other.Phi_w_, sizeof Phi_w_);
    have_Q_ = other.have_Q_;
    have_Phi_ = other.have_Phi_;
    have_Phi_w_ = other.have_Phi_w_;
    if (have_Q_) PushCosts();
    bgg::Instance inst;
    Check(bgg_get_instance(other.h_, 0, &inst));
    Check(bgg_set_instance(h_, 0, &inst));
    quality_ = other.quality_;
    cost_ = other.cost_;
    cost_sum_ = other.cost_sum_;
    solves_ = other.solves_;
    dHdtheta_ = other.dHdtheta_;
    deriv_ready_ = false;
    return *this;
}

void MPC::PushCosts() {
    Check(bgg_set_costs(h_, Q_, xdes_, have_Phi_ ? Phi_ : nullptr, have_Phi_w_ ? Phi_w_ : nullptr));
}

void MPC::AddQuadraticTrackingCost(const vector_t& state_des, const matrix_t& Q) {
    if (Q.rows() != 12 || Q.cols() != 12 || state_des.size() != 12)
        throw std::runtime_error("Supplied quadratic cost term is the wrong size.");   // mpc.cpp:122-124
    for (int i = 0; i < 12; ++i) {
        Q_[i] = Q(i, i);
        xdes_[i] = state_des(i);
    }
    have_Q_ = true;
    PushCosts();
}
void MPC::SetQuadraticFinalCost(const matrix_t& Phi) {
    if (Phi.rows() != 12 || Phi.cols() != 12) throw std::runtime_error("Supplied quadratic cost term is the wrong size.");
    for (int i = 0; i < 12; ++i) Phi_[i] = Phi(i, i);
    have_Phi_ = true;
    if (have_Q_) PushCosts();
}
void MPC::SetLinearFinalCost(const vector_t& w) {
    if (w.size() != 12) throw std::runtime_error("Supplied linear cost term is the wrong size.");
    for (int i = 0; i < 12; ++i) Phi_w_[i] = w(i);
    have_Phi_w_ = true;
    if (have_Q_) PushCosts();
}
void MPC::AddForceCost(double weight) {
    // force_cost is fixed at construction in the ABI (bgg_config.force_cost); the reference's drivers pass info.force_cost
    if (weight != info_.force_cost) throw std::runtime_error("AddForceCost: weight differs from MPCInfo::force_cost");
}

std::vector<std::vector<double>> MPC::CreateDefaultSwitchingTimes(int num_switches, int num_ee, double horizon) {
    (void)num_switches;
    (void)horizon;   // the reference ignores both and hard-codes the schedule (mpc.cpp:566-608)
    return std::vector<std::vector<double>>(num_ee, std::vector<double>{0, 0.3, 0.6, 0.9, 1.2});
}
void MPC::SetDefaultGaitTrajectory(Gaits gait, int num_polys, const std::vector<vector_3t>& ee_pos) {
    (void)num_polys;
    (void)ee_pos;
    // everything the reference once did for Trot is commented out (mpc.cpp:626-684); the other gaits throw
    if (gait == Amble) throw std::runtime_error("Amble not implemented yet!");
    if (gait == Static_Walk) throw std::runtime_error("Static Walk not implemented yet!");
    if (gait != Trot) throw std::runtime_error("Unsupported gait.");
}
void MPC::SetStateTrajectoryWarmStart(const std::vector<vector_t>& states) {
    if (static_cast<int>(states.size()) != info_.num_nodes + 1) throw std::runtime_error("warm start has the wrong number of nodes");
    std::vector<double> flat(static_cast<size_t>(info_.num_nodes + 1) * 13);
    for (size_t k = 0; k < states.size(); ++k) {
        if (states[k].size() != 13) throw std::runtime_error("warm start state has the wrong size");
        for (int i = 0; i < 13; ++i) flat[13 * k + i] = states[k](i);
    }
    Check(bgg_set_warm_states(h_, flat.data(), 1));
}

Trajectory MPC::Solve(const vector_t& state, double init_time, const std::vector<vector_3t>& ee_start_locations) {
    if (state.size() != 13) throw std::runtime_error("state has the wrong size");
    if (!have_Q_) throw std::runtime_error("no cost has been set");
    double ee[12];
    FlattenEE(ee_start_locations, ee);
    int32_t status = 0, iters = 0;
    const auto tic = std::chrono::steady_clock::now();   // utils::Timer, utils/timer.cpp:16-23
    Check(bgg_solve_batch(h_, state.data(), &init_time, ee, &status, &iters, &alpha_, &cost_, nullptr, 0));
    last_solve_ms_ = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tic).count();
    quality_ = static_cast<SolveQuality>(status);
    iters_ = iters;
    cost_sum_ += cost_;
    solves_++;
    deriv_ready_ = false;
    return GetTrajectory();
}
Trajectory MPC::CreateInitialRun(const vector_t& state, const std::vector<vector_3t>& ee_start_locations) {
    Trajectory t;
    for (int i = 0; i < 10; ++i) t = Solve(state, 0.0, ee_start_locations);   // mpc.cpp:78-90
    return t;
}
Trajectory MPC::GetRealTimeUpdate(const vector_t& state, double init_time, const std::vector<vector_3t>& ee_start_locations,
                                  bool high_quality) {
    (void)high_quality;   // both branches of the reference end in Solve (mpc.cpp:92-108)
    return Solve(state, init_time, ee_start_locations);
}
Trajectory MPC::GetTrajectory() const {
    bgg::Instance inst;
    Check(bgg_get_instance(h_, 0, &inst));
    return Trajectory(inst, info_.num_nodes, info_.integrator_dt);
}
void MPC::SetWarmStartTrajectory(const Trajectory& trajectory) {
    // prev_traj_ = trajectory; init_time_ = trajectory.GetTime(0) (mpc.cpp:110-119) -- and nothing else: the adaptive foot
    // box and the run count belong to this MPC, not to the trajectory that is handed in
    bgg::Instance inst;
    Check(bgg_get_instance(h_, 0, &inst));
    const bgg::Instance& src = trajectory.Raw();
    std::memcpy(inst.states, src.states, sizeof(inst.states));
    std::memcpy(inst.foot, src.foot, sizeof(inst.foot));
    inst.init_time = src.init_time;
    Check(bgg_set_instance(h_, 0, &inst));
}
void MPC::UpdateContactTimes(std::vector<time_v>& contact_times) {
    Trajectory t = GetTrajectory();
    t.UpdateContactTimes(contact_times);
    SetWarmStartTrajectory(t);
}
void MPC::AdjustForCurrentContacts(double time, const controller::Contact& contact) {
    Trajectory t = GetTrajectory();
    const controller::Contact tc = t.GetDesiredContacts(time);
    bool changed = false;
    for (int e = 0; e < 4; ++e)
        if (contact.in_contact_.at(e) && !tc.in_contact_.at(e) && std::abs(t.GetNextContactTime(e, time) - time) < 7e-2) {
            t.SetEEInContact(e, time);
            changed = true;
        }
    if (changed) SetWarmStartTrajectory(t);
}
int MPC::GetNumDecisionVars() const {
    bgg_sizes sz;
    Check(bgg_get_sizes(h_, 0, &sz));
    return sz.n;
}
int MPC::GetNumConstraints() const {
    bgg_sizes sz;
    Check(bgg_get_sizes(h_, 0, &sz));
    return 12 * (info_.num_nodes + 1) + sz.n_eq + sz.m_ineq;
}
vector_t MPC::GetQPSolution() const {
    bgg_sizes sz;
    Check(bgg_get_sizes(h_, 0, &sz));
    vector_t z(sz.n);
    Check(bgg_get_solution(h_, 0, nullptr, z.data(), nullptr, nullptr, nullptr));
    return z;
}
const QPData& MPC::GetQPData() const {
    bgg_sizes sz;
    Check(bgg_get_sizes(h_, 0, &sz));
    const int n_stride = 12 * (info_.num_nodes + 1) + 160, m_stride = 12 * (info_.num_nodes + 1) + 6 * 160 + 2 * (info_.num_nodes - 3) * 8 + 16;
    const int nnz_cap = 25000;   // the reference's own reserve (mpc.cpp:47)
    std::vector<int32_t> dims(6), cp(n_stride + 1), ri(nnz_cap);
    std::vector<double> va(nnz_cap), pd(n_stride), q(n_stride), ub(m_stride);
    Check(bgg_export_qp_csc(h_, 0, 1, dims.data(), cp.data(), ri.data(), va.data(), nnz_cap, pd.data(), q.data(), ub.data(), n_stride, m_stride));
    if (dims[5]) throw std::runtime_error("QP export failed");
    const int n = dims[0], m = dims[1], nnz = dims[2];
    QPData& d = data_;
    d.sparse_constraint_.rows = m;
    d.sparse_constraint_.cols = n;
    d.sparse_constraint_.outer.assign(cp.begin(), cp.begin() + n + 1);
    d.sparse_constraint_.inner.assign(ri.begin(), ri.begin() + nnz);
    d.sparse_constraint_.values.assign(va.begin(), va.begin() + nnz);
    d.cost_diag_.resize(n);
    d.cost_linear.resize(n);
    d.ub_.resize(m);
    for (int i = 0; i < n; ++i) {
        d.cost_diag_(i) = pd[i];
        d.cost_linear(i) = q[i];
    }
    for (int i = 0; i < m; ++i) d.ub_(i) = ub[i];
    d.num_decision_vars = n;
    d.num_dynamics_constraints = 12 * (info_.num_nodes + 1);
    d.num_force_box_constraints_ = 2 * sz.n_samples;
    d.num_cone_constraints_ = 4 * sz.n_samples;
    d.num_ee_location_constraints_ = 2 * sz.n_eebox;
    d.num_td_pos_constraints_ = sz.n_td;
    d.num_start_ee_constraints_ = sz.n_eq - sz.n_td;
    d.num_equality_ = dims[3];
    d.num_inequality_ = dims[4];
    d.sparse_cost_.rows = d.sparse_cost_.cols = n;    // P is diagonal on this path (mpc.cpp:542-564, 791-802, 1090-1095)
    d.sparse_cost_.outer.resize(n + 1);
    d.sparse_cost_.inner.resize(n);
    d.sparse_cost_.values.resize(n);
    for (int i = 0; i < n; ++i) {
        d.sparse_cost_.outer[i] = i;
        d.sparse_cost_.inner[i] = i;
        d.sparse_cost_.values[i] = pd[i];
    }
    d.sparse_cost_.outer[n] = n;
    d.constraints_ = {Dynamics, ForceBox, FrictionCone, EndEffectorLocation, TDPosition, EndEffectorStart};   // single_rigid_body_model.cpp:22-29
    return d;
}

// ------------------------------------------------------------------------------------------------ solver seam
std::string QPInterface::GetSolveQualityAsString() const {   // qp_interface.cpp:19-41
    switch (GetSolveQuality()) {
        case Solved: return "Solved";
        case SolvedInacc: return "Solved Inaccurate";
        case MaxIter: return "Max Iterations";
        case PrimalInfeasible: return "Primal Infeasible";
        case DualInfeasible: return "Dual Infeasible";
        case PrimalInfeasibleInacc: return "Primal Infeasible Inaccurate";
        case DualInfeasibleInacc: return "Dual Infeasible Inaccurate";
        case Unsolved: return "Unsolved";
        default: return "Other";
    }
}

static bgg_handle* MakeSolverHandle() {   // the seam needs a device, a stream and the solver settings: a handle without a batch
    bgg_config cfg{};
    cfg.num_nodes = 8;
    cfg.integrator_dt = 0.05;
    cfg.ee_box_size[0] = cfg.ee_box_size[1] = 0.15;
    bgg_robot rb{};
    rb.mass = 1.0;
    for (int i = 0; i < 3; ++i) rb.Ir[4 * i] = rb.Ir_inv[4 * i] = 1.0;
    bgg_handle* h = nullptr;
    Check(bgg_create(&cfg, &rb, &h));
    return h;
}
ClarabelInterface::ClarabelInterface(const QPData& data, bool verbose) : QPInterface(data.num_decision_vars), h_(MakeSolverHandle()), verbose_(verbose) {}
ClarabelInterface::ClarabelInterface(const ClarabelInterface& other)
    : QPInterface(other.num_decision_vars_), h_(MakeSolverHandle()), verbose_(other.verbose_), is_eq_(other.is_eq_),
      solve_quality_(other.solve_quality_), dual_(other.dual_), primal_(other.primal_), slacks_(other.slacks_), dx_(other.dx_),
      have_solution_(other.have_solution_), have_derivative_(other.have_derivative_), d_x_(other.d_x_), d_y_(other.d_y_), d_dz_(other.d_dz_),
      d_dy_(other.d_dy_), d_pattern_(other.d_pattern_), d_is_eq_(other.d_is_eq_) {}
ClarabelInterface& ClarabelInterface::operator=(const ClarabelInterface& other) {
    if (this != &other) {
        num_decision_vars_ = other.num_decision_vars_;
        verbose_ = other.verbose_;
        is_eq_ = other.is_eq_;
        solve_quality_ = other.solve_quality_;
        dual_ = other.dual_;
        primal_ = other.primal_;
        slacks_ = other.slacks_;
        dx_ = other.dx_;
        have_solution_ = other.have_solution_;
        have_derivative_ = other.have_derivative_;
        d_x_ = other.d_x_;
        d_y_ = other.d_y_;
        d_dz_ = other.d_dz_;
        d_dy_ = other.d_dy_;
        d_pattern_ = other.d_pattern_;
        d_is_eq_ = other.d_is_eq_;
    }
    return *this;
}
ClarabelInterface::~ClarabelInterface() { bgg_destroy(h_); }

void ClarabelInterface::SetupQP(QPData& data, const vector_t& /*warm_start*/) {
    // cone list in constraint-block order: Zero cones for Dynamics / TDPosition / EndEffectorStart / Raibert, Nonnegative
    // cones for EndEffectorLocation / ForceBox / FrictionCone (clarabel_interface.cpp:29-64)
    is_eq_.clear();
    for (const Constraints c : data.constraints_) {
        int n = 0;
        uint8_t eq = 0;
        switch (c) {
            case Dynamics: n = data.num_dynamics_constraints; eq = 1; break;
            case EndEffectorLocation: n = data.num_ee_location_constraints_; break;
            case ForceBox: n = data.num_force_box_constraints_; break;
            case FrictionCone: n = data.num_cone_constraints_; break;
            case TDPosition: n = data.num_td_pos_constraints_; eq = 1; break;
            case EndEffectorStart: n = data.num_start_ee_constraints_; eq = 1; break;
            case Raibert: n = data.num_raibert_constraints_; eq = 1; break;
            case JointForwardKinematics: throw std::runtime_error("not supported yet");
            case JointBox: throw std::runtime_error("Joint box not implemented with clarabel yet");
        }
        is_eq_.insert(is_eq_.end(), static_cast<size_t>(n), eq);
    }
    if (static_cast<int>(is_eq_.size()) != data.sparse_constraint_.rows) throw std::runtime_error("constraint blocks do not add up to the rows of the constraint matrix");
}

vector_t ClarabelInterface::Solve(const QPData& data) {
    const int n = data.sparse_constraint_.cols, m = data.sparse_constraint_.rows;
    if (n > 128)
        throw std::runtime_error("ClarabelInterface over bgg_qp_solve_batch takes up to 128 variables; the MPC QP is solved inside MPC::Solve (bgg_solve_batch)");
    primal_.resize(n);
    dual_.resize(m);
    slacks_.resize(m);
    int32_t status = 0, iters = 0;
    Check(bgg_qp_solve_batch(h_, 1, n, m, data.sparse_cost_.outer.data(), data.sparse_cost_.inner.data(), data.sparse_cost_.values.data(),
                             data.sparse_constraint_.outer.data(), data.sparse_constraint_.inner.data(), data.sparse_constraint_.values.data(),
                             data.cost_linear.data(), data.ub_.data(), is_eq_.data(), primal_.data(), dual_.data(), slacks_.data(), &status, &iters));
    solve_quality_ = static_cast<SolveQuality>(status);
    have_solution_ = true;
    have_derivative_ = false;
    if (solve_quality_ == PrimalInfeasible) {
        const std::string error = "Primal infeasible.";
        throw (error);   // what the caller catches (mpc_single_rigid_body.cpp:115-129)
    }
    return primal_;
}

vector_t ClarabelInterface::Computedx(const SparseCsc& P, const vector_t& q, const vector_t& xstar) {
    dx_.resize(q.size());
    for (int i = 0; i < q.size(); ++i) dx_(i) = q(i);
    for (int j = 0; j < P.cols; ++j)
        for (int k = P.outer[j]; k < P.outer[j + 1]; ++k) dx_(P.inner[k]) += P.values[k] * xstar(j);
    return dx_;
}

void ClarabelInterface::SetupDerivativeCalcs(const vector_t& dx, double dl, double du, const QPData& data) {
    if (dl != 0.0 || du != 0.0) throw std::runtime_error("ClarabelInterface::SetupDerivativeCalcs: dl and du are OSQP's bound terms and must be 0");
    if (!have_solution_) throw std::runtime_error("ClarabelInterface::SetupDerivativeCalcs: no solution is held (call Solve first)");
    const SparseCsc& A = data.sparse_constraint_;
    const int n = A.cols, m = A.rows;
    if (dx.size() != n || primal_.size() != n || dual_.size() != m || static_cast<int>(is_eq_.size()) != m)
        throw std::runtime_error("ClarabelInterface::SetupDerivativeCalcs: the QP data does not match the last Solve");
    d_dz_.resize(n);
    d_dy_.resize(m);
    int32_t status = 0;
    Check(bgg_qp_adjoint_batch(h_, 1, n, m, data.sparse_cost_.outer.data(), data.sparse_cost_.inner.data(), data.sparse_cost_.values.data(),
                               A.outer.data(), A.inner.data(), A.values.data(), is_eq_.data(), primal_.data(), dual_.data(), slacks_.data(),
                               dx.data(), d_dz_.data(), d_dy_.data(), nullptr, nullptr, &status));
    if (status != 0)
        throw std::runtime_error(status == 1 ? "ClarabelInterface::SetupDerivativeCalcs: the differential system is singular"
                                             : "ClarabelInterface::SetupDerivativeCalcs: a slack is not positive or an input is not finite");
    d_x_ = primal_;
    d_y_ = dual_;
    d_pattern_ = A;
    d_is_eq_ = is_eq_;
    have_derivative_ = true;
}

void ClarabelInterface::CalcDerivativeWrtVecs(QPPartialsDense& partials) const {
    if (!have_derivative_) throw std::runtime_error("ClarabelInterface::CalcDerivativeWrtVecs: SetupDerivativeCalcs has not run");
    const int m = d_dy_.size();
    int me = 0;
    for (uint8_t e : d_is_eq_) me += e ? 1 : 0;
    partials.dq = d_dz_;
    partials.db = vector_t::Zero(me);
    partials.dh = vector_t::Zero(m - me);
    for (int r = 0, ie = 0, ii = 0; r < m; ++r) {
        if (d_is_eq_[r]) partials.db(ie++) = -d_dy_(r);
        else partials.dh(ii++) = -d_y_(r) * d_dy_(r);   // 0 on an inequality row without entries (dlam = 0 there)
    }
}

void ClarabelInterface::CalcDerivativeWrtMats(QPPartialsDense& partials) const {
    if (!have_derivative_) throw std::runtime_error("ClarabelInterface::CalcDerivativeWrtMats: SetupDerivativeCalcs has not run");
    const int n = d_dz_.size(), m = d_dy_.size();
    std::vector<int> idx(m);   // row -> row of dA (equality) or dG (inequality)
    int me = 0, mi = 0;
    for (int r = 0; r < m; ++r) idx[r] = d_is_eq_[r] ? me++ : mi++;
    partials.dA = matrix_t::Zero(me, n);
    partials.dG = matrix_t::Zero(mi, n);
    for (int j = 0; j < n; ++j)
        for (int k = d_pattern_.outer[j]; k < d_pattern_.outer[j + 1]; ++k) {
            const int r = d_pattern_.inner[k];
            if (d_is_eq_[r]) partials.dA(idx[r], j) = d_dy_(r) * d_x_(j) + d_y_(r) * d_dz_(j);
            else partials.dG(idx[r], j) = d_y_(r) * d_dy_(r) * d_x_(j) + d_y_(r) * d_dz_(j);
        }
}

bool MPC::ComputeDerivativeTerms() {
    if (quality_ != Solved) return false;   // mpc.cpp:1047-1057
    int32_t status = 0, nct[4] = {0, 0, 0, 0};
    double dh[4 * BGG_MAX_CONTACTS];
    Check(bgg_gait_gradient_batch(h_, &status, nct, dh));
    if (status != 0) return false;
    dHdtheta_.clear();
    for (int e = 0; e < 4; ++e)
        for (int i = 0; i < nct[e]; ++i) dHdtheta_.push_back(dh[e * BGG_MAX_CONTACTS + i]);
    deriv_ready_ = true;
    return true;
}
bool MPC::GetQPPartials(QPPartialsDense& partials) const {
    if (quality_ != Solved) return false;
    partials.source = this;
    return true;
}
void MPC::PrintStats() const {
    std::printf("solves: %d, last cost: %g, avg cost: %g, last alpha: %g, last qp iterations: %d, solve quality: %d\n", solves_, cost_,
                GetAvgCost(), alpha_, iters_, static_cast<int>(quality_));
}
void MPC::PrintStatLineToFile(std::ofstream& log_file) const {
    // Same header and the same ten 15-wide columns as the reference's log (mpc.cpp:901-989), so its log readers keep working.
    char buf[512];
    const int col = 15, table = 10 * col;
    auto put = [&](const char* s, int n) { log_file.write(s, n); };
    auto rule = [&]() {
        std::string r(table, '-');
        r += "\n";
        put(r.c_str(), static_cast<int>(r.size()));
    };
    if (!used_log_file_) {
        const std::time_t now = std::time(nullptr);
        rule();
        int n = std::snprintf(buf, sizeof buf, "%*sMPC Statistics\nMPC started at: %s", table / 2 - 7, "", std::ctime(&now));
        put(buf, n);
        n = std::snprintf(buf, sizeof buf,
                          "Number of nodes: %d\nMPC time step: %g\nForce bounds: %g\nEnd Effector box size: %g %g\nForce cost: %g\n"
                          "Foot offset: %g\nSwing height: %g\n",
                          info_.num_nodes, info_.integrator_dt, info_.force_bound, info_.ee_box_size(0), info_.ee_box_size(1), info_.force_cost,
                          info_.foot_offset, info_.swing_height);
        put(buf, n);
        rule();
        n = std::snprintf(buf, sizeof buf, "%-15s%-15s%-15s%-15s%-15s%-15s%-15s%-15s%-15s%-15s\n", "Solve #", "Time (ms)", "Constraints",
                          "Step Norm", "Alpha", "Cost", "Merit", "Merit dd", "Solve Type", "QP Cost");
        put(buf, n);
        rule();
        used_log_file_ = true;
    }
    static const char* names[] = {"Solved", "Solved Inacc", "Max Iter", "P - Infeasible", "D - Infeasible", "P - Infeasible Inacc",
                                  "D - Infeasible Inacc", "Unsolved", "Other"};
    bgg_sizes sz;
    Check(bgg_get_sizes(h_, 0, &sz));
    const int n = std::snprintf(buf, sizeof buf, "%-15d%-15g%-15g%-15g%-15g%-15g%-15g%-15g%-15s%-15g\n", solves_ - 1, last_solve_ms_,
                                sz.eq_violation, sz.step_norm, sz.alpha, sz.cost, sz.merit, sz.merit_dd,
                                names[quality_ <= Other ? quality_ : Other], sz.qp_cost);
    put(buf, n);
}

// ------------------------------------------------------------------------------------------------------ MPCSingleRigidBody
bool MPCSingleRigidBody::ComputeParamPartialsClarabel(const Trajectory& traj, QPPartials& partials, int ee, int idx) {
    (void)traj;
    if (quality_ != Solved) return false;   // mpc_single_rigid_body.cpp:643
    partials.source = this;
    partials.ee = ee;
    partials.idx = idx;
    if (!export_partials_) return true;   // gait-optimisation path: the partial is generated and contracted on the device (csrc/bgg_gradient.cu)
    // the matrices themselves (:648-790), triplets in the reference's numbering -> column-compressed, duplicates summed
    int32_t counts[4] = {0, 0, 0, 0};
    int cap = 1 << 15;
    std::vector<int32_t> Ar, Ac, Gr, Gc;
    std::vector<double> Av, Gv, db;
    for (int attempt = 0; attempt < 2; ++attempt) {
        Ar.assign(cap, 0); Ac.assign(cap, 0); Gr.assign(cap, 0); Gc.assign(cap, 0);
        Av.assign(cap, 0.0); Gv.assign(cap, 0.0);
        db.assign(static_cast<size_t>(12) * (info_.num_nodes + 1) + 64, 0.0);
        const int rc = bgg_param_partials(h_, 0, ee, idx, cap, counts, Ar.data(), Ac.data(), Av.data(), Gr.data(), Gc.data(), Gv.data(), db.data());
        if (rc == 1) return false;
        if (rc == BGG_OK) break;
        if (attempt == 1 || std::max(counts[0], counts[1]) <= cap) throw std::runtime_error(std::string("bgg_param_partials: ") + bgg_last_error());
        cap = std::max(counts[0], counts[1]);
    }
    const int n = GetNumDecisionVars();
    auto to_csc = [n](int rows, int nnz, const std::vector<int32_t>& r, const std::vector<int32_t>& c, const std::vector<double>& v) {
        std::vector<std::map<int, double>> cols(n);   // setFromTriplets: duplicates summed, rows ascending within a column
        for (int k = 0; k < nnz; ++k) cols[c[k]][r[k]] += v[k];
        SparseCsc m;
        m.rows = rows;
        m.cols = n;
        m.outer.assign(n + 1, 0);
        for (int j = 0; j < n; ++j) {
            for (const auto& kv : cols[j]) {
                m.inner.push_back(kv.first);
                m.values.push_back(kv.second);
            }
            m.outer[j + 1] = static_cast<int>(m.values.size());
        }
        return m;
    };
    partials.dA = to_csc(counts[2], counts[0], Ar, Ac, Av);
    partials.dG = to_csc(counts[3], counts[1], Gr, Gc, Gv);
    partials.db = vector_t::Zero(counts[2]);
    for (int i = 0; i < counts[2]; ++i) partials.db(i) = db[i];
    partials.dh = vector_t::Zero(counts[3]);
    partials.dq = vector_t::Zero(n);
    return true;
}
std::vector<vector_2t> MPCSingleRigidBody::GetEEBoxCenter() {
    std::vector<vector_2t> c;
    for (int e = 0; e < 4; ++e) c.emplace_back(robot_.hip_xy[2 * e], robot_.hip_xy[2 * e + 1]);
    return c;
}

// ------------------------------------------------------------------------------------------------------ GaitOptimizer
GaitOptimizer::GaitOptimizer(int num_ee, int num_contact_nodes, int num_decision_vars, int num_constraints, double contact_time_ub,
                             double min_time)
    : num_ee_(num_ee) {
    (void)num_contact_nodes;
    (void)contact_time_ub;
    (void)min_time;
    if (num_ee != 4) throw std::runtime_error("GaitOptimizer: four end effectors expected");
    UpdateSizes(num_decision_vars, num_constraints);
}
void GaitOptimizer::UpdateSizes(int num_decision_vars, int num_constraints) {
    (void)num_decision_vars;
    (void)num_constraints;
    param_partials_.assign(num_ee_, {});
}
void GaitOptimizer::SetContactTimes(const std::vector<time_v>& contact_times) {
    contact_times_ = contact_times;
    xkp1_.clear();
    for (const time_v& tv : contact_times_)
        for (const SplineTimes& t : tv) xkp1_.push_back(t.GetTime());   // ContactTimesToQPVec, gait_optimizer.cpp:623-633
}
void GaitOptimizer::SetNumContactTimes(int ee, int num_times) {
    contact_times_.at(ee).resize(num_times);
    param_partials_.at(ee).resize(num_times);
}
QPPartials& GaitOptimizer::GetParameterPartials(int ee, int idx) { return param_partials_.at(ee).at(idx); }

void GaitOptimizer::ComputeCostFcnDerivWrtContactTimes() {
    const MPC* src = qp_partials_.source;
    if (!src) throw std::runtime_error("GaitOptimizer: GetQPPartials has not been called on a solved MPC");
    dHdth = src->CostDerivWrtContactTimes();   // computed by MPC::ComputeDerivativeTerms on the device
}
void GaitOptimizer::OptimizeContactTimes(double time, double actual_red_cost) { OptimizeContactTimes(time, actual_red_cost, 1, true); }
void GaitOptimizer::OptimizeContactTimes(double time, double actual_red_cost, double alpha, bool adapt_trust_region) {
    (void)actual_red_cost;
    (void)adapt_trust_region;   // trust-region adaptation is commented out in the reference (gait_optimizer.cpp:199-211)
    const MPC* src = qp_partials_.source;
    if (!src) throw std::runtime_error("GaitOptimizer: no MPC attached");
    double grad[4 * BGG_MAX_CONTACTS] = {}, step[4 * BGG_MAX_CONTACTS], xk[4 * BGG_MAX_CONTACTS], nt[4 * BGG_MAX_CONTACTS];
    int32_t st[4];
    size_t k = 0;
    for (int e = 0; e < 4; ++e)
        for (size_t i = 0; i < contact_times_[e].size(); ++i) grad[e * BGG_MAX_CONTACTS + i] = dHdth.at(k++);
    Check(bgg_optimize_contact_times_batch(src->Handle(), &time, Delta_, alpha, grad, step, xk, nt, st));
    for (int e = 0; e < 4; ++e)
        if (st[e] != 0) std::fprintf(stderr, "Max iterations reached on the gait optimization.\n");
    xk_ = xkp1_;
    step_.clear();
    xkp1_.clear();
    for (int e = 0; e < 4; ++e)
        for (size_t i = 0; i < contact_times_[e].size(); ++i) {
            step_.push_back(step[e * BGG_MAX_CONTACTS + i]);
            xkp1_.push_back(xk_[step_.size() - 1] + step_.back());
        }
    contact_times_ = ConvertQPVecToContactTimes(xkp1_);
    run_num_++;
}
std::vector<time_v> GaitOptimizer::ConvertQPVecToContactTimes(const std::vector<double>& vec) const {
    std::vector<time_v> c = contact_times_;
    size_t k = 0;
    for (int e = 0; e < num_ee_; ++e)
        for (size_t i = 0; i < c[e].size(); ++i, ++k) {
            c[e][i].SetTime(vec.at(k));
            if (i > 0) {
                const double d = c[e][i - 1].GetTime() - c[e][i].GetTime();
                if (d <= 1e-3 && d > 0) c[e][i] = c[e][i - 1];
            }
        }
    return c;
}
std::vector<time_v> GaitOptimizer::GetContactTimes(double alpha) const {
    std::vector<double> v(xk_.size());
    for (size_t i = 0; i < v.size(); ++i) v[i] = xk_[i] + alpha * step_[i];
    return ConvertQPVecToContactTimes(v);
}
double GaitOptimizer::GetStepNorm() const {
    double s = 0;
    for (double x : step_) s += x * x;
    return std::sqrt(s);
}
std::pair<std::vector<time_v>, double> GaitOptimizer::LineSearch(MPCSingleRigidBody& mpc, double time,
                                                                  const std::vector<vector_3t>& ee_locations, const vector_t& state) {
    double xk[4 * BGG_MAX_CONTACTS] = {}, step[4 * BGG_MAX_CONTACTS] = {}, ee[12], costs[LS_SIZE];
    int32_t best = -1, quality[LS_SIZE];
    size_t k = 0;
    for (int e = 0; e < 4; ++e)
        for (size_t i = 0; i < contact_times_[e].size(); ++i, ++k) {
            xk[e * BGG_MAX_CONTACTS + i] = xk_.at(k);
            step[e * BGG_MAX_CONTACTS + i] = step_.at(k);
        }
    FlattenEE(ee_locations, ee);
    Check(bgg_line_search_batch(mpc.Handle(), LS_SIZE, xk, step, state.data(), &time, ee, &best, costs, quality));
    double cost_min = 1e10;
    if (best >= 0) cost_min = costs[best];
    else std::fprintf(stderr, "no valid trajectories... using the current one.\n");
    const double alpha = static_cast<double>(best) / LS_SIZE;   // as the reference: computed before the -1 check (:735)
    return std::make_pair(GetContactTimes(alpha), cost_min);
}

}  // namespace mpc
