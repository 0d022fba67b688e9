// Host-shim test of the derivative half of the solver seam, in the shape of the reference's "Clarabel Solver" test
// (test/mpc_test.cpp:857-1004): the 3-variable QP through QPData + ClarabelInterface::SetupQP / Solve, then Computedx,
// SetupDerivativeCalcs(dx, 0, 0, qp), CalcDerivativeWrtVecs and CalcDerivativeWrtMats.  Prints "key value..." lines that
// tests/test_gpu_qp_adjoint.py checks against the oracle and the closed-form optimum.  Needs a GPU.
#include <cstdio>
#include <stdexcept>
#include <string>

#include "mpc_b200.h"

using namespace mpc;

static void PrintVec(const char* key, const vector_t& v) {
    std::printf("%s", key);
    for (int i = 0; i < v.size(); ++i) std::printf(" %.17e", v(i));
    std::printf("\n");
}
static void PrintMat(const char* key, const matrix_t& M) {   // row major
    std::printf("%s %d %d", key, static_cast<int>(M.rows()), static_cast<int>(M.cols()));
    for (int i = 0; i < M.rows(); ++i)
        for (int j = 0; j < M.cols(); ++j) std::printf(" %.17e", M(i, j));
    std::printf("\n");
}

int main() {
    try {
        // rows in Clarabel form: the two equalities, then G x <= ub and -G x <= -lb (test/mpc_test.cpp:857-904)
        QPData qp;
        qp.num_decision_vars = 3;
        qp.constraints_ = {Dynamics, ForceBox};
        qp.num_dynamics_constraints = 2;
        qp.num_force_box_constraints_ = 4;
        qp.num_equality_ = 2;
        qp.num_inequality_ = 4;
        qp.sparse_cost_.rows = qp.sparse_cost_.cols = 3;
        qp.sparse_cost_.outer = {0, 1, 2, 3};
        qp.sparse_cost_.inner = {0, 1, 2};
        qp.sparse_cost_.values = {3.001, 4.0, 0.5};
        const double A[6][3] = {{1, 1, 0}, {1.3, 0, 0.2}, {-2, 0, 0.9}, {1, 8, 5}, {2, 0, -0.9}, {-1, -8, -5}};
        const double b[6] = {1, 3, 3.1, 13.3, 2, 5};
        qp.sparse_constraint_.rows = 6;
        qp.sparse_constraint_.cols = 3;
        qp.sparse_constraint_.outer.push_back(0);
        for (int j = 0; j < 3; ++j) {
            for (int i = 0; i < 6; ++i)
                if (A[i][j] != 0.0) {
                    qp.sparse_constraint_.inner.push_back(i);
                    qp.sparse_constraint_.values.push_back(A[i][j]);
                }
            qp.sparse_constraint_.outer.push_back(static_cast<int>(qp.sparse_constraint_.inner.size()));
        }
        qp.cost_linear = vector_t(3);
        qp.cost_linear(0) = 0.1; qp.cost_linear(1) = 4.6; qp.cost_linear(2) = 2.0;
        qp.ub_ = vector_t(6);
        for (int i = 0; i < 6; ++i) qp.ub_(i) = b[i];

        ClarabelInterface clarabel(qp, false);
        clarabel.SetupQP(qp, vector_t::Zero(3));
        bool threw = false;   // no Solve yet: nothing to differentiate
        try {
            clarabel.SetupDerivativeCalcs(vector_t::Zero(3), 0, 0, qp);
        } catch (const std::runtime_error&) {
            threw = true;
        }
        std::printf("throws_before_solve %d\n", threw ? 1 : 0);

        const vector_t xs = clarabel.Solve(qp);
        std::printf("quality %d\n", static_cast<int>(clarabel.GetSolveQuality()));
        PrintVec("x", xs);
        PrintVec("y", clarabel.GetDualSolution());
        PrintVec("s", clarabel.GetSlacks());
        const vector_t dx = clarabel.Computedx(qp.sparse_cost_, qp.cost_linear, xs);
        PrintVec("dx", dx);
        clarabel.SetupDerivativeCalcs(dx, 0, 0, qp);   // the reference's call shape (mpc.cpp:1047-1056)
        QPPartialsDense partials;
        clarabel.CalcDerivativeWrtVecs(partials);
        clarabel.CalcDerivativeWrtMats(partials);
        PrintVec("dq", partials.dq);
        PrintVec("db", partials.db);
        PrintVec("dh", partials.dh);
        PrintMat("dA", partials.dA);
        PrintMat("dG", partials.dG);
        std::printf("done 1\n");
    } catch (const std::exception& e) {
        std::printf("exception %s\n", e.what());
        return 1;
    }
    return 0;
}
