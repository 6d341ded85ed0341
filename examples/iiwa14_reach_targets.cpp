// iiwa14_reach_targets.cpp -- one batched UnOCPSolver, every instance with its own end-effector position target:
//
//   iiwa14_reach_targets [batch] [iterations]
//
// TaskSpace3DCost on frame 22 with per-instance reference tables (SolverBase::setTaskReference(table_per_instance)): the
// batch counterpart of one reference solver object per target, each with its own TaskSpace3DCost::set_q_3d_ref.  The targets
// lie on a line segment in front of the robot.  Prints, per instance, its target, the KKT error after the iterations and the
// final distance of the end effector to the target (host forward kinematics of the compiled-in model).  Build:
//   g++ -std=c++17 -Iinclude examples/iiwa14_reach_targets.cpp -Lidocp_b200 -lidocp_b200 -Wl,-rpath,$PWD/idocp_b200
#include <cmath>
#include <cstdlib>
#include <iomanip>
#include <iostream>
#include <memory>
#include <vector>

#include "idocp_b200/idocp_b200.hpp"
#include "../idocp_b200/csrc/model_iiwa14.h"

namespace ob = idocp_b200;

namespace {

// end-effector position of configuration q: the joint placements of the model, each joint revolute about its local z axis
void end_effector_position(const double* q, double p[3]) {
  double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, t[3] = {0, 0, 0};
  auto compose = [&](const double* Rj, const double* pj) {   // (R, t) <- (R, t) * (Rj, pj)
    double Rn[9];
    for (int r = 0; r < 3; ++r) {
      t[r] += R[3 * r] * pj[0] + R[3 * r + 1] * pj[1] + R[3 * r + 2] * pj[2];
      for (int c = 0; c < 3; ++c) Rn[3 * r + c] = R[3 * r] * Rj[c] + R[3 * r + 1] * Rj[3 + c] + R[3 * r + 2] * Rj[6 + c];
    }
    for (int k = 0; k < 9; ++k) R[k] = Rn[k];
  };
  const double zero[3] = {0, 0, 0};
  for (int j = 0; j < IIWA14_NV; ++j) {
    compose(IIWA14_PLACEMENT_R[j], IIWA14_PLACEMENT_P[j]);
    const double c = std::cos(q[j]), s = std::sin(q[j]);
    const double Rz[9] = {c, -s, 0, s, c, 0, 0, 0, 1};
    compose(Rz, zero);
  }
  compose(IIWA14_EE_PLACEMENT_R, IIWA14_EE_PLACEMENT_P);
  for (int k = 0; k < 3; ++k) p[k] = t[k];
}

}  // namespace

int main(int argc, char* argv[]) {
  const int batch = argc > 1 ? std::atoi(argv[1]) : 8;
  const int iterations = argc > 2 ? std::atoi(argv[2]) : 20;
  if (batch <= 0 || iterations < 0) {
    std::cerr << "usage: iiwa14_reach_targets [batch > 0] [iterations >= 0]\n";
    return EXIT_FAILURE;
  }
  ob::Robot robot("");
  const int n = robot.dimv();
  robot.setJointEffortLimit(ob::VectorXd::Constant(n, 50));
  robot.setJointVelocityLimit(ob::VectorXd::Constant(n, M_PI_2));
  auto cost = std::make_shared<ob::CostFunction>();
  auto joint_cost = std::make_shared<ob::ConfigurationSpaceCost>(robot);
  joint_cost->set_q_weight(ob::VectorXd::Constant(n, 0.1));    // a position cost has rank 3 in q: a small posture weight
  joint_cost->set_qf_weight(ob::VectorXd::Constant(n, 0.1));
  joint_cost->set_v_weight(ob::VectorXd::Constant(n, 0.01));
  joint_cost->set_vf_weight(ob::VectorXd::Constant(n, 0.01));
  joint_cost->set_a_weight(ob::VectorXd::Constant(n, 0.01));
  cost->push_back(joint_cost);
  auto task = std::make_shared<ob::TaskSpace3DCost>(robot, 22);
  task->set_q_3d_ref(ob::Vector3d(0.546, 0.0, 0.76));           // replaced by the per-instance tables below
  task->set_q_3d_weight(ob::Vector3d::Constant(1000));
  task->set_qf_3d_weight(ob::Vector3d::Constant(1000));
  cost->push_back(task);
  ob::JointConstraintsFactory factory(robot);
  const double T = 1.5;
  const int N = 30;
  ob::UnOCPSolver solver(robot, cost, factory.create(), T, N, 1, batch);

  // constant target of instance b in every row of its table: identity rotation (unused by the 3D cost), position p_b
  std::vector<double> targets(static_cast<size_t>(batch) * 3), tables(static_cast<size_t>(batch) * (N + 1) * 12, 0.0);
  for (int b = 0; b < batch; ++b) {
    const double s = batch > 1 ? static_cast<double>(b) / (batch - 1) : 0.5;
    const double p[3] = {0.5, -0.15 + 0.3 * s, 0.7 + 0.1 * s};
    for (int k = 0; k < 3; ++k) targets[static_cast<size_t>(b) * 3 + k] = p[k];
    for (int i = 0; i <= N; ++i) {
      double* row = &tables[(static_cast<size_t>(b) * (N + 1) + i) * 12];
      row[0] = row[4] = row[8] = 1.0;
      for (int k = 0; k < 3; ++k) row[9 + k] = p[k];
    }
  }
  solver.setTaskReference(tables.data());

  ob::VectorXd q0(n);
  for (int j = 0; j < n; ++j) q0[j] = (j % 2 == 1) ? M_PI_2 : 0.0;
  const ob::VectorXd v0 = ob::VectorXd::Zero(n);
  solver.setSolution("q", q0);
  solver.setSolution("v", v0);
  for (int k = 0; k < iterations; ++k) solver.updateSolution(0.0, q0, v0);
  solver.computeKKTResidual(0.0, q0, v0);
  const std::vector<double> kkt = solver.KKTErrors();
  std::vector<double> q(static_cast<size_t>(batch) * (N + 1) * n);
  solver.getSolutionBatch("q", q.data());
  std::cout << std::setprecision(17);
  for (int b = 0; b < batch; ++b) {
    double p[3];
    end_effector_position(&q[(static_cast<size_t>(b) * (N + 1) + N) * n], p);
    const double* tb = &targets[static_cast<size_t>(b) * 3];
    const double dist = std::sqrt((p[0] - tb[0]) * (p[0] - tb[0]) + (p[1] - tb[1]) * (p[1] - tb[1]) + (p[2] - tb[2]) * (p[2] - tb[2]));
    std::cout << "instance " << b << ": target [" << tb[0] << " " << tb[1] << " " << tb[2] << "] KKT error = " << kkt[b]
              << " distance = " << dist << std::endl;
  }
  return EXIT_SUCCESS;
}
