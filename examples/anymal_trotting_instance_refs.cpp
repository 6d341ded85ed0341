// anymal_trotting_instance_refs.cpp -- the trotting problem of anymal_trotting.cpp with a different cost reference in every
// instance of the batch: instance b trots with its own base height offset and knee swing amplitude, on the same footholds
// and contact schedule, in one OCPSolver.  Prints the KKT error of every instance after the iterations.
//   g++ -std=c++17 -Iinclude examples/anymal_trotting_instance_refs.cpp -Lidocp_b200 -lidocp_b200
//       -Wl,-rpath,$PWD/idocp_b200 -o build/anymal_trotting_instance_refs
//   build/anymal_trotting_instance_refs [batch = 4] [iterations = 10]
#include <cstdlib>
#include <iomanip>
#include <iostream>
#include <memory>
#include <string>
#include <vector>

#include "idocp_b200/ocp_solver.hpp"

namespace idocp = idocp_b200;

// the variation of instance b
double baseHeightOffset(const int b) { return 0.01 * (b % 5) - 0.02; }
double kneeSwing(const int b) { return 1.3 + 0.1 * (b % 9); }

int main(int argc, char* argv[]) {
  const int batch = argc > 1 ? std::atoi(argv[1]) : 4;
  const int iterations = argc > 2 ? std::atoi(argv[2]) : 10;
  std::vector<int> contact_frames = {14, 24, 34, 44};  // LF, LH, RF, RH
  idocp::QuadrupedRobot robot("", contact_frames);

  const double step_length = 0.15;
  const double t_start = 0.5;
  const double t_period = 0.5;

  auto cost = std::make_shared<idocp::HybridCostFunction>();
  idocp::VectorXd q_standing = {0, 0, 0.4792, 0, 0, 0, 1, -0.1, 0.7, -1.0, -0.1, -0.7, 1.0, 0.1, 0.7, -1.0, 0.1, -0.7, 1.0};
  idocp::VectorXd q_weight = idocp::VectorXd::Constant(robot.dimv(), 10);
  idocp::VectorXd v_weight = {1, 1, 1, 1, 1, 1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.1};
  idocp::VectorXd a_weight = {0.1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01};
  idocp::TrottingSwingAngles swing_angles;
  swing_angles.front_swing_knee = 1.7;
  swing_angles.hip_swing_knee = 1.7;
  auto config_cost = std::make_shared<idocp::TrottingConfigurationSpaceCost>(robot);
  config_cost->set_ref(t_start, t_period, q_standing, step_length, swing_angles);
  config_cost->set_q_weight(q_weight);
  config_cost->set_qf_weight(q_weight);
  config_cost->set_qi_weight(q_weight);
  config_cost->set_v_weight(v_weight);
  config_cost->set_vf_weight(v_weight);
  config_cost->set_vi_weight(v_weight);
  config_cost->set_a_weight(a_weight);
  config_cost->set_dvi_weight(a_weight);
  cost->push_back(config_cost);

  auto contact_cost = std::make_shared<idocp::ContactForceCost>(robot);
  std::vector<idocp::Vector3d> f_weight(contact_frames.size(), idocp::Vector3d(0.001, 0.001, 0.001));
  contact_cost->set_f_weight(f_weight);
  contact_cost->set_fi_weight(f_weight);
  contact_cost->set_f_ref(robot);
  cost->push_back(contact_cost);

  auto constraints = std::make_shared<idocp::HybridConstraints>();
  const double mu = 0.7;
  constraints->push_back(std::make_shared<idocp::JointPositionLowerLimit>(robot));
  constraints->push_back(std::make_shared<idocp::JointPositionUpperLimit>(robot));
  constraints->push_back(std::make_shared<idocp::JointVelocityLowerLimit>(robot));
  constraints->push_back(std::make_shared<idocp::JointVelocityUpperLimit>(robot));
  constraints->push_back(std::make_shared<idocp::JointTorquesLowerLimit>(robot));
  constraints->push_back(std::make_shared<idocp::JointTorquesUpperLimit>(robot));
  constraints->push_back(std::make_shared<idocp::LinearizedFrictionCone>(robot, mu));
  constraints->push_back(std::make_shared<idocp::LinearizedImpulseFrictionCone>(robot, mu));

  const double T = 1.55;
  const int N = 30;
  const int max_num_impulse_phase = 2;
  const double t = 0;
  idocp::OCPSolver ocp_solver(robot, cost, constraints, T, N, max_num_impulse_phase + 1, 1, batch);

  // one trotting reference per instance: the shared one with the instance's base height and knee swing amplitude
  std::vector<idocp::TrottingConfigurationSpaceCost> refs;
  for (int b = 0; b < batch; ++b) {
    idocp::VectorXd q_b = q_standing;
    q_b[2] += baseHeightOffset(b);
    idocp::TrottingSwingAngles swing_b;
    swing_b.front_swing_knee = kneeSwing(b);
    swing_b.hip_swing_knee = kneeSwing(b);
    refs.emplace_back(robot);
    refs.back().set_ref(t_start, t_period, q_b, step_length, swing_b);
  }
  ocp_solver.setInstanceCostReference([&refs](double time, double* q_ref, double* v_ref) {
    idocp::VectorXd q(19);
    for (size_t b = 0; b < refs.size(); ++b) {
      refs[b].update_q_ref(time, q);
      const idocp::VectorXd v = refs[b].v_ref(time);
      for (int j = 0; j < 19; ++j) q_ref[b * 19 + j] = q[j];
      for (int j = 0; j < 18; ++j) v_ref[b * 18 + j] = v[j];
    }
  });

  robot.updateFrameKinematics(q_standing);
  std::vector<idocp::Vector3d> contact_points(robot.maxPointContacts());
  robot.getContactPoints(contact_points);
  auto contact_status_initial = robot.createContactStatus();
  contact_status_initial.activateContacts({0, 1, 2, 3});
  contact_status_initial.setContactPoints(idocp::toPoints(contact_points));
  ocp_solver.setContactStatusUniformly(contact_status_initial);

  auto contact_status_even = robot.createContactStatus();
  contact_status_even.activateContacts({1, 2});
  contact_status_even.setContactPoints(idocp::toPoints(contact_points));
  ocp_solver.pushBackContactStatus(contact_status_even, t_start);

  auto contact_status_odd = robot.createContactStatus();
  contact_points[0].coeffRef(0) += 0.5 * step_length;
  contact_points[3].coeffRef(0) += 0.5 * step_length;
  contact_status_odd.activateContacts({0, 3});
  contact_status_odd.setContactPoints(idocp::toPoints(contact_points));
  ocp_solver.pushBackContactStatus(contact_status_odd, t_start + t_period);

  contact_points[1].coeffRef(0) += step_length;
  contact_points[2].coeffRef(0) += step_length;
  contact_status_even.setContactPoints(idocp::toPoints(contact_points));
  ocp_solver.pushBackContactStatus(contact_status_even, t_start + 2 * t_period);

  idocp::VectorXd q = q_standing;
  idocp::VectorXd v = idocp::VectorXd::Zero(robot.dimv());
  ocp_solver.setSolution("q", q);
  ocp_solver.setSolution("v", v);
  idocp::Vector3d f_init(0, 0, 0.25 * robot.totalWeight());
  ocp_solver.setSolution("f", f_init);
  ocp_solver.initConstraints(t);

  for (int i = 0; i < iterations; ++i) ocp_solver.updateSolution(t, q, v);
  ocp_solver.computeKKTResidual(t, q, v);
  const std::vector<double> kkt = ocp_solver.KKTErrors();
  std::cout << std::setprecision(17);
  for (int b = 0; b < batch; ++b)
    std::cout << "instance " << b << ": base height offset = " << baseHeightOffset(b) << " knee swing = " << kneeSwing(b)
              << " KKT error = " << kkt[b] << std::endl;
  return 0;
}
