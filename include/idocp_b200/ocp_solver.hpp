// ocp_solver.hpp -- C++ host layer of the hybrid OCPSolver (floating-base ANYmal with point contacts) on top of the
// C-ABI (include/idocp_b200.h, idocp_b200_fb_*).  Header-only; link against libidocp_b200.so.
//
// Same idea as idocp_b200.hpp: the reference's class and method names, argument meaning and call order
// (examples/anymal/anymal_trotting.cpp compiles against this header after replacing the namespace):
//   idocp::Robot(path_to_urdf, contact_frames)   include/idocp/robot/robot.hpp   -> QuadrupedRobot
//   idocp::TrottingConfigurationSpaceCost        include/idocp/cost/trotting_configuration_space_cost.hpp
//   idocp::ContactForceCost                      include/idocp/cost/contact_force_cost.hpp
//   idocp::Joint{Position,Velocity,Torques,Acceleration}{Lower,Upper}Limit, LinearizedFrictionCone, LinearizedImpulseFrictionCone,
//   FrictionCone, ImpulseFrictionCone, ContactDistance
//                                                include/idocp/constraints/ *.hpp
//   idocp::OCPSolver                             include/idocp/ocp/ocp_solver.hpp:28-230
// The reference's cost / constraint plug-ins are host virtuals; here they are a closed registry of POD-parameterised
// components, and the one user-defined piece (a time-varying configuration reference, update_q_ref) stays a host
// virtual that is sampled at the time of every stage before each call (SURVEY §8b).
#ifndef IDOCP_B200_OCP_SOLVER_HPP_
#define IDOCP_B200_OCP_SOLVER_HPP_

#include <array>
#include <cmath>
#include <cstring>
#include <functional>

#include "idocp_b200.hpp"

namespace idocp_b200 {

// Robot(path_to_urdf, contact_frames) of idocp_b200.hpp is the floating-base robot; this name keeps the default arguments
class QuadrupedRobot : public Robot {
 public:
  explicit QuadrupedRobot(const std::string& path_to_urdf = "", const std::vector<int>& contact_frames = {14, 24, 34, 44})
      : Robot(path_to_urdf, contact_frames) {}
};

inline std::vector<Point3> toPoints(const std::vector<Vector3d>& v) {
  std::vector<Point3> out;
  for (const auto& e : v) out.push_back(Point3{e[0], e[1], e[2]});
  return out;
}

namespace detail {
inline void copyN(const VectorXd& v, double* dst, int n, const char* what) {
  if (v.size() != n) die(std::string("invalid size: ") + what + ".size() must be " + std::to_string(n) + "!");
  for (int i = 0; i < n; ++i) dst[i] = v[i];
}
}  // namespace detail

// Configuration-space costs of the floating-base robot.  The reference q_ref(t) (and v_ref(t)) is a host-side function
// of the stage time in every one of the reference's classes; it is sampled per stage and call (SURVEY section 8b).
class ConfigurationSpaceCostBase {
 public:
  ConfigurationSpaceCostBase() { std::memset(&w_, 0, sizeof(w_)); }
  virtual ~ConfigurationSpaceCostBase() {}
  virtual void update_q_ref(const double t, VectorXd& q_ref) const = 0;
  virtual VectorXd v_ref(const double t) const = 0;
  void set_q_weight(const VectorXd& v) { detail::copyN(v, w_.q_weight, 18, "q_weight"); }
  void set_v_weight(const VectorXd& v) { detail::copyN(v, w_.v_weight, 18, "v_weight"); }
  void set_a_weight(const VectorXd& v) { detail::copyN(v, w_.a_weight, 18, "a_weight"); }
  void set_qf_weight(const VectorXd& v) { detail::copyN(v, w_.qf_weight, 18, "qf_weight"); }
  void set_vf_weight(const VectorXd& v) { detail::copyN(v, w_.vf_weight, 18, "vf_weight"); }
  void set_qi_weight(const VectorXd& v) { detail::copyN(v, w_.qi_weight, 18, "qi_weight"); }
  void set_vi_weight(const VectorXd& v) { detail::copyN(v, w_.vi_weight, 18, "vi_weight"); }
  void set_dvi_weight(const VectorXd& v) { detail::copyN(v, w_.dvi_weight, 18, "dvi_weight"); }
  const idocp_b200_fb_problem& weights() const { return w_; }
 protected:
  idocp_b200_fb_problem w_;
};
// user-defined references derive from this name, as from the reference's cost classes
typedef ConfigurationSpaceCostBase ConfigurationReferenceBase;

// cost/configuration_space_cost.hpp for the floating base: constant q_ref, v_ref
class FloatingBaseConfigurationSpaceCost : public ConfigurationSpaceCostBase {
 public:
  explicit FloatingBaseConfigurationSpaceCost(const Robot&) : q_ref_(19), v_ref_(18) { q_ref_[6] = 1.0; }
  void set_q_ref(const VectorXd& q) { if (q.size() != 19) detail::die("invalid size: q_ref.size() must be 19!"); q_ref_ = q; }
  void set_v_ref(const VectorXd& v) { if (v.size() != 18) detail::die("invalid size: v_ref.size() must be 18!"); v_ref_ = v; }
  void update_q_ref(const double, VectorXd& q_ref) const override { q_ref = q_ref_; }
  VectorXd v_ref(const double) const override { return v_ref_; }
  // from a ConfigurationSpaceCost built with the floating-base Robot (name -> vector, idocp_b200.hpp)
  void adopt(const std::map<std::string, VectorXd>& params) {
    for (const auto& kv : params) {
      const std::string& n = kv.first;
      const VectorXd& v = kv.second;
      if (n == "q_ref") set_q_ref(v);
      else if (n == "v_ref") set_v_ref(v);
      else if (n == "q_weight") set_q_weight(v);
      else if (n == "v_weight") set_v_weight(v);
      else if (n == "a_weight") set_a_weight(v);
      else if (n == "qf_weight") set_qf_weight(v);
      else if (n == "vf_weight") set_vf_weight(v);
      else if (n == "qi_weight") set_qi_weight(v);
      else if (n == "vi_weight") set_vi_weight(v);
      else if (n == "dvi_weight") set_dvi_weight(v);
      else if (n == "u_weight" || n == "u_ref") {
        for (int i = 0; i < v.size(); ++i)
          if (n == "u_weight" && v[i] != 0.0) detail::die("unsupported: a torque cost (u_weight) on the floating-base path");
      }
    }
  }
 private:
  VectorXd q_ref_, v_ref_;
};

// cost/time_varying_configuration_space_cost.hpp:98-118: the reference moves with v_ref between t_begin and t_end.
// (integrateConfiguration(q_begin, v_ref, dt) on the free-flyer is evaluated for a base twist that is a pure
// translation, which is what the reference's examples use; a general twist is rejected.)
class TimeVaryingConfigurationSpaceCost : public ConfigurationSpaceCostBase {
 public:
  explicit TimeVaryingConfigurationSpaceCost(const Robot&) {}
  void set_ref(const Robot&, const double t_begin, const double t_end, const VectorXd& q_begin, const VectorXd& v) {
    if (t_begin >= t_end) detail::die("invalid argment: t_begin < t_end must be hold!");
    if (q_begin.size() != 19) detail::die("invalid size: q_begin.size() must be 19!");
    if (v.size() != 18) detail::die("invalid size: v.size() must be 18!");
    if (v[3] != 0.0 || v[4] != 0.0 || v[5] != 0.0) detail::die("unsupported: the reference twist must not rotate the base");
    t_begin_ = t_begin; t_end_ = t_end; q_begin_ = q_begin; v_ref_ = v;
    q_end_ = moved(t_end - t_begin);
  }
  void update_q_ref(const double t, VectorXd& q_ref) const override {
    if (t > t_begin_ && t < t_end_) q_ref = moved(t - t_begin_);
    else if (t <= t_begin_) q_ref = q_begin_;
    else q_ref = q_end_;
  }
  VectorXd v_ref(const double t) const override { return (t > t_begin_ && t < t_end_) ? v_ref_ : VectorXd::Zero(18); }
 private:
  VectorXd moved(const double dt) const {
    VectorXd q = q_begin_;
    // p += R(quat) * (v_lin dt); joints += v dt
    const double x = q[3], y = q[4], z = q[5], w = q[6];
    const double R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                         2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                         2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)};
    for (int i = 0; i < 3; ++i) q[i] += dt * (R[3 * i] * v_ref_[0] + R[3 * i + 1] * v_ref_[1] + R[3 * i + 2] * v_ref_[2]);
    for (int j = 0; j < 12; ++j) q[7 + j] += dt * v_ref_[6 + j];
    return q;
  }
  double t_begin_ = 0, t_end_ = 1;
  VectorXd q_begin_, q_end_, v_ref_;
};

struct TrottingSwingAngles {
  double front_swing_thigh = 0, front_swing_knee = 0, front_stance_thigh = 0, front_stance_knee = 0, hip_swing_thigh = 0,
         hip_swing_knee = 0, hip_stance_thigh = 0, hip_stance_knee = 0;
};

// trotting_configuration_space_cost.hpp:52-164
class TrottingConfigurationSpaceCost : public ConfigurationSpaceCostBase {
 public:
  explicit TrottingConfigurationSpaceCost(const Robot&) {}
  void set_ref(const double t_start, const double t_period, const VectorXd& q_standing, const double step_length,
               const TrottingSwingAngles& swing_angles) {
    if (q_standing.size() != 19) detail::die("invalid size: q_standing.size() must be 19!");
    if (t_period <= 0) detail::die("invalid argment: t_period must be positive!");
    if (step_length <= 0) detail::die("invalid argment: step_length must be positive!");
    t_start_ = t_start; t_period_ = t_period; q_standing_ = q_standing; step_length_ = step_length;
    v_ref_ = VectorXd::Zero(18);
    v_ref_[0] = step_length / t_period;
    swing_ = swing_angles;
  }
  void update_q_ref(const double t, VectorXd& q_ref) const override {
    q_ref = q_standing_;
    if (t > t_start_) {
      const double tau = t - t_start_;
      const int steps = static_cast<int>(std::floor(tau / t_period_));
      const double rate = (tau - steps * t_period_) / t_period_;
      const double sin2 = std::sin(M_PI_2 * rate);
      q_ref[0] += (steps + rate) * step_length_;
      if (steps % 2 == 0) {
        q_ref[9] -= sin2 * swing_.front_swing_knee;
        q_ref[12] -= sin2 * swing_.hip_stance_knee;
        q_ref[15] += sin2 * swing_.front_stance_knee;
        q_ref[18] += sin2 * swing_.hip_swing_knee;
      } else {
        q_ref[9] += sin2 * swing_.front_stance_knee;
        q_ref[12] += sin2 * swing_.hip_swing_knee;
        q_ref[15] -= sin2 * swing_.front_swing_knee;
        q_ref[18] -= sin2 * swing_.hip_stance_knee;
      }
    }
  }
  VectorXd v_ref(const double) const override { return v_ref_; }
 private:
  double t_start_ = 0, t_period_ = 1, step_length_ = 0;
  VectorXd q_standing_, v_ref_;
  TrottingSwingAngles swing_;
};

// contact_force_cost.hpp
class ContactForceCost {
 public:
  explicit ContactForceCost(const Robot&) { std::memset(&w_, 0, sizeof(w_)); }
  void set_f_ref(const Robot& robot) {
    for (int i = 0; i < 4; ++i) { w_.f_ref[3 * i] = 0; w_.f_ref[3 * i + 1] = 0; w_.f_ref[3 * i + 2] = robot.totalWeight() / 4; }
  }
  void set_f_ref(const std::vector<Vector3d>& f) { set3(f, w_.f_ref, "f_ref"); }
  void set_f_weight(const std::vector<Vector3d>& f) { set3(f, w_.f_weight, "f_weight"); }
  void set_fi_ref(const std::vector<Vector3d>& f) { set3(f, w_.fi_ref, "f_ref"); }
  void set_fi_weight(const std::vector<Vector3d>& f) { set3(f, w_.fi_weight, "f_weight"); }
  const idocp_b200_fb_problem& weights() const { return w_; }
 private:
  static void set3(const std::vector<Vector3d>& f, double* dst, const char* what) {
    if (f.size() != 4) detail::die(std::string("invalid size: ") + what + ".size() must be 4!");
    for (int i = 0; i < 4; ++i)
      for (int x = 0; x < 3; ++x) dst[3 * i + x] = f[i][x];
  }
  idocp_b200_fb_problem w_;
};

// idocp::CostFunction / idocp::Constraints are the classes of idocp_b200.hpp; the Hybrid* names of round 1 remain as aliases
using HybridCostFunction = CostFunction;
using HybridConstraints = Constraints;

// constraints: closed registry, one tag class per reference component
struct HybridConstraintComponent {
  int id;
  double mu;
  int nonlinear = 0;            // FrictionCone / ImpulseFrictionCone: the cone itself instead of its pyramid
  std::vector<double> bound;    // JointAcceleration{Lower,Upper}Limit: amin / amax
};
#define IDOCP_B200_JOINT_LIMIT(Name, Id)                                   \
  struct Name : HybridConstraintComponent {                                 \
    explicit Name(const Robot&) : HybridConstraintComponent{Id, 0.0, 0, {}} {} \
  }
IDOCP_B200_JOINT_LIMIT(JointPositionLowerLimit, IDOCP_B200_FB_POSITION_LOWER);
IDOCP_B200_JOINT_LIMIT(JointPositionUpperLimit, IDOCP_B200_FB_POSITION_UPPER);
IDOCP_B200_JOINT_LIMIT(JointVelocityLowerLimit, IDOCP_B200_FB_VELOCITY_LOWER);
IDOCP_B200_JOINT_LIMIT(JointVelocityUpperLimit, IDOCP_B200_FB_VELOCITY_UPPER);
IDOCP_B200_JOINT_LIMIT(JointTorquesLowerLimit, IDOCP_B200_FB_TORQUES_LOWER);
IDOCP_B200_JOINT_LIMIT(JointTorquesUpperLimit, IDOCP_B200_FB_TORQUES_UPPER);
#undef IDOCP_B200_JOINT_LIMIT
struct LinearizedFrictionCone : HybridConstraintComponent {
  LinearizedFrictionCone(const Robot&, const double mu) : HybridConstraintComponent{IDOCP_B200_FB_FRICTION_CONE, mu, 0, {}} {
    if (mu <= 0) detail::die("invalid value: mu must be positive!");
  }
};
struct LinearizedImpulseFrictionCone : HybridConstraintComponent {
  LinearizedImpulseFrictionCone(const Robot&, const double mu)
      : HybridConstraintComponent{IDOCP_B200_FB_IMPULSE_FRICTION_CONE, mu, 0, {}} {
    if (mu <= 0) detail::die("invalid value: mu must be positive!");
  }
};
// FrictionCone / ImpulseFrictionCone (src/constraints/friction_cone.cpp, impulse_friction_cone.cpp): two rows per contact,
// -fz <= 0 and fx^2 + fy^2 - mu^2 fz^2 <= 0; they take the place of the linearised cone of the same level
struct FrictionCone : HybridConstraintComponent {
  FrictionCone(const Robot&, const double mu) : HybridConstraintComponent{IDOCP_B200_FB_FRICTION_CONE, mu, 1, {}} {
    if (mu <= 0) detail::die("invalid value: mu must be positive!");
  }
};
struct ImpulseFrictionCone : HybridConstraintComponent {
  ImpulseFrictionCone(const Robot&, const double mu) : HybridConstraintComponent{IDOCP_B200_FB_IMPULSE_FRICTION_CONE, mu, 1, {}} {
    if (mu <= 0) detail::die("invalid value: mu must be positive!");
  }
};
// JointAccelerationLowerLimit(robot, amin) / JointAccelerationUpperLimit(robot, amax) (joint_acceleration_*_limit.cpp:
// amin <= a.tail(dimc) <= amax on the actuated joints; any vector type with size() and operator[])
struct JointAccelerationLowerLimit : HybridConstraintComponent {
  template <typename Vector>
  JointAccelerationLowerLimit(const Robot&, const Vector& amin) : HybridConstraintComponent{IDOCP_B200_FB_NUM_CONSTRAINTS, 0.0, 0, {}} {
    for (int j = 0; j < static_cast<int>(amin.size()); ++j) bound.push_back(amin[j]);
  }
};
struct JointAccelerationUpperLimit : HybridConstraintComponent {
  template <typename Vector>
  JointAccelerationUpperLimit(const Robot&, const Vector& amax) : HybridConstraintComponent{IDOCP_B200_FB_NUM_CONSTRAINTS + 1, 0.0, 0, {}} {
    for (int j = 0; j < static_cast<int>(amax.size()); ++j) bound.push_back(amax[j]);
  }
};
// ContactDistance(robot) (src/constraints/contact_distance.cpp): the contact frames of the legs in the air stay above z = 0.
// The reference builds the gradient / Hessian rows from row 2 of getFrameJacobian, which is the LOCAL-frame Jacobian
// (robot.hxx:182-188) and not the derivative of the height unless the foot frame is level; `consistent = true` uses d z / d q
// instead (the literal form does not converge on a trot, tests/test_oracle_fb_ocp.py).
struct ContactDistance : HybridConstraintComponent {
  explicit ContactDistance(const Robot&, const bool consistent = false)
      : HybridConstraintComponent{IDOCP_B200_FB_NUM_CONSTRAINTS + 2, 0.0, consistent ? 2 : 1, {}} {}
};
// OCPSolver(robot, cost, constraints, T, N, max_num_impulse, nthreads) for `batch` instances
class OCPSolver {
 public:
  OCPSolver(const Robot& robot, const std::shared_ptr<CostFunction>& cost,
            const std::shared_ptr<Constraints>& constraints, const double T, const int N, const int max_num_impulse = 0,
            const int nthreads = 1, const int batch = 1, const int device = 0)
      : OCPSolver(robot, cost, constraints, T, N, max_num_impulse, nthreads, batch, std::vector<int>{device}) {}
  // the batch sharded over several GPUs of this node by ONE solver object (idocp_b200_fb_create_sharded): the GPU counterpart
  // of the reference's nthreads.  One device is one shard.
  OCPSolver(const Robot& robot, const std::shared_ptr<CostFunction>& cost,
            const std::shared_ptr<Constraints>& constraints, const double T, const int N, const int max_num_impulse,
            const int nthreads, const int batch, const std::vector<int>& devices)
      : cost_(cost), batch_(batch) {
    if (T <= 0) detail::die("invalid value: T must be positive!");
    if (N <= 0) detail::die("invalid value: N must be positive!");
    if (max_num_impulse < 0) detail::die("invalid value: max_num_impulse must be non-negative!");
    if (nthreads <= 0) detail::die("invalid value: nthreads must be positive!");
    if (!robot.hasFloatingBase()) {
      // OCPSolver on a fixed-base robot without contacts (examples/iiwa14/ocp_benchmark.cpp): the same Newton iteration as
      // UnOCPSolver -- the general class eliminates (a, f) through ContactDynamics with dimf = 0, the specialised one u through
      // UnconstrainedDynamics; exact eliminations of one KKT system, so the iterates agree up to rounding (stated, not
      // checkable here: the reference cannot be built).  Forwarded to the specialised GPU solver.
      if (max_num_impulse != 0) detail::die("idocp_b200: a fixed-base robot has no contacts: max_num_impulse must be 0");
      un_ = std::make_shared<UnOCPSolver>(robot, cost, constraints, T, N, nthreads, batch, devices);
      return;
    }
    if (!cost || !constraints) detail::die("idocp_b200: cost and constraints must not be null");
    idocp_b200_fb_problem p = robot.fbLimits();
    p.T = T; p.N = N; p.max_num_impulse = max_num_impulse;
    if (!cost->fbConfig() && cost->fbPlain()) {   // ConfigurationSpaceCost(robot) of the floating-base robot
      auto fc = std::make_shared<FloatingBaseConfigurationSpaceCost>(robot);
      fc->adopt(cost->fbPlain()->floatingParams());
      cost->push_back(std::shared_ptr<ConfigurationSpaceCostBase>(fc));
    }
    if (cost->fbConfig()) {
      const idocp_b200_fb_problem& w = cost->fbConfig()->weights();
      std::memcpy(p.q_weight, w.q_weight, sizeof(double) * 18 * 8);   // q_weight .. dvi_weight are contiguous
    }
    if (cost->force()) {
      const idocp_b200_fb_problem& w = cost->force()->weights();
      std::memcpy(p.f_weight, w.f_weight, sizeof(double) * 12 * 4);   // f_weight, f_ref, fi_weight, fi_ref
    }
    for (int c = 0; c < IDOCP_B200_FB_NUM_CONSTRAINTS; ++c) p.enable[c] = constraints->enable()[c];
    p.mu = constraints->mu(); p.barrier = constraints->barrier(); p.fraction_rate = constraints->fractionToBoundaryRate();
    if ((constraints->enableAccelerationLimit()[0] || constraints->enableAccelerationLimit()[1]) && constraints->accelerationLimitDim() != 12)
      detail::die("invalid size: amin / amax must have one entry per actuated joint (12)");
    for (int k = 0; k < 2; ++k) {
      p.cone_nonlinear[k] = constraints->coneNonlinear()[k];
      p.enable_acceleration_limit[k] = constraints->enableAccelerationLimit()[k];
    }
    for (int j = 0; j < 12; ++j) { p.a_min[j] = constraints->aMin()[j]; p.a_max[j] = constraints->aMax()[j]; }
    p.enable_contact_distance = constraints->contactDistance();
    idocp_b200_contact_sequence* cs = nullptr;
    detail::check(idocp_b200_contact_sequence_create(4, 2 * max_num_impulse + 2, &cs));
    cs_.reset(cs, [](idocp_b200_contact_sequence* x) { idocp_b200_contact_sequence_destroy(x); });
    if (devices.empty()) detail::die("idocp_b200: OCPSolver needs at least one device");
    idocp_b200_fb_sharded* sh = nullptr;
    detail::check(idocp_b200_fb_create_sharded(&p, cs, batch, devices.data(), static_cast<int>(devices.size()), &sh));
    sh_.reset(sh, [](idocp_b200_fb_sharded* x) { idocp_b200_fb_sharded_destroy(x); });
    prob_ = p;
  }
  int batch() const { return batch_; }
  // contact schedule (ocp_solver.cpp:173-194)
  void setContactStatusUniformly(const ContactStatus& s) {
    if (un_) { if (s.maxPointContacts() != 0) detail::die("idocp_b200: a fixed-base robot has no contacts"); return; }
    std::vector<int> a; std::vector<double> pts;
    pack(s, a, pts);
    detail::check(idocp_b200_contact_sequence_set_uniform(cs_.get(), a.data(), pts.data()));
  }
  void pushBackContactStatus(const ContactStatus& s, const double switching_time) {
    std::vector<int> a; std::vector<double> pts;
    pack(s, a, pts);
    detail::check(idocp_b200_contact_sequence_push_back(cs_.get(), a.data(), pts.data(), switching_time));
  }
  void popBackContactStatus() { detail::check(idocp_b200_contact_sequence_pop_back(cs_.get())); }
  void popFrontContactStatus() { detail::check(idocp_b200_contact_sequence_pop_front(cs_.get())); }
  void setContactPoints(const int contact_phase, const std::vector<Vector3d>& contact_points) {
    std::vector<double> pts;
    for (const auto& e : contact_points) { pts.push_back(e[0]); pts.push_back(e[1]); pts.push_back(e[2]); }
    detail::check(idocp_b200_contact_sequence_set_contact_points(cs_.get(), contact_phase, pts.data()));
  }
  // setSolution(name, value): broadcast to every instance and stage ("f": one 3-vector for every contact)
  void setSolution(const std::string& name, const VectorXd& value) {
    if (un_) { un_->setSolution(name, value); return; }
    detail::check(idocp_b200_fb_sharded_set_solution(sh_.get(), name.c_str(), value.data(), 0));
  }
  void setSolution(const std::string& name, const Vector3d& value) {
    detail::check(idocp_b200_fb_sharded_set_solution(sh_.get(), name.c_str(), value.d, 0));
  }
  void setSolution(const std::string& name, const double* value_per_instance) {
    detail::check(idocp_b200_fb_sharded_set_solution(sh_.get(), name.c_str(), value_per_instance, 1));
  }
  void initConstraints(const double t) {
    if (un_) { un_->initConstraints(); return; }
    sampleReference(t);
    detail::check(idocp_b200_fb_sharded_init_constraints(sh_.get(), t));
  }
  void updateSolution(const double t, const VectorXd& q, const VectorXd& v, const bool line_search = false) {
    if (un_) { un_->updateSolution(t, q, v, line_search); return; }
    replicate(q, v);
    updateSolution(t, q_.data(), v_.data(), line_search);
  }
  void updateSolution(const double t, const double* q, const double* v, const bool line_search = false) {
    if (un_) { un_->updateSolution(t, q, v, line_search); return; }
    sampleReference(t);
    detail::check(idocp_b200_fb_sharded_update_solution(sh_.get(), t, q, v, line_search ? 1 : 0));
  }
  void computeKKTResidual(const double t, const VectorXd& q, const VectorXd& v) {
    if (un_) { un_->computeKKTResidual(t, q, v); return; }
    replicate(q, v);
    computeKKTResidual(t, q_.data(), v_.data());
  }
  void computeKKTResidual(const double t, const double* q, const double* v) {
    if (un_) { un_->computeKKTResidual(t, q, v); return; }
    sampleReference(t);
    detail::check(idocp_b200_fb_sharded_compute_kkt_residual(sh_.get(), t, q, v));
  }
  void clearLineSearchFilter() {
    if (un_) { un_->clearLineSearchFilter(); return; }
    detail::check(idocp_b200_fb_sharded_clear_line_search_filter(sh_.get()));
  }
  // Per-instance configuration references: ref(t, q_ref, v_ref) writes q_ref [batch][19] and v_ref [batch][18], row b the
  // reference of instance b at time t.  While it is set, every call samples it at the time of every stage instead of the
  // cost's reference; the line-search filter is kept, as on a change of the shared reference.
  using InstanceCostReference = std::function<void(double t, double* q_ref, double* v_ref)>;
  void setInstanceCostReference(InstanceCostReference ref) {
    if (un_) detail::die("idocp_b200: per-instance references of a fixed-base robot: use UnOCPSolver::setCostReference");
    if (!ref) detail::die("invalid argument: the per-instance reference must not be empty");
    instance_ref_ = std::move(ref);
  }
  // back to the cost's reference for every instance (it is not sampled while per-instance references are set: the next
  // initConstraints / updateSolution / computeKKTResidual samples it again)
  void clearInstanceCostReferences() {
    if (un_) return;
    instance_ref_ = nullptr;
    detail::check(idocp_b200_fb_sharded_clear_instance_cost_references(sh_.get()));
  }
  // assert(isWellDefined()) of OCPDiscretizer::discretizeOCP as a run-time error (default) or ignored like a Release build
  void setStrictDiscretization(bool strict) { detail::check(idocp_b200_fb_sharded_set_strict_discretization(sh_.get(), strict ? 1 : 0)); }
  double KKTError() { return KKTErrors()[0]; }
  std::vector<double> KKTErrors() {
    if (un_) return un_->KKTErrors();
    std::vector<double> out(batch_);
    detail::check(idocp_b200_fb_sharded_kkt_error(sh_.get(), out.data()));
    return out;
  }
  // getSolution(name): the grid stages 0..N (q, v) or 0..N-1 (a, f, u) of one instance (ocp_solver.cpp:244-280)
  std::vector<VectorXd> getSolution(const std::string& name, const int instance = 0) {
    if (un_) return un_->getSolution(name, instance);
    const int n = discretize();
    std::vector<VectorXd> out;
    std::vector<double> buf(static_cast<size_t>(batch_) * 36 * 36);
    for (int e = 0; e < n; ++e) {
      const bool grid = kind_[e] == 0, terminal = kind_[e] == 4;
      if (!(grid || (terminal && (name == "q" || name == "v")))) continue;
      const int dim = idocp_b200_fb_sharded_get(sh_.get(), e, name.c_str(), buf.data());
      detail::check(dim);
      VectorXd x(name == "f" ? dimf_[e] : dim);
      if (name == "f") {   // f_stack(): the active contacts only
        int k = 0;
        for (int i = 0; i < 4; ++i)
          if (active_[e][i]) { for (int c = 0; c < 3; ++c) x[k++] = buf[static_cast<size_t>(instance) * dim + 3 * i + c]; }
      } else {
        for (int j = 0; j < dim; ++j) x[j] = buf[static_cast<size_t>(instance) * dim + j];
      }
      out.push_back(x);
    }
    return out;
  }
  // getStateFeedbackGain(time_stage, Kq, Kv) (ocp_solver.cpp:103-113, riccati_recursion_solver.cpp:254-260): the LQR
  // gain du = Kq dq + Kv dv of the last Riccati sweep at a grid stage, row-major 12 x 18 each
  void getStateFeedbackGain(const int time_stage, std::vector<double>& Kq, std::vector<double>& Kv, const int instance = 0) {
    const int n = discretize();
    for (int e = 0; e < n; ++e) {
      if (kind_[e] != 0 || index_[e] != time_stage) continue;
      std::vector<double> buf(static_cast<size_t>(batch_) * 12 * 36);
      detail::check(idocp_b200_fb_sharded_get(sh_.get(), e, "K", buf.data()));
      Kq.assign(12 * 18, 0.0);
      Kv.assign(12 * 18, 0.0);
      for (int r = 0; r < 12; ++r)
        for (int c = 0; c < 18; ++c) {
          Kq[r * 18 + c] = buf[static_cast<size_t>(instance) * 432 + r * 36 + c];
          Kv[r * 18 + c] = buf[static_cast<size_t>(instance) * 432 + r * 36 + 18 + c];
        }
      return;
    }
    detail::die("invalid argument: time_stage outside the horizon");
  }
  void sync() {
    if (un_) { un_->sync(); return; }
    detail::check(idocp_b200_fb_sharded_sync(sh_.get()));
  }
  // the single-device solver of shard `shard` (the whole batch when the solver was built on one device)
  idocp_b200_fb_solver* handle(int shard = 0) {
    idocp_b200_fb_solver* h = nullptr;
    detail::check(idocp_b200_fb_sharded_shard(sh_.get(), shard, &h));
    return h;
  }
  // time of the first scheduled discrete event (impulse or lift); false when the schedule has none
  bool firstEventTime(double& time) const {
    int phases = 0, impulses = 0, lifts = 0;
    detail::check(idocp_b200_contact_sequence_counts(cs_.get(), &phases, &impulses, &lifts));
    bool any = false;
    if (impulses > 0) {
      int act[4]; double pts[12], ti = 0.0;
      detail::check(idocp_b200_contact_sequence_get_impulse(cs_.get(), 0, act, pts, &ti));
      time = ti; any = true;
    }
    if (lifts > 0) {
      double tl = 0.0;
      detail::check(idocp_b200_contact_sequence_get_lift_time(cs_.get(), 0, &tl));
      if (!any || tl < time) time = tl;
      any = true;
    }
    return any;
  }
  // first control input of every instance: out [batch][12]
  void getFirstControlInput(double* out) { detail::check(idocp_b200_fb_sharded_get(sh_.get(), 0, "u", out)); }

 private:
  static void pack(const ContactStatus& s, std::vector<int>& a, std::vector<double>& pts) {
    if (s.maxPointContacts() != 4) detail::die("invalid argument: contact status must have 4 contacts");
    for (int i = 0; i < 4; ++i) {
      a.push_back(s.isContactActive(i) ? 1 : 0);
      for (int c = 0; c < 3; ++c) pts.push_back(s.contactPoint(i)[c]);
    }
  }
  int discretize() {
    const int cap = IDOCP_B200_MAX_GRID + 1 + 3 * IDOCP_B200_MAX_EVENTS;
    kind_.assign(cap, 0); index_.assign(cap, 0); t_.assign(cap, 0.0); dimf_.assign(cap, 0);
    std::vector<int> act(static_cast<size_t>(cap) * 4, 0);
    const int n = idocp_b200_fb_sharded_discretize(sh_.get(), t_last_, cap, kind_.data(), index_.data(), t_.data(), nullptr,
                                                   dimf_.data(), nullptr, act.data());
    detail::check(n);
    active_.assign(n, {0, 0, 0, 0});
    for (int e = 0; e < n; ++e)
      for (int i = 0; i < 4; ++i) active_[e][i] = act[4 * e + i];
    return n;
  }
  // the reference evaluates update_q_ref(t) inside every cost call; here once per stage and call
  void sampleReference(const double t) {
    t_last_ = t;
    const int n = discretize();
    if (instance_ref_) {
      std::vector<double> q_ref(static_cast<size_t>(batch_) * 19), v_ref(static_cast<size_t>(batch_) * 18);
      for (int e = 0; e < n; ++e) {
        instance_ref_(t_[e], q_ref.data(), v_ref.data());
        const int kind = kind_[e] == 4 ? 0 : kind_[e];
        detail::check(idocp_b200_fb_sharded_set_instance_cost_reference(sh_.get(), kind, index_[e], q_ref.data(), v_ref.data()));
      }
      return;
    }
    if (!cost_->fbConfig()) return;
    VectorXd q_ref(19);
    for (int e = 0; e < n; ++e) {
      cost_->fbConfig()->update_q_ref(t_[e], q_ref);
      const int kind = kind_[e] == 4 ? 0 : kind_[e];
      const VectorXd v_ref = cost_->fbConfig()->v_ref(t_[e]);
      detail::check(idocp_b200_fb_sharded_set_cost_reference(sh_.get(), kind, index_[e], q_ref.data(), v_ref.data()));
    }
  }
  void replicate(const VectorXd& q, const VectorXd& v) {
    if (q.size() != 19) detail::die("invalid size: q.size() must be 19!");
    if (v.size() != 18) detail::die("invalid size: v.size() must be 18!");
    q_.resize(static_cast<size_t>(batch_) * 19);
    v_.resize(static_cast<size_t>(batch_) * 18);
    for (int b = 0; b < batch_; ++b) {
      for (int j = 0; j < 19; ++j) q_[static_cast<size_t>(b) * 19 + j] = q[j];
      for (int j = 0; j < 18; ++j) v_[static_cast<size_t>(b) * 18 + j] = v[j];
    }
  }
  std::shared_ptr<CostFunction> cost_;
  std::shared_ptr<idocp_b200_contact_sequence> cs_;
  std::shared_ptr<idocp_b200_fb_sharded> sh_;
  std::shared_ptr<UnOCPSolver> un_;             // fixed-base robot without contacts: the specialised solver does the work
  idocp_b200_fb_problem prob_;
  int batch_ = 1;
  double t_last_ = 0.0;
  std::vector<int> kind_, index_, dimf_;
  std::vector<double> t_, q_, v_;
  std::vector<std::array<int, 4>> active_;
  InstanceCostReference instance_ref_;
};

// hybrid/collision_checker.hxx:22-53: which contact frames are at or below the ground (z <= 0) at configuration q.  Host
// arithmetic on the four frame positions (Robot::updateFrameKinematics), not on the solver path.
class CollisionChecker {
 public:
  explicit CollisionChecker(const Robot& robot) : contact_points_(robot.maxPointContacts()) {}
  CollisionChecker() {}
  std::vector<bool> check(Robot& robot, const VectorXd& q) {
    robot.updateFrameKinematics(q);
    robot.getContactPoints(contact_points_);
    std::vector<bool> is_impulse;
    for (const auto& p : contact_points_) is_impulse.push_back(p[2] <= 0);
    return is_impulse;
  }
  const std::vector<Vector3d>& contactFramePositions() const { return contact_points_; }
  void printContactFramePositions() const {
    for (size_t i = 0; i < contact_points_.size(); ++i)
      std::cout << "contact index " << i << ": " << contact_points_[i][0] << " " << contact_points_[i][1] << " " << contact_points_[i][2] << std::endl;
  }
 private:
  std::vector<Vector3d> contact_points_;
};

// ParNMPCSolver(robot, cost, constraints, T, N, max_num_impulse, nthreads) (include/idocp/ocp/parnmpc_solver.hpp:41-193).
// Fixed-base robot without contacts (examples/iiwa14/parnmpc_benchmark.cpp): forwarded to UnParNMPCSolver, the specialisation the
// reference ships for exactly this case (same backward-correction iteration with u eliminated first; iterates agree up to
// rounding -- stated, not checkable here).  Floating-base robot with contacts: SURVEY 8(f1), NOT implemented -- the constructor
// says so and stops, it never falls back to anything else.
class ParNMPCSolver {
 public:
  ParNMPCSolver(const Robot& robot, const std::shared_ptr<CostFunction>& cost, const std::shared_ptr<Constraints>& constraints,
                const double T, const int N, const int max_num_impulse = 0, const int nthreads = 1, const int batch = 1,
                const int device = 0) {
    if (robot.hasFloatingBase())
      detail::die("idocp_b200: ParNMPCSolver for the floating-base robot with contacts is not implemented (SURVEY.md 8(f1)); "
                  "use OCPSolver");
    if (max_num_impulse != 0) detail::die("idocp_b200: a fixed-base robot has no contacts: max_num_impulse must be 0");
    un_ = std::make_shared<UnParNMPCSolver>(robot, cost, constraints, T, N, nthreads, batch, device);
  }
  void initConstraints(const double = 0.0) { un_->initConstraints(); }
  void initBackwardCorrection(const double t) { un_->initBackwardCorrection(t); }
  void updateSolution(const double t, const VectorXd& q, const VectorXd& v, const bool line_search = false) {
    un_->updateSolution(t, q, v, line_search);
  }
  void computeKKTResidual(const double t, const VectorXd& q, const VectorXd& v) { un_->computeKKTResidual(t, q, v); }
  double KKTError() { return un_->KKTError(); }
  std::vector<double> KKTErrors() { return un_->KKTErrors(); }
  void setSolution(const std::string& name, const VectorXd& value) { un_->setSolution(name, value); }
  void setSolution(const std::string&, const Vector3d&) { detail::die("idocp_b200: a fixed-base robot has no contact forces"); }
  std::vector<VectorXd> getSolution(const std::string& name, const int instance = 0) { return un_->getSolution(name, instance); }
  void clearLineSearchFilter() { un_->clearLineSearchFilter(); }
  bool isCurrentSolutionFeasible() { return un_->isCurrentSolutionFeasible(); }
  void setContactStatusUniformly(const ContactStatus& s) { if (s.maxPointContacts() != 0) detail::die("idocp_b200: a fixed-base robot has no contacts"); }
  void pushBackContactStatus(const ContactStatus&, const double) { detail::die("idocp_b200: a fixed-base robot has no contacts"); }
  void popBackContactStatus() { detail::die("idocp_b200: a fixed-base robot has no contacts"); }
  void popFrontContactStatus() { detail::die("idocp_b200: a fixed-base robot has no contacts"); }
  void sync() { un_->sync(); }
 private:
  std::shared_ptr<UnParNMPCSolver> un_;
};

// One control tick of a BATCH of MPC loops around OCPSolver (SURVEY.md 8f rank 2; Python twin: idocp_b200/mpc.py).  idocp has no
// MPC class: its consumers call, every control period, popFrontContactStatus() once the first switching time has passed
// (ocp_solver.cpp:174-194), updateSolution(t, q, v) a fixed number of times -- the iterate of the previous tick stays in
// place as the warm start -- and read getSolution(0).u.  tick() is that sequence for all instances at once.
class BatchedMPC {
 public:
  explicit BatchedMPC(OCPSolver& solver, const int iterations = 1, const bool line_search = false)
      : solver_(solver), iterations_(iterations), line_search_(line_search) {}
  // q [batch][19], v [batch][18] measured states; u0 [batch][12] receives the first control inputs
  void tick(const double t, const double* q, const double* v, double* u0) {
    double te = 0.0;
    while (solver_.firstEventTime(te) && te <= t) {   // an event before t makes the discretisation ill-defined
      solver_.popFrontContactStatus();
      ++popped_;
    }
    for (int it = 0; it < iterations_; ++it) solver_.updateSolution(t, q, v, line_search_);
    solver_.getFirstControlInput(u0);
  }
  int numPoppedPhases() const { return popped_; }
 private:
  OCPSolver& solver_;
  int iterations_;
  bool line_search_;
  int popped_ = 0;
};

}  // namespace idocp_b200
#endif  // IDOCP_B200_OCP_SOLVER_HPP_
