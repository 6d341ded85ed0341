// idocp_b200.hpp -- C++ host layer: idocp's solver-facing class API re-created on top of the
// C-ABI (include/idocp_b200.h).  Header-only; link against libidocp_b200.so.
//
// A user of the reference switches by replacing `#include "idocp/..."` with this header and the
// namespace `idocp` with `idocp_b200`; the class and method names, argument meaning and call
// order are those of the reference:
//   idocp::Robot                      include/idocp/robot/robot.hpp           (limits only: the rigid-body
//                                                                             arithmetic lives in the kernels)
//   idocp::ConfigurationSpaceCost     include/idocp/cost/configuration_space_cost.hpp
//   idocp::CostFunction               include/idocp/cost/cost_function.hpp
//   idocp::Constraints, JointConstraintsFactory   include/idocp/constraints/constraints.hpp,
//                                     include/idocp/utils/joint_constraints_factory.hpp
//   idocp::UnOCPSolver                include/idocp/unocp/unocp_solver.hpp:25-188
//   idocp::UnParNMPCSolver            include/idocp/unocp/unparnmpc_solver.hpp:37-171
//   idocp::ocpbenchmarker             include/idocp/utils/ocp_benchmarker.hxx:13-51
// Differences, all additive: Eigen is not required (a minimal VectorXd is provided), and every
// solver takes an optional `batch` (default 1 = exactly the reference object) with batched
// overloads taking row-major [batch][dimv] arrays.  Like the reference, argument errors print to
// std::cerr and std::exit(EXIT_FAILURE) (unocp_solver.cpp:33-47); `nthreads` is accepted and ignored.
#ifndef IDOCP_B200_HPP_
#define IDOCP_B200_HPP_

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <map>
#include <memory>
#include <random>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "../idocp_b200.h"
#include "hybrid.hpp"

namespace idocp_b200 {

// minimal dense vector standing in for Eigen::VectorXd
class VectorXd {
 public:
  VectorXd() {}
  explicit VectorXd(int n) : d_(n, 0.0) {}
  VectorXd(std::initializer_list<double> v) : d_(v) {}
  static VectorXd Zero(int n) { return VectorXd(n); }
  static VectorXd Constant(int n, double v) { VectorXd x(n); for (auto& e : x.d_) e = v; return x; }
  int size() const { return static_cast<int>(d_.size()); }
  double& operator[](int i) { return d_[i]; }
  double operator[](int i) const { return d_[i]; }
  double& operator()(int i) { return d_[i]; }
  double operator()(int i) const { return d_[i]; }
  double& coeffRef(int i) { return d_[i]; }
  double coeff(int i) const { return d_[i]; }
  const double* data() const { return d_.data(); }
  double* data() { return d_.data(); }
  // Eigen's comma initialiser:  v << 1, 2, 3;
  struct CommaInitializer {
    double* p;
    double* end;
    CommaInitializer& operator,(double x) {
      if (p == end) { std::cerr << "invalid size: too many coefficients in the comma initialiser\n"; std::exit(EXIT_FAILURE); }
      *p++ = x;
      return *this;
    }
    // a nested vector (Eigen block syntax:  q << 0, 0, 1, quat, joints;)
    CommaInitializer& operator,(const VectorXd& v) {
      for (int i = 0; i < v.size(); ++i) (*this), v[i];
      return *this;
    }
  };
  CommaInitializer operator<<(double x) {
    CommaInitializer c{d_.data(), d_.data() + d_.size()};
    c, x;
    return c;
  }
  void setConstant(double v) { for (auto& e : d_) e = v; }
  void setZero() { setConstant(0.0); }
 private:
  std::vector<double> d_;
};

namespace detail {
[[noreturn]] inline void die(const std::string& what) {
  std::cerr << what << '\n';
  std::exit(EXIT_FAILURE);
}
inline void check(int rc) {
  if (rc < 0) die(std::string("idocp_b200: ") + idocp_b200_last_error());
}
// The robot models are compiled into the kernels (tools/gen_robot_model.py), so a URDF path cannot change them.  A path that
// is given is therefore CHECKED: the file must exist and its kinematic / inertial content -- the text with comments,
// <visual>, <collision>, <material>, <gazebo>, <transmission> blocks and all white space removed -- must hash (FNV-1a 64)
// to the URDF the tables were generated from; anything else stops the program like the reference's failed
// pinocchio::urdf::buildModel (src/robot/robot.cpp:26,62).  An empty path selects the compiled-in model explicitly.
inline unsigned long long urdf_content_hash(const std::string& text) {
  std::string s = text;
  const char* blocks[][2] = {{"<!--", "-->"}, {"<visual", "</visual>"}, {"<collision", "</collision>"},
                             {"<gazebo", "</gazebo>"}, {"<transmission", "</transmission>"}, {"<material", "</material>"}};
  for (const auto& b : blocks) {
    std::string out;
    size_t i = 0;
    for (;;) {
      const size_t j = s.find(b[0], i);
      if (j == std::string::npos) { out.append(s, i, std::string::npos); break; }
      out.append(s, i, j - i);
      const size_t k = s.find(b[1], j);
      if (k == std::string::npos) break;
      i = k + std::string(b[1]).size();
    }
    s.swap(out);
  }
  unsigned long long h = 0xcbf29ce484222325ULL;
  for (unsigned char c : s) {
    if (c <= 32) continue;
    h ^= c;
    h *= 0x100000001b3ULL;
  }
  return h;
}
inline void verify_urdf(const std::string& path, std::initializer_list<unsigned long long> accepted, const char* robot) {
  if (path.empty()) return;
  std::ifstream f(path, std::ios::binary);
  if (!f) die("idocp_b200: cannot open the URDF file '" + path + "'");
  std::stringstream ss;
  ss << f.rdbuf();
  const unsigned long long h = urdf_content_hash(ss.str());
  for (unsigned long long a : accepted)
    if (a == h) return;
  std::ostringstream msg;
  msg << "idocp_b200: '" << path << "' is not the " << robot << " URDF the compiled-in model was generated from (content hash 0x"
      << std::hex << h << "); the kernels are specialised for that kinematic tree (tools/gen_robot_model.py)";
  die(msg.str());
}
// idocp's examples/iiwa14/iiwa_description/urdf/iiwa14.urdf (= test/urdf/iiwa14/iiwa14.urdf up to mesh paths)
constexpr unsigned long long kUrdfHashIiwa14 = 0x74d27ade0ac05ccdULL;
// examples/anymal/anymal_b_simple_description/urdf/anymal.urdf and test/urdf/anymal/anymal.urdf
constexpr unsigned long long kUrdfHashAnymalExamples = 0x4ad2ccdac3b34101ULL, kUrdfHashAnymalTests = 0xed1cb1b607c99c55ULL;
inline void copy7(const VectorXd& v, double* dst, const char* what) {
  if (v.size() != IDOCP_B200_DIMV) die(std::string("invalid size: ") + what + ".size() must be 7!");
  for (int i = 0; i < IDOCP_B200_DIMV; ++i) dst[i] = v[i];
}
}  // namespace detail

// minimal stand-ins for Eigen::Vector3d / Eigen::Matrix3d / pinocchio::SE3 in the task-space reference plug-in
struct Vector3d {
  double d[3] = {0, 0, 0};
  Vector3d() {}
  Vector3d(double x, double y, double z) { d[0] = x; d[1] = y; d[2] = z; }
  static Vector3d Constant(double v) { return Vector3d(v, v, v); }
  static Vector3d Zero() { return Vector3d(); }
  struct CommaInitializer {
    double* p;
    CommaInitializer& operator,(double x) { *p++ = x; return *this; }
  };
  CommaInitializer operator<<(double x) { d[0] = x; return CommaInitializer{d + 1}; }
  double& operator[](int i) { return d[i]; }
  double& operator()(int i) { return d[i]; }
  double operator()(int i) const { return d[i]; }
  double coeff(int i) const { return d[i]; }
  double& coeffRef(int i) { return d[i]; }
  double operator[](int i) const { return d[i]; }
};
struct Matrix3d {
  double d[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};   // row-major
  double& operator()(int r, int c) { return d[3 * r + c]; }
  double operator()(int r, int c) const { return d[3 * r + c]; }
  struct CommaInitializer {                    // Eigen fills row by row: R << r00, r01, r02, r10, ...;
    double* p;
    CommaInitializer& operator,(double x) { *p++ = x; return *this; }
  };
  CommaInitializer operator<<(double x) { d[0] = x; return CommaInitializer{d + 1}; }
};
struct SE3 {
  Matrix3d rotation;
  Vector3d translation;
  SE3() {}
  SE3(const Matrix3d& R, const Vector3d& p) : rotation(R), translation(p) {}
};

// Robot(path_to_urdf): the fixed-base iiwa14; Robot(path_to_urdf, contact_frames): ANYmal-B with the four foot frames
// {14, 24, 34, 44} (LF, LH, RF, RH) -- the two constructors of idocp::Robot (include/idocp/robot/robot.hpp:33-47).  The URDFs
// themselves are turned into constant tables off-line (tools/gen_robot_model.py); a path, when given, is verified against
// them (detail::verify_urdf).
class Robot {
 public:
  explicit Robot(const std::string& path_to_urdf = "") : urdf_(path_to_urdf) {
    detail::verify_urdf(path_to_urdf, {detail::kUrdfHashIiwa14}, "iiwa14");
    detail::check(idocp_b200_problem_default(IDOCP_B200_ROBOT_IIWA14, &p_));
  }
  Robot(const std::string& path_to_urdf, const std::vector<int>& contact_frames)
      : urdf_(path_to_urdf), frames_(contact_frames), floating_(true) {
    if (contact_frames != std::vector<int>{14, 24, 34, 44})
      detail::die("invalid argument: the contact frames of ANYmal must be {14, 24, 34, 44}");
    detail::verify_urdf(path_to_urdf, {detail::kUrdfHashAnymalExamples, detail::kUrdfHashAnymalTests}, "ANYmal");
    detail::check(idocp_b200_fb_problem_default(&fb_));
  }
  int dimq() const { return floating_ ? IDOCP_B200_FB_NQ : IDOCP_B200_DIMV; }
  int dimv() const { return floating_ ? IDOCP_B200_FB_NV : IDOCP_B200_DIMV; }
  int dimu() const { return floating_ ? IDOCP_B200_FB_NU : IDOCP_B200_DIMV; }
  int max_dimf() const { return floating_ ? IDOCP_B200_FB_MAXF : 0; }
  int dim_passive() const { return floating_ ? 6 : 0; }
  bool hasFloatingBase() const { return floating_; }
  int maxPointContacts() const { return floating_ ? 4 : 0; }
  // robot.hxx:721
  ContactStatus createContactStatus() const { return ContactStatus(maxPointContacts()); }
  double totalWeight() const {
    if (!floating_) detail::die("idocp_b200: totalWeight() is provided for the floating-base robot");
    return idocp_b200_fb_total_weight();
  }
  void updateFrameKinematics(const VectorXd& q) {
    if (!floating_ || q.size() != dimq()) detail::die("invalid size: q.size() must be 19 (floating-base robot)");
    detail::check(idocp_b200_fb_contact_frame_positions(q.data(), points_));
  }
  void getContactPoints(std::vector<Vector3d>& contact_points) const {
    contact_points.resize(4);
    for (int i = 0; i < 4; ++i) contact_points[i] = Vector3d(points_[3 * i], points_[3 * i + 1], points_[3 * i + 2]);
  }
  // robot.hxx:731-735: the contact points of the status become the current positions of the contact frames
  template <typename ContactStatusType>
  void setContactPoints(ContactStatusType& contact_status) const {
    std::vector<Vector3d> pts;
    getContactPoints(pts);
    contact_status.setContactPoints(pts);
  }
  void setJointEffortLimit(const VectorXd& v) { detail::copy7(v, p_.u_max, "joint_effort_limit"); }
  void setJointVelocityLimit(const VectorXd& v) { detail::copy7(v, p_.v_max, "joint_velocity_limit"); }
  void setLowerJointPositionLimit(const VectorXd& v) { detail::copy7(v, p_.q_min, "lower_joint_position_limit"); }
  void setUpperJointPositionLimit(const VectorXd& v) { detail::copy7(v, p_.q_max, "upper_joint_position_limit"); }
  const idocp_b200_problem& limits() const { return p_; }          // fixed base
  const idocp_b200_fb_problem& fbLimits() const { return fb_; }    // floating base
 private:
  std::string urdf_;
  std::vector<int> frames_;
  bool floating_ = false;
  idocp_b200_problem p_ = idocp_b200_problem();
  idocp_b200_fb_problem fb_ = idocp_b200_fb_problem();
  double points_[12] = {0};
};

class ConfigurationSpaceCost {
 public:
  // one class for both robots, as in the reference (cost/configuration_space_cost.hpp): with the floating-base Robot the
  // vectors have dimq = 19 / dimv = 18 entries and OCPSolver turns them into its constant-reference configuration cost
  // (examples/anymal/ocp_benchmark.cpp)
  explicit ConfigurationSpaceCost(const Robot& robot) : floating_(robot.hasFloatingBase()) { detail::check(idocp_b200_problem_default(0, &p_)); }
  void set_q_ref(const VectorXd& v) { if (!keep("q_ref", v, 19)) detail::copy7(v, p_.q_ref, "q_ref"); }
  void set_v_ref(const VectorXd& v) { if (!keep("v_ref", v, 18)) detail::copy7(v, p_.v_ref, "v_ref"); }
  void set_u_ref(const VectorXd& v) { if (!keep("u_ref", v, 12)) detail::copy7(v, p_.u_ref, "u_ref"); }
  void set_q_weight(const VectorXd& v) { if (!keep("q_weight", v, 18)) detail::copy7(v, p_.q_weight, "q_weight"); }
  void set_v_weight(const VectorXd& v) { if (!keep("v_weight", v, 18)) detail::copy7(v, p_.v_weight, "v_weight"); }
  void set_a_weight(const VectorXd& v) { if (!keep("a_weight", v, 18)) detail::copy7(v, p_.a_weight, "a_weight"); }
  void set_u_weight(const VectorXd& v) { if (!keep("u_weight", v, 12)) detail::copy7(v, p_.u_weight, "u_weight"); }
  void set_qf_weight(const VectorXd& v) { if (!keep("qf_weight", v, 18)) detail::copy7(v, p_.qf_weight, "qf_weight"); }
  void set_vf_weight(const VectorXd& v) { if (!keep("vf_weight", v, 18)) detail::copy7(v, p_.vf_weight, "vf_weight"); }
  // impulse-stage weights (configuration_space_cost.hpp:61-65): no impulse stages on the fixed-base path
  void set_qi_weight(const VectorXd& v) { keep("qi_weight", v, 18); }
  void set_vi_weight(const VectorXd& v) { keep("vi_weight", v, 18); }
  void set_dvi_weight(const VectorXd& v) { keep("dvi_weight", v, 18); }
  const idocp_b200_problem& params() const { return p_; }
  bool floating() const { return floating_; }
  const std::map<std::string, VectorXd>& floatingParams() const { return fb_; }
 private:
  bool keep(const char* name, const VectorXd& v, int n) {
    if (!floating_) return false;
    if (v.size() != n) detail::die(std::string("invalid size: ") + name + ".size() must be " + std::to_string(n) + "!");
    fb_[name] = v;
    return true;
  }
  idocp_b200_problem p_;
  bool floating_ = false;
  std::map<std::string, VectorXd> fb_;
};

// cost/time_varying_task_space_6d_cost.hpp:22-41: user-derived reference; a HOST virtual, sampled by the solver
// at the time of every stage and uploaded as a table (idocp_b200_set_task_reference)
class TimeVaryingTaskSpace6DRefBase {
 public:
  TimeVaryingTaskSpace6DRefBase() {}
  virtual ~TimeVaryingTaskSpace6DRefBase() {}
  virtual void compute_q_6d_ref(const double t, SE3& se3_ref) const = 0;
};

// cost/time_varying_task_space_6d_cost.hpp:44-150.  Supported frame: the end-effector frame of the iiwa14
// (frame id 22 = iiwa_link_ee_kuka, examples/iiwa14/task_space_ocp.cpp:67).
class TimeVaryingTaskSpace6DCost {
 public:
  TimeVaryingTaskSpace6DCost(const Robot&, const int frame_id, const std::shared_ptr<TimeVaryingTaskSpace6DRefBase>& ref)
      : ref_(ref) {
    if (frame_id != 22) detail::die("idocp_b200: TimeVaryingTaskSpace6DCost supports frame_id 22 (iiwa_link_ee_kuka) only");
    for (int k = 0; k < 6; ++k) q_[k] = qf_[k] = 0.0;
  }
  void set_ref(const std::shared_ptr<TimeVaryingTaskSpace6DRefBase>& ref) { ref_ = ref; }
  // arguments exactly as in the reference: (position_weight, rotation_weight)
  void set_q_6d_weight(const Vector3d& position_weight, const Vector3d& rotation_weight) {
    for (int k = 0; k < 3; ++k) { q_[k] = position_weight[k]; q_[3 + k] = rotation_weight[k]; }
  }
  void set_qf_6d_weight(const Vector3d& position_weight, const Vector3d& rotation_weight) {
    for (int k = 0; k < 3; ++k) { qf_[k] = position_weight[k]; qf_[3 + k] = rotation_weight[k]; }
  }
  const double* q_6d_weight() const { return q_; }
  const double* qf_6d_weight() const { return qf_; }
  const std::shared_ptr<TimeVaryingTaskSpace6DRefBase>& ref() const { return ref_; }
  // idocp_b200_problem::task_enabled of this component: 1 = 6D (log6 error), 2 = 3D position error (the 3D classes below)
  int kind() const { return kind_; }
  void set_kind(int kind) { kind_ = kind; }
 private:
  std::shared_ptr<TimeVaryingTaskSpace6DRefBase> ref_;
  double q_[6], qf_[6];
  int kind_ = 1;
};

// cost/time_varying_task_space_3d_cost.hpp:18-38: user-derived position reference (host virtual, sampled per stage)
class TimeVaryingTaskSpace3DRefBase {
 public:
  TimeVaryingTaskSpace3DRefBase() {}
  virtual ~TimeVaryingTaskSpace3DRefBase() {}
  virtual void compute_q_3d_ref(const double t, Vector3d& q_3d_ref) const = 0;
};

// cost/time_varying_task_space_3d_cost.hpp:40-150, src/cost/time_varying_task_space_3d_cost.cpp: 1/2 dt sum w (p_frame - p_ref(t))^2
// with J_3d = frameRotation * J_frame(LOCAL).topRows<3>().  Device path: the task-space cost kernels in their 3D mode
// (task_space_cost.cuh, kind 2); the reference table carries p_ref(t) of every stage (rotation entries unused).
class TimeVaryingTaskSpace3DCost {
 public:
  TimeVaryingTaskSpace3DCost(const Robot& robot, const int frame_id, const std::shared_ptr<TimeVaryingTaskSpace3DRefBase>& ref)
      : adapter_(std::make_shared<Adapter>()), cost_(std::make_shared<TimeVaryingTaskSpace6DCost>(robot, frame_id, adapter_)) {
    adapter_->ref = ref;
    cost_->set_kind(2);
  }
  void set_ref(const std::shared_ptr<TimeVaryingTaskSpace3DRefBase>& ref) { adapter_->ref = ref; }
  void set_q_3d_weight(const Vector3d& w) { cost_->set_q_6d_weight(w, Vector3d()); }
  void set_qf_3d_weight(const Vector3d& w) { cost_->set_qf_6d_weight(w, Vector3d()); }
  void set_qi_3d_weight(const Vector3d&) {}   // no impulse stages on the fixed-base path
  const std::shared_ptr<TimeVaryingTaskSpace6DCost>& component() const { return cost_; }
 private:
  struct Adapter final : TimeVaryingTaskSpace6DRefBase {
    std::shared_ptr<TimeVaryingTaskSpace3DRefBase> ref;
    void compute_q_6d_ref(const double t, SE3& se3_ref) const override {
      Vector3d p;
      if (ref) ref->compute_q_3d_ref(t, p);
      se3_ref = SE3(Matrix3d(), p);
    }
  };
  std::shared_ptr<Adapter> adapter_;
  std::shared_ptr<TimeVaryingTaskSpace6DCost> cost_;
};

// cost/task_space_3d_cost.hpp:18-60, src/cost/task_space_3d_cost.cpp:56-140: the same with a constant reference position
class TaskSpace3DCost {
 public:
  TaskSpace3DCost(const Robot& robot, const int frame_id)
      : ref_(std::make_shared<ConstantRef>()), cost_(std::make_shared<TimeVaryingTaskSpace3DCost>(robot, frame_id, ref_)) {}
  void set_q_3d_ref(const Vector3d& q_3d_ref) { ref_->p = q_3d_ref; }
  void set_q_3d_weight(const Vector3d& w) { cost_->set_q_3d_weight(w); }
  void set_qf_3d_weight(const Vector3d& w) { cost_->set_qf_3d_weight(w); }
  void set_qi_3d_weight(const Vector3d& w) { cost_->set_qi_3d_weight(w); }
  const std::shared_ptr<TimeVaryingTaskSpace6DCost>& component() const { return cost_->component(); }
 private:
  struct ConstantRef final : TimeVaryingTaskSpace3DRefBase {
    Vector3d p;
    void compute_q_3d_ref(const double, Vector3d& q_3d_ref) const override { q_3d_ref = p; }
  };
  std::shared_ptr<ConstantRef> ref_;
  std::shared_ptr<TimeVaryingTaskSpace3DCost> cost_;
};

// cost/task_space_6d_cost.hpp:22-60, src/cost/task_space_6d_cost.cpp:41-176: the same stage arithmetic as the
// time-varying component (log6 of ref^-1 * frame placement, Jlog6 * frame Jacobian) with a constant reference; it runs
// on the same device path with the reference table filled with one placement.
class TaskSpace6DCost {
 public:
  TaskSpace6DCost(const Robot& robot, const int frame_id)
      : ref_(std::make_shared<ConstantRef>()), cost_(std::make_shared<TimeVaryingTaskSpace6DCost>(robot, frame_id, ref_)) {}
  void set_q_6d_ref(const Vector3d& position_ref, const Matrix3d& rotation_ref) { ref_->se3 = SE3(rotation_ref, position_ref); }
  void set_q_6d_weight(const Vector3d& position_weight, const Vector3d& rotation_weight) {
    cost_->set_q_6d_weight(position_weight, rotation_weight);
  }
  void set_qf_6d_weight(const Vector3d& position_weight, const Vector3d& rotation_weight) {
    cost_->set_qf_6d_weight(position_weight, rotation_weight);
  }
  // impulse stages do not exist on the fixed-base path; accepted for source compatibility
  void set_qi_6d_weight(const Vector3d&, const Vector3d&) {}
  const std::shared_ptr<TimeVaryingTaskSpace6DCost>& component() const { return cost_; }
 private:
  struct ConstantRef final : TimeVaryingTaskSpace6DRefBase {
    SE3 se3;
    void compute_q_6d_ref(const double, SE3& se3_ref) const override { se3_ref = se3; }
  };
  std::shared_ptr<ConstantRef> ref_;
  std::shared_ptr<TimeVaryingTaskSpace6DCost> cost_;
};

// closed registry of cost components: one ConfigurationSpaceCost and, optionally, one task-space cost
// (TimeVaryingTaskSpace6DCost, TaskSpace6DCost, TimeVaryingTaskSpace3DCost or TaskSpace3DCost; push_back order of the reference examples: configuration cost first)
class ConfigurationSpaceCostBase;   // the configuration-space costs of the floating-base robot (ocp_solver.hpp)
class ContactForceCost;
class CostFunction {
 public:
  // floating-base components (ocp_solver.hpp): one configuration-space cost with a time-dependent reference
  // (TrottingConfigurationSpaceCost, TimeVaryingConfigurationSpaceCost, FloatingBaseConfigurationSpaceCost) and ContactForceCost
  void push_back(const std::shared_ptr<ConfigurationSpaceCostBase>& c) { fb_config_ = c; }
  void push_back(const std::shared_ptr<ContactForceCost>& c) { force_ = c; }
  const std::shared_ptr<ConfigurationSpaceCostBase>& fbConfig() const { return fb_config_; }
  const std::shared_ptr<ContactForceCost>& force() const { return force_; }
  void push_back(const std::shared_ptr<ConfigurationSpaceCost>& c) {
    if (c->floating()) { fb_plain_ = c; return; }   // OCPSolver converts it (ocp_solver.hpp)
    if (config_) detail::die("idocp_b200: only one ConfigurationSpaceCost component is supported");
    if (task_) detail::die("idocp_b200: push the ConfigurationSpaceCost before the task-space cost");
    config_ = c;
  }
  void push_back(const std::shared_ptr<TimeVaryingTaskSpace6DCost>& c) {
    if (task_) detail::die("idocp_b200: only one task-space 6D cost component is supported");
    task_ = c;
  }
  void push_back(const std::shared_ptr<TaskSpace6DCost>& c) { push_back(c->component()); }
  void push_back(const std::shared_ptr<TimeVaryingTaskSpace3DCost>& c) { push_back(c->component()); }
  void push_back(const std::shared_ptr<TaskSpace3DCost>& c) { push_back(c->component()); }
  const std::shared_ptr<ConfigurationSpaceCost>& config() const { return config_; }
  const std::shared_ptr<ConfigurationSpaceCost>& fbPlain() const { return fb_plain_; }
  const std::shared_ptr<TimeVaryingTaskSpace6DCost>& task() const { return task_; }
 private:
  std::shared_ptr<ConfigurationSpaceCost> fb_plain_;
  std::shared_ptr<ConfigurationSpaceCost> config_;
  std::shared_ptr<TimeVaryingTaskSpace6DCost> task_;
  std::shared_ptr<ConfigurationSpaceCostBase> fb_config_;
  std::shared_ptr<ContactForceCost> force_;
};

class Constraints {
 public:
  // constraints.hpp push_back: the components are tag classes {id, mu, nonlinear, bound} (ocp_solver.hpp:
  // JointPositionLowerLimit ... LinearizedImpulseFrictionCone, FrictionCone, ImpulseFrictionCone, JointAcceleration*Limit);
  // the fixed-base solvers always use the six joint limits of JointConstraintsFactory
  template <typename Component>
  void push_back(const std::shared_ptr<Component>& c) {
    if (c->id == IDOCP_B200_FB_NUM_CONSTRAINTS + 2) { contact_distance_ = c->nonlinear; return; }   // ContactDistance(robot[, consistent])
    if (c->id >= IDOCP_B200_FB_NUM_CONSTRAINTS) {   // JointAcceleration{Lower,Upper}Limit(robot, amin / amax)
      const int k = c->id - IDOCP_B200_FB_NUM_CONSTRAINTS;
      const int nb = static_cast<int>(c->bound.size());   // 7 (fixed-base iiwa14) or 12 (actuated joints of ANYmal)
      if (nb != 7 && nb != 12) detail::die("invalid size: the acceleration limit takes one bound per actuated joint (7 or 12)");
      enable_acc_[k] = 1;
      acc_dim_ = nb;
      for (int j = 0; j < nb; ++j) (k == 0 ? a_min_ : a_max_)[j] = c->bound[j];
      return;
    }
    enable_[c->id] = 1;
    if (c->mu > 0) mu_ = c->mu;
    if (c->id >= IDOCP_B200_FB_FRICTION_CONE) cone_nonlinear_[c->id - IDOCP_B200_FB_FRICTION_CONE] = c->nonlinear;
  }
  const int* coneNonlinear() const { return cone_nonlinear_; }
  const int* enableAccelerationLimit() const { return enable_acc_; }
  int accelerationLimitDim() const { return acc_dim_; }
  int contactDistance() const { return contact_distance_; }
  const double* aMin() const { return a_min_; }
  const double* aMax() const { return a_max_; }
  const int* enable() const { return enable_; }
  double mu() const { return mu_; }
  void setBarrier(double b) { if (!(b > 0)) detail::die("invalid argment: barrier must be positive"); barrier_ = b; }
  void setFractionToBoundaryRate(double r) {
    if (!(r > 0) || r > 1) detail::die("invalid argment: fraction_to_boundary_rate must be in (0, 1]");
    rate_ = r;
  }
  double barrier() const { return barrier_; }
  double fractionToBoundaryRate() const { return rate_; }
 private:
  double barrier_ = 1.0e-04, rate_ = 0.995;
  int enable_[IDOCP_B200_FB_NUM_CONSTRAINTS] = {0};
  int cone_nonlinear_[2] = {0, 0}, enable_acc_[2] = {0, 0}, acc_dim_ = 0, contact_distance_ = 0;
  double a_min_[12] = {0}, a_max_[12] = {0};
  double mu_ = 0.7;
};

// src/utils/joint_constraints_factory.cpp:22-37: position, velocity, torque lower+upper limits
class JointConstraintsFactory {
 public:
  explicit JointConstraintsFactory(const Robot&) {}
  std::shared_ptr<Constraints> create() const { return std::make_shared<Constraints>(); }
};

namespace detail {
inline idocp_b200_problem make_problem(const Robot& robot, const std::shared_ptr<CostFunction>& cost,
                                       const std::shared_ptr<Constraints>& constraints, double T, int N) {
  if (!cost || !cost->config()) die("idocp_b200: the cost function needs a ConfigurationSpaceCost component");
  if (!constraints) die("idocp_b200: constraints must not be null");
  idocp_b200_problem p = cost->config()->params();
  const idocp_b200_problem& l = robot.limits();
  for (int i = 0; i < IDOCP_B200_DIMV; ++i) {
    p.q_min[i] = l.q_min[i]; p.q_max[i] = l.q_max[i]; p.v_max[i] = l.v_max[i]; p.u_max[i] = l.u_max[i];
  }
  p.barrier = constraints->barrier();
  p.fraction_rate = constraints->fractionToBoundaryRate();
  if (constraints->enableAccelerationLimit()[0] || constraints->enableAccelerationLimit()[1]) {
    // JointAccelerationLowerLimit(robot, amin) / JointAccelerationUpperLimit(robot, amax) pushed on top of the factory's six
    if (constraints->accelerationLimitDim() != IDOCP_B200_DIMV) detail::die("invalid size: amin / amax must have dimv = 7 entries");
    for (int k = 0; k < 2; ++k) p.enable_acceleration_limit[k] = constraints->enableAccelerationLimit()[k];
    for (int j = 0; j < IDOCP_B200_DIMV; ++j) { p.a_min[j] = constraints->aMin()[j]; p.a_max[j] = constraints->aMax()[j]; }
  }
  p.T = T;
  p.N = N;
  if (cost->task()) {
    p.task_enabled = cost->task()->kind();
    for (int k = 0; k < 6; ++k) {
      p.task_q_weight[k] = cost->task()->q_6d_weight()[k];
      p.task_qf_weight[k] = cost->task()->qf_6d_weight()[k];
    }
  }
  return p;
}

class SolverBase {
 public:
  // `devices`: the GPUs of this node the batch is sharded over (contiguous shards, one device + stream each, no collective:
  // idocp_b200_create_sharded).  This is the GPU counterpart of the reference's `nthreads` (unocp_solver.cpp:11-49).
  SolverBase(int kind, const Robot& robot, const std::shared_ptr<CostFunction>& cost,
             const std::shared_ptr<Constraints>& constraints, double T, int N, int nthreads, int batch,
             const std::vector<int>& devices)
      : N_(N), batch_(batch), kind_(kind), T_(T), task_(cost ? cost->task() : nullptr) {
    try {
      if (T <= 0) throw std::out_of_range("invalid value: T must be positive!");
      if (N <= 0) throw std::out_of_range("invalid value: N must be positive!");
      if (nthreads <= 0) throw std::out_of_range("invalid value: nthreads must be positive!");
      if (batch <= 0) throw std::out_of_range("invalid value: batch must be positive!");
      if (devices.empty()) throw std::out_of_range("invalid value: devices must not be empty!");
    } catch (const std::exception& e) {
      die(e.what());
    }
    const idocp_b200_problem p = make_problem(robot, cost, constraints, T, N);
    idocp_b200_sharded* hs = nullptr;
    check(idocp_b200_create_sharded(&p, kind, batch, devices.data(), static_cast<int>(devices.size()), &hs));
    hs_ = std::shared_ptr<idocp_b200_sharded>(hs, [](idocp_b200_sharded* x) { idocp_b200_sharded_destroy(x); });
    int n = 0;
    first_.resize(devices.size() + 1);
    check(idocp_b200_sharded_num_shards(hs, &n, first_.data()));
    for (int k = 0; k < n; ++k) {
      idocp_b200_solver* h = nullptr;
      check(idocp_b200_sharded_shard(hs, k, &h));
      shards_.push_back(h);
    }
  }
  int numShards() const { return static_cast<int>(shards_.size()); }
  int batch() const { return batch_; }
  void initConstraints() { check(idocp_b200_sharded_init_constraints(hs_.get())); }
  // reference signature (one x0, broadcast to the whole batch)
  void updateSolution(double t, const VectorXd& q, const VectorXd& v, bool line_search = false) {
    rep(q, v);
    sampleTaskReference(t);
    check(idocp_b200_sharded_update_solution(hs_.get(), t, qb_.data(), vb_.data(), line_search ? 1 : 0));
  }
  // batched: q, v row-major [batch][dimv]
  void updateSolution(double t, const double* q, const double* v, bool line_search = false) {
    sampleTaskReference(t);
    check(idocp_b200_sharded_update_solution(hs_.get(), t, q, v, line_search ? 1 : 0));
  }
  void computeKKTResidual(double t, const VectorXd& q, const VectorXd& v) {
    rep(q, v);
    sampleTaskReference(t);
    check(idocp_b200_sharded_compute_kkt_residual(hs_.get(), t, qb_.data(), vb_.data()));
  }
  void computeKKTResidual(double t, const double* q, const double* v) {
    sampleTaskReference(t);
    check(idocp_b200_sharded_compute_kkt_residual(hs_.get(), t, q, v));
  }
  // KKT error of instance 0 (the reference return value); KKTErrors() gives all of them
  double KKTError() { return KKTErrors()[0]; }
  std::vector<double> KKTErrors() {
    std::vector<double> k(batch_);
    check(idocp_b200_sharded_kkt_error(hs_.get(), k.data()));
    return k;
  }
  void setSolution(const std::string& name, const VectorXd& value) {
    try {
      if (name != "q" && name != "v" && name != "a" && name != "u")
        throw std::invalid_argument("invalid arugment: name must be q, v, a, or u!");
    } catch (const std::exception& e) {
      die(e.what());
    }
    double x[IDOCP_B200_DIMV];
    copy7(value, x, name.c_str());
    check(idocp_b200_sharded_set_solution(hs_.get(), name.c_str(), x, 1));
  }
  void setSolution(const std::string& name, const double* value_per_instance) {
    check(idocp_b200_sharded_set_solution(hs_.get(), name.c_str(), value_per_instance, 0));
  }
  // getSolution(name) of instance `instance`: one VectorXd per stage
  std::vector<VectorXd> getSolution(const std::string& name, int instance = 0) const {
    const bool full = (name == "q" || name == "v" || name == "lmd" || name == "gmm") && kind_ == IDOCP_B200_SOLVER_UNOCP;
    const int ns = full ? N_ + 1 : N_;
    std::vector<double> buf(static_cast<size_t>(batch_) * ns * IDOCP_B200_DIMV);
    check(idocp_b200_sharded_get_solution(hs_.get(), name.c_str(), buf.data()));
    std::vector<VectorXd> out;
    for (int i = 0; i < ns; ++i) {
      VectorXd x(IDOCP_B200_DIMV);
      for (int j = 0; j < IDOCP_B200_DIMV; ++j) x[j] = buf[(static_cast<size_t>(instance) * ns + i) * IDOCP_B200_DIMV + j];
      out.push_back(x);
    }
    return out;
  }
  void getSolutionBatch(const std::string& name, double* out) const {
    check(idocp_b200_sharded_get_solution(hs_.get(), name.c_str(), out));
  }
  // unocp_solver.cpp:312-352 / unparnmpc_solver.cpp: one stage per line, coefficients followed by a blank, default
  // stream formatting.  `instance` selects the member of the batch (the reference has one).
  void saveSolution(const std::string& path_to_file, const std::string& name, int instance = 0) const {
    std::ofstream file(path_to_file);
    if (name == "q" || name == "v" || name == "a" || name == "u") {
      for (const VectorXd& x : getSolution(name, instance)) {
        for (int j = 0; j < x.size(); ++j) file << x[j] << " ";
        file << "\n";
      }
    }
    file.close();
  }
  // unocp_solver.cpp:264-310: "q[i] = ..." lines in Eigen's row-vector format (columns right-aligned to the widest
  // coefficient).  "end-effector" needs the frame kinematics on the host and is not provided.
  void printSolution(const std::string& name = "all", const std::vector<int> frames = {}, int instance = 0) const {
    (void)frames;
    const bool unocp = kind_ == IDOCP_B200_SOLVER_UNOCP;
    auto row = [](const char* n, int i, const VectorXd& x) {
      std::vector<std::string> c;
      size_t w = 0;
      for (int j = 0; j < x.size(); ++j) {
        std::ostringstream o;
        o << x[j];
        c.push_back(o.str());
        w = std::max(w, c.back().size());
      }
      std::cout << n << "[" << i << "] = ";
      for (size_t j = 0; j < c.size(); ++j) std::cout << (j ? " " : "") << std::string(w - c[j].size(), ' ') << c[j];
      std::cout << std::endl;
    };
    if (name == "all") {
      const auto q = getSolution("q", instance), v = getSolution("v", instance), a = getSolution("a", instance),
                 u = getSolution("u", instance);
      for (int i = 0; i < N_; ++i) { row("q", i, q[i]); row("v", i, v[i]); row("a", i, a[i]); row("u", i, u[i]); }
      if (unocp) { row("q", N_, q[N_]); row("v", N_, v[N_]); }
    } else if (name == "q" || name == "v" || name == "a" || name == "u") {
      const auto x = getSolution(name, instance);
      for (size_t i = 0; i < x.size(); ++i) row(name.c_str(), static_cast<int>(i), x[i]);
    } else if (name == "end-effector") {
      std::cout << "idocp_b200: printSolution(\"end-effector\") is not provided (frame kinematics live on the device)" << std::endl;
    }
  }
  void clearLineSearchFilter() { check(idocp_b200_sharded_clear_line_search_filter(hs_.get())); }
  // Per-instance cost references (idocp_b200_set_instance_reference): the batch counterpart of one solver object per instance,
  // each with its own ConfigurationSpaceCost::set_q_ref / set_v_ref / set_u_ref.  name in {"q_ref", "v_ref", "u_ref"},
  // per_instance row-major [batch][dimv]; the fields not set start as the cost's.  The line-search filter is kept.
  void setCostReference(const std::string& name, const double* per_instance) {
    check(idocp_b200_sharded_set_instance_reference(hs_.get(), name.c_str(), per_instance));
  }
  // per-instance task-space reference table_per_instance[batch][N+1][12] = [R row-major (9), p (3)] per stage index, rows as
  // the cost's reference is sampled (sampleTaskReference); while it is set, the cost's reference object is not sampled
  void setTaskReference(const double* table_per_instance) {
    check(idocp_b200_sharded_set_instance_task_reference(hs_.get(), table_per_instance));
    instance_tables_ = true;
  }
  // back to the cost's references for every instance (the reference object is sampled again at the next call)
  void clearInstanceReferences() {
    check(idocp_b200_sharded_clear_instance_references(hs_.get()));
    instance_tables_ = false;
    task_sampled_ = false;
  }
  // fuse the update with the linearisation of the new iterate (UnOCPSolver, default on; results are bit-identical)
  void setPipelining(bool enabled) { for (idocp_b200_solver* h : shards_) check(idocp_b200_set_pipelining(h, enabled ? 1 : 0)); }
  bool isCurrentSolutionFeasible() {
    std::vector<int> f(batch_);
    for (size_t k = 0; k < shards_.size(); ++k) check(idocp_b200_is_feasible(shards_[k], f.data() + first_[k]));
    for (int b = 0; b < batch_; ++b)
      if (!f[b]) { std::cout << "INFEASIBLE instance " << b << std::endl; return false; }
    return true;
  }
  void sync() { check(idocp_b200_sharded_sync(hs_.get())); }
  // the single-device solver of shard `shard` (the whole batch when the solver was built on one device)
  idocp_b200_solver* handle(int shard = 0) { return shards_[shard]; }

  // DerivativeChecker's device pass (idocp_b200_check_cost_derivatives, first shard): n <= batch samples of (q, v, a, u),
  // task-space reference at time t; out[n][IDOCP_B200_DC_DOUBLES]
  void checkCostDerivatives(double t, bool terminal, int n, const double* q, const double* v, const double* a, const double* u,
                            double finite_diff, double* out) {
    sampleTaskReference(t);
    check(idocp_b200_check_cost_derivatives(shards_[0], terminal ? 1 : 0, 0, n, q, v, a, u, finite_diff, out));
  }

 protected:
  // the user's compute_q_6d_ref at the time of every stage index (unocp_solver.cpp:80-93: t + i dt, terminal
  // t + T; unbackward_correction.cpp:73-95: t + (i+1) dt, last stage t + T), re-sampled only when t changes
  void sampleTaskReference(double t) {
    if (!task_ || !task_->ref() || instance_tables_) return;
    if (task_sampled_ && t == task_t_) return;
    const double dt = T_ / N_;
    std::vector<double> table(static_cast<size_t>(N_ + 1) * 12);
    for (int i = 0; i <= N_; ++i) {
      double ti;
      if (kind_ == IDOCP_B200_SOLVER_UNOCP) ti = i < N_ ? t + i * dt : t + T_;
      else ti = i < N_ - 1 ? t + (i + 1) * dt : (i == N_ - 1 ? t + T_ : t + N_ * dt);
      SE3 ref;
      task_->ref()->compute_q_6d_ref(ti, ref);
      for (int k = 0; k < 9; ++k) table[static_cast<size_t>(i) * 12 + k] = ref.rotation.d[k];
      for (int k = 0; k < 3; ++k) table[static_cast<size_t>(i) * 12 + 9 + k] = ref.translation.d[k];
    }
    check(idocp_b200_sharded_set_task_reference(hs_.get(), table.data()));
    task_sampled_ = true;
    task_t_ = t;
  }
  void rep(const VectorXd& q, const VectorXd& v) {
    qb_.resize(static_cast<size_t>(batch_) * IDOCP_B200_DIMV);
    vb_.resize(qb_.size());
    double x[IDOCP_B200_DIMV], y[IDOCP_B200_DIMV];
    copy7(q, x, "q");
    copy7(v, y, "v");
    for (int b = 0; b < batch_; ++b)
      for (int j = 0; j < IDOCP_B200_DIMV; ++j) {
        qb_[static_cast<size_t>(b) * IDOCP_B200_DIMV + j] = x[j];
        vb_[static_cast<size_t>(b) * IDOCP_B200_DIMV + j] = y[j];
      }
  }
  std::shared_ptr<idocp_b200_sharded> hs_;
  std::vector<idocp_b200_solver*> shards_;   // borrowed from hs_
  std::vector<int> first_;                   // first instance of every shard, first_[n] = batch
  int N_, batch_, kind_;
  double T_;
  std::shared_ptr<TimeVaryingTaskSpace6DCost> task_;
  bool task_sampled_ = false;
  bool instance_tables_ = false;   // setTaskReference(table_per_instance) is in force: the cost's reference is not sampled
  double task_t_ = 0.0;
  std::vector<double> qb_, vb_;
};
}  // namespace detail

class UnOCPSolver : public detail::SolverBase {
 public:
  UnOCPSolver(const Robot& robot, const std::shared_ptr<CostFunction>& cost,
              const std::shared_ptr<Constraints>& constraints, const double T, const int N, const int nthreads = 1,
              const int batch = 1, const int device = 0)
      : SolverBase(IDOCP_B200_SOLVER_UNOCP, robot, cost, constraints, T, N, nthreads, batch, std::vector<int>{device}) {}
  // the batch sharded over several GPUs of this node
  UnOCPSolver(const Robot& robot, const std::shared_ptr<CostFunction>& cost,
              const std::shared_ptr<Constraints>& constraints, const double T, const int N, const int nthreads,
              const int batch, const std::vector<int>& devices)
      : SolverBase(IDOCP_B200_SOLVER_UNOCP, robot, cost, constraints, T, N, nthreads, batch, devices) {}
};

class UnParNMPCSolver : public detail::SolverBase {
 public:
  UnParNMPCSolver(const Robot& robot, const std::shared_ptr<CostFunction>& cost,
                  const std::shared_ptr<Constraints>& constraints, const double T, const int N,
                  const int nthreads = 1, const int batch = 1, const int device = 0)
      : SolverBase(IDOCP_B200_SOLVER_UNPARNMPC, robot, cost, constraints, T, N, nthreads, batch, std::vector<int>{device}) {}
  UnParNMPCSolver(const Robot& robot, const std::shared_ptr<CostFunction>& cost,
                  const std::shared_ptr<Constraints>& constraints, const double T, const int N, const int nthreads,
                  const int batch, const std::vector<int>& devices)
      : SolverBase(IDOCP_B200_SOLVER_UNPARNMPC, robot, cost, constraints, T, N, nthreads, batch, devices) {}
  void initBackwardCorrection(const double t) {
    sampleTaskReference(t);
    detail::check(idocp_b200_sharded_init_backward_correction(hs_.get(), t));
  }
};

// include/idocp/utils/derivative_checker.hpp:14-66 (src/utils/derivative_checker.cpp:47-312), evaluated on the device: at
// `samples` random split solutions (SplitSolution::Random: uniform in [-1, 1]) and a random time the analytic gradient of the
// cost component -- the lineariser's device functions -- is compared with forward differences of the cost value -- the line
// search's device functions -- and the analytic Hessian with forward differences of the gradient, block by block with Eigen's
// isApprox(test_tol); the first block that fails is reported like the reference's message.  The reference draws one sample;
// here every sample has to pass.  Fixed-base robot only: the stage / impulse costs of the floating-base robot are checked
// against finite differences on the oracle (tests/test_oracle_fb_ocp.py), which the kernels equal bit for bit.
class DerivativeChecker {
 public:
  explicit DerivativeChecker(const Robot& robot, const double finite_diff = 1.0e-08, const double test_tol = 1.0e-04,
                             const int samples = 8, const int device = 0)
      : robot_(robot), finite_diff_(finite_diff), test_tol_(test_tol), samples_(samples), device_(device) {
    if (robot.hasFloatingBase()) detail::die("idocp_b200: DerivativeChecker covers the fixed-base robot (SURVEY.md 8(f3))");
    if (samples <= 0) detail::die("invalid value: samples must be positive!");
  }
  void setFiniteDifference(const double finite_diff = 1.0e-08) { finite_diff_ = finite_diff; }
  void setTestTolerance(const double test_tol = 1.0e-04) { test_tol_ = test_tol; }
  template <class Cost> bool checkFirstOrderStageCostDerivatives(const std::shared_ptr<Cost>& cost) { return run(cost, false, false); }
  template <class Cost> bool checkSecondOrderStageCostDerivatives(const std::shared_ptr<Cost>& cost) { return run(cost, false, true); }
  template <class Cost> bool checkFirstOrderTerminalCostDerivatives(const std::shared_ptr<Cost>& cost) { return run(cost, true, false); }
  template <class Cost> bool checkSecondOrderTerminalCostDerivatives(const std::shared_ptr<Cost>& cost) { return run(cost, true, true); }

 private:
  static void add(CostFunction& cf, const Robot&, const std::shared_ptr<ConfigurationSpaceCost>& c) { cf.push_back(c); }
  template <class Task>
  static void add(CostFunction& cf, const Robot& robot, const std::shared_ptr<Task>& c) {
    auto zero = std::make_shared<ConfigurationSpaceCost>(robot);   // the solver's problem always carries the quadratic term
    const VectorXd z = VectorXd::Zero(IDOCP_B200_DIMV);
    zero->set_q_weight(z); zero->set_v_weight(z); zero->set_a_weight(z); zero->set_u_weight(z); zero->set_qf_weight(z); zero->set_vf_weight(z);
    cf.push_back(zero);
    cf.push_back(c);
  }
  // Eigen: a.isApprox(b, prec)  <=>  |a - b|^2 <= prec^2 min(|a|^2, |b|^2)
  static bool approx(const double* a, const double* b, int n, double prec) {
    double d2 = 0, a2 = 0, b2 = 0;
    for (int i = 0; i < n; ++i) { d2 += (a[i] - b[i]) * (a[i] - b[i]); a2 += a[i] * a[i]; b2 += b[i] * b[i]; }
    return d2 <= prec * prec * std::min(a2, b2);
  }
  template <class Cost>
  bool run(const std::shared_ptr<Cost>& cost, bool terminal, bool second) {
    auto cf = std::make_shared<CostFunction>();
    add(*cf, robot_, cost);
    UnOCPSolver solver(robot_, cf, std::make_shared<Constraints>(), 1.0, 2, 1, samples_, device_);   // dt = 0.5
    const int n = IDOCP_B200_DIMV;
    std::vector<double> x[4], out(static_cast<size_t>(samples_) * IDOCP_B200_DC_DOUBLES);
    for (auto& block : x) {
      block.resize(static_cast<size_t>(samples_) * n);
      for (auto& e : block) e = uniform();
    }
    solver.checkCostDerivatives(std::abs(uniform()), terminal, samples_, x[0].data(), x[1].data(), x[2].data(), x[3].data(), finite_diff_,
                                out.data());
    static const char* const first[4] = {"lq", "lv", "la", "lu"};
    static const char* const hess[4] = {"Qqq", "Qvv", "Qaa", "Quu"};
    const int blocks = terminal ? 2 : 4;
    for (int b = 0; b < samples_; ++b) {
      const double* o = out.data() + static_cast<size_t>(b) * IDOCP_B200_DC_DOUBLES;
      for (int k = 0; k < blocks; ++k) {
        bool ok;
        if (!second) {
          ok = approx(o + 1 + k * n, o + 29 + k * n, n, test_tol_);
        } else {
          double H[49] = {0};
          if (k == 0) std::copy(o + 57, o + 106, H);
          else for (int i = 0; i < n; ++i) H[i * n + i] = o[106 + (k - 1) * n + i];
          ok = approx(H, o + 127 + 49 * k, 49, test_tol_);
        }
        if (!ok) {
          std::cout << (second ? hess[k] : first[k]) << " is not correct! (sample " << b << ")" << std::endl;
          return false;
        }
      }
    }
    return true;
  }
  double uniform() { return std::uniform_real_distribution<double>(-1.0, 1.0)(rng_); }
  Robot robot_;
  double finite_diff_, test_tol_;
  int samples_, device_;
  std::mt19937 rng_{20240017u};
};

// include/idocp/utils/ocp_benchmarker.hxx:13-51
namespace ocpbenchmarker {
template <typename OCPSolverType>
inline void CPUTime(OCPSolverType& ocp_solver, const double t, const VectorXd& q, const VectorXd& v,
                    const int num_iteration, const bool line_search) {
  ocp_solver.sync();
  const auto start_clock = std::chrono::system_clock::now();
  for (int i = 0; i < num_iteration; ++i) ocp_solver.updateSolution(t, q, v, line_search);
  ocp_solver.sync();
  const auto end_clock = std::chrono::system_clock::now();
  const double ms = 1e-03 * std::chrono::duration_cast<std::chrono::microseconds>(end_clock - start_clock).count();
  std::cout << "---------- OCP benchmark : CPU time ----------" << std::endl;
  std::cout << "total CPU time: " << ms << "[ms]" << std::endl;
  std::cout << "CPU time per update: " << ms / num_iteration << "[ms]" << std::endl;
  std::cout << "-----------------------------------" << std::endl << std::endl;
}

template <typename OCPSolverType>
inline void Convergence(OCPSolverType& ocp_solver, const double t, const VectorXd& q, const VectorXd& v,
                        const int num_iteration, const bool line_search) {
  std::cout << "---------- OCP benchmark : Convergence ----------" << std::endl;
  ocp_solver.computeKKTResidual(t, q, v);
  std::cout << "Initial KKT error = " << ocp_solver.KKTError() << std::endl;
  for (int i = 0; i < num_iteration; ++i) {
    ocp_solver.updateSolution(t, q, v, line_search);
    ocp_solver.computeKKTResidual(t, q, v);
    std::cout << "KKT error after iteration " << i + 1 << " = " << ocp_solver.KKTError() << std::endl;
  }
  std::cout << "-----------------------------------" << std::endl << std::endl;
}
}  // namespace ocpbenchmarker

}  // namespace idocp_b200

#endif  // IDOCP_B200_HPP_
