// qlb_adapter.hpp - C++ host-side mirror of the reference's balance_controller math classes on top of
// the C ABI (include/qlb.h).  A batch of 1 through these classes reproduces one controller tick.
//
// What it mirrors (same method names, argument meaning and bool-return error convention):
//   balance_controller::ContactForceDistributionBase / ContactForceDistribution
//       (balance_controller/include/balance_controller/contact_force_distribution/
//        ContactForceDistributionBase.hpp:60-159, ContactForceDistribution.hpp:73-200)
//   balance_controller::MotionControllerBase / VirtualModelController
//       (.../motion_control/MotionControllerBase.hpp:58-123, VirtualModelController.cpp:89-102)
//   the slice of free_gait::State the path reads and writes
//       (free_gait_core/src/executor/State.cpp:59-67,93-101,227-235; quadruped_state.cpp:108-120,202-215,334-354)
//
// The reference's argument types are kindr/Eigen wrappers (Force, Torque, Position, RotationQuaternion,
// JointPositions ...).  Neither library is available in this build environment, so the adapter uses the
// plain 3-/4-/12-vectors below; in the reference tree they are replaced by `toImplementation()` views
// of the kindr types (see INTEGRATION.md).
#pragma once

#include <array>
#include <map>
#include <memory>
#include <utility>
#include <vector>
#include <stdexcept>
#include <string>

#include "qlb.h"
#include "qlb_models.h"

namespace qlb_host {

using Vector3 = std::array<double, 3>;
using Force = Vector3;
using Torque = Vector3;
using Position = Vector3;
using LinearVelocity = Vector3;
using LocalAngularVelocity = Vector3;
using Quaternion = std::array<double, 4>;       // (w, x, y, z), base -> world, like kindr RotationQuaternion
using JointPositions = std::array<double, 12>;  // LF, RF, RH, LH x (HAA, HFE, KFE)
using JointEfforts = std::array<double, 12>;
using JointEffortsLeg = Vector3;

// quadruped_model::QuadrupedDescription::LimbEnum (QuadrupedModel.hpp:47-53)
enum class LimbEnum : int { LF_LEG = 0, RF_LEG = 1, RH_LEG = 2, LH_LEG = 3 };

// The part of free_gait::State / quadruped_model::QuadrupedState that the hot path touches.  Unlike the
// reference (class-static members, quadruped_state.h:99-109) every instance owns its data.
class State {
 public:
  State() {
    support_.fill(true);
    for (auto& n : normals_) n = {0.0, 0.0, 1.0};
    efforts_.fill(0.0);
    joints_.fill(0.0);
  }
  // State.cpp:59-67
  bool isSupportLeg(LimbEnum limb) const { return support_[static_cast<int>(limb)]; }
  void setSupportLeg(LimbEnum limb, bool v) { support_[static_cast<int>(limb)] = v; }
  // State.cpp:93-101
  const Vector3& getSurfaceNormal(LimbEnum limb) const { return normals_[static_cast<int>(limb)]; }
  void setSurfaceNormal(LimbEnum limb, const Vector3& n) { normals_[static_cast<int>(limb)] = n; }
  // State.cpp:227-235
  void setJointEffortsForLimb(LimbEnum limb, const JointEffortsLeg& e) {
    for (int j = 0; j < 3; j++) efforts_[3 * static_cast<int>(limb) + j] = e[j];
  }
  const JointEfforts& getAllJointEfforts() const { return efforts_; }
  // quadruped_state.cpp:334-354 (the reference also caches FK here; ours is computed on the GPU)
  void setCurrentLimbJoints(const JointPositions& q) { joints_ = q; }
  const JointPositions& getJointPositionFeedback() const { return joints_; }
  // quadruped_state.cpp:108-120
  void setPoseBaseToWorld(const Position& p, const Quaternion& q) { position_ = p; orientation_ = q; }
  void setBaseStateFromFeedback(const LinearVelocity& v, const LocalAngularVelocity& w) { lin_vel_ = v; ang_vel_ = w; }
  const Position& getPositionWorldToBaseInWorldFrame() const { return position_; }
  const Quaternion& getOrientationBaseToWorld() const { return orientation_; }
  const LinearVelocity& getLinearVelocityBaseInWorldFrame() const { return lin_vel_; }
  const LocalAngularVelocity& getAngularVelocityBaseInBaseFrame() const { return ang_vel_; }
  // quadruped_state.cpp:202-215,258-267
  void setTargetPoseBaseToWorld(const Position& p, const Quaternion& q) { t_position_ = p; t_orientation_ = q; }
  void setTargetBaseTwist(const LinearVelocity& v, const LocalAngularVelocity& w) { t_lin_vel_ = v; t_ang_vel_ = w; }
  const Position& getTargetPositionWorldToBaseInWorldFrame() const { return t_position_; }
  const Quaternion& getTargetOrientationBaseToWorld() const { return t_orientation_; }
  const LinearVelocity& getTargetLinearVelocityBaseInWorldFrame() const { return t_lin_vel_; }
  const LocalAngularVelocity& getTargetAngularVelocityBaseInBaseFrame() const { return t_ang_vel_; }

 private:
  std::array<bool, 4> support_;
  std::array<Vector3, 4> normals_;
  JointEfforts efforts_;
  JointPositions joints_;
  Position position_{{0, 0, 0}}, t_position_{{0, 0, 0}};
  Quaternion orientation_{{1, 0, 0, 0}}, t_orientation_{{1, 0, 0, 0}};
  LinearVelocity lin_vel_{{0, 0, 0}}, t_lin_vel_{{0, 0, 0}};
  LocalAngularVelocity ang_vel_{{0, 0, 0}}, t_ang_vel_{{0, 0, 0}};
};

// Stand-in for the ROS parameter server behind ros::NodeHandle::hasParam / getParam, which the reference's
// loadParameters() functions query key by key (ContactForceDistribution.cpp:818-886, VirtualModelController.cpp:
// 429-548).  Keys are the reference's parameter paths; loadYaml() takes the text of a file laid out like
// balance_controller/config/controller_gains.yaml.
class ParameterServer {
 public:
  bool hasParam(const std::string& key) const { return values_.count(key) != 0; }
  bool getParam(const std::string& key, double& value) const {
    auto it = values_.find(key);
    if (it == values_.end()) return false;
    value = it->second;
    return true;
  }
  void setParam(const std::string& key, double value) { values_[key] = value; }
  void deleteParam(const std::string& key) { values_.erase(key); }
  void clear() { values_.clear(); }
  // every `a: {b: {c: number}}` leaf of the text becomes "/a/b/c"
  void loadYaml(const std::string& text) {
    std::vector<std::pair<int, std::string>> stack;
    size_t pos = 0;
    while (pos <= text.size()) {
      size_t eol = text.find('\n', pos);
      if (eol == std::string::npos) eol = text.size();
      std::string line = text.substr(pos, eol - pos);
      pos = eol + 1;
      const size_t hash = line.find('#');
      if (hash != std::string::npos) line.erase(hash);
      while (!line.empty() && (line.back() == ' ' || line.back() == '\r' || line.back() == '\t')) line.pop_back();
      size_t indent = 0;
      while (indent < line.size() && line[indent] == ' ') indent++;
      const size_t colon = line.find(':', indent);
      if (line.size() == indent || colon == std::string::npos) continue;
      while (!stack.empty() && stack.back().first >= (int)indent) stack.pop_back();
      const std::string key = (stack.empty() ? std::string() : stack.back().second) + "/" + line.substr(indent, colon - indent);
      size_t v = colon + 1;
      while (v < line.size() && line[v] == ' ') v++;
      if (v >= line.size()) { stack.emplace_back((int)indent, key); continue; }
      try { values_[key] = std::stod(line.substr(v)); } catch (...) {}
    }
  }

 private:
  std::map<std::string, double> values_;
};

// Shared owner of one qlb_context (one GPU).  The reference constructs ContactForceDistribution and
// VirtualModelController around one shared free_gait::State (ros_balance_controller.cpp:73-74); here
// they additionally share the device context.
class Device {
 public:
  explicit Device(const qlb_leg_model* legs = QLB_MODEL_QUADRUPED_MODEL, int device = 0) {
    qlb_default_params(&params_);
    const int rc = qlb_create(&ctx_, legs, &params_, device, 1);
    if (rc != QLB_OK) throw std::runtime_error(std::string("qlb_create: ") + qlb_strerror(rc));
    // the parameter server starts with the values of the reference's controller_gains.yaml (the library defaults),
    // as after `rosparam load`; parameters().clear() gives an empty server
    for (int k = 0; k < qlb_params_num_keys(); k++) {
      double v = 0.0;
      if (qlb_params_get_key(&params_, qlb_params_key(k), &v) >= 0) server_.setParam(qlb_params_key(k), v);
    }
  }
  ~Device() { qlb_destroy(ctx_); }
  Device(const Device&) = delete;
  Device& operator=(const Device&) = delete;
  qlb_context* ctx() { return ctx_; }
  qlb_params& params() { return params_; }
  ParameterServer& parameters() { return server_; }
  bool commit() { return qlb_set_params(ctx_, &params_) == QLB_OK; }
  // getParam for a list of keys, as the reference's loadParameters() does: false as soon as one is missing
  bool loadKeys(const char* prefix) {
    for (int k = 0; k < qlb_params_num_keys(); k++) {
      const std::string key = qlb_params_key(k);
      if (key.compare(0, std::string(prefix).size(), prefix) != 0) continue;
      double v = 0.0;
      if (!server_.getParam(key, v)) { missing_ = key; return false; }
      qlb_params_set_key(&params_, key.c_str(), v);
    }
    return true;
  }
  const std::string& missingParameter() const { return missing_; }

 private:
  qlb_context* ctx_ = nullptr;
  qlb_params params_;
  ParameterServer server_;
  std::string missing_;
};

class ContactForceDistributionBase {
 public:
  virtual ~ContactForceDistributionBase() = default;
  virtual bool loadParameters() = 0;
  virtual bool computeForceDistribution(const Force& virtualForceInBaseFrame, const Torque& virtualTorqueInBaseFrame) = 0;
  virtual bool getNetForceAndTorqueOnBase(Force& netForce, Torque& netTorque) = 0;
};

class ContactForceDistribution : public ContactForceDistributionBase {
 public:
  // ContactForceDistribution.hpp:73-89
  struct LegInfo {
    bool isPartOfForceDistribution_ = false;
    bool isLoadConstraintActive_ = false;
    int indexInStanceLegList_ = 0;
    int startIndexInVectorX_ = 0;
    Force desiredContactForce_{{0, 0, 0}};
    double frictionCoefficient_ = 0.6;
    unsigned activeRows_ = 0;  // extension: 5 active-set bits of this leg (include/qlb.h flags word)
  };

  ContactForceDistribution(std::shared_ptr<Device> device, std::shared_ptr<State> robot_state)
      : device_(std::move(device)), robot_state_(std::move(robot_state)) {
    for (int l = 0; l < 4; l++) legInfos_[static_cast<LimbEnum>(l)] = LegInfo();
  }

  // ContactForceDistribution::loadParameters (ContactForceDistribution.cpp:818-886): the nine keys under
  // /balance_controller/contact_force_distribution are read from the parameter server; a missing key makes it fail
  // (isParametersLoaded_ stays false and computeForceDistribution refuses to run), like the reference.
  bool loadParameters() override {
    isParametersLoaded_ = false;
    if (!device_->loadKeys("/balance_controller/contact_force_distribution/")) return false;
    for (auto& kv : legInfos_) kv.second.frictionCoefficient_ = device_->params().friction_default;
    isParametersLoaded_ = device_->commit();
    return isParametersLoaded_;
  }
  // the setters stand in for `rosparam set`: they write the parameter server, loadParameters() picks the values up
  void setVirtualForceWeights(const std::array<double, 6>& w) {
    static const char* const names[6] = {"force/heading", "force/lateral", "force/vertical", "torque/roll", "torque/pitch", "torque/yaw"};
    for (int i = 0; i < 6; i++) device_->parameters().setParam(std::string("/balance_controller/contact_force_distribution/weights/") + names[i], w[i]);
  }
  void setGroundForceWeight(double w) { device_->parameters().setParam("/balance_controller/contact_force_distribution/weights/regularizer/value", w); }
  void setMinimalNormalGroundForce(double f) { device_->parameters().setParam("/balance_controller/contact_force_distribution/constraints/minimal_normal_force", f); }
  void setFrictionCoefficient(double mu) { device_->parameters().setParam("/balance_controller/contact_force_distribution/constraints/friction_coefficient", mu); }
  double getGroundForceWeight() const { return device_->params().ground_force_weight; }
  double getMinimalNormalGroundForce() const { return device_->params().min_normal_force; }
  double getVirtualForceWeight(int index) const { return device_->params().wrench_weights[index]; }
  double getFrictionCoefficient(LimbEnum leg) const { return legInfos_.at(leg).frictionCoefficient_; }

  // ContactForceDistribution::computeForceDistribution (ContactForceDistribution.cpp:99-136)
  bool computeForceDistribution(const Force& F, const Torque& T) override {
    if (!isParametersLoaded_) return false;  // checkIfParametersLoaded
    isForceDistributionComputed_ = false;
    double q[12], quat[4], wrench[6], mu[4], normals[12];
    uint8_t mask = 0;
    const JointPositions& jq = robot_state_->getJointPositionFeedback();
    for (int i = 0; i < 12; i++) q[i] = jq[i];
    for (int i = 0; i < 4; i++) quat[i] = robot_state_->getOrientationBaseToWorld()[i];
    for (int i = 0; i < 3; i++) { wrench[i] = F[i]; wrench[3 + i] = T[i]; }
    mask = prepareLegLoading();
    for (int l = 0; l < 4; l++) {
      const LimbEnum limb = static_cast<LimbEnum>(l);
      mu[l] = legInfos_[limb].frictionCoefficient_;
      for (int a = 0; a < 3; a++) normals[3 * l + a] = robot_state_->getSurfaceNormal(limb)[a];
    }
    double grf[12], tau[12], net[6];
    uint32_t flags = 0;
    const int rc = qlb_solve_wrench_host(device_->ctx(), 1, q, quat, wrench, &mask, mu, normals, grf, tau, &flags, net);
    if (rc != QLB_OK) return false;
    return applyResult(grf, tau, net, flags);
  }

  // prepareLegLoading + resetOptimization for the current stance flags (CFD.cpp:138-166,580-596); returns the mask
  uint8_t prepareLegLoading() {
    uint8_t mask = 0;
    int nstance = 0;
    isForceDistributionComputed_ = false;
    for (int l = 0; l < 4; l++) {
      const LimbEnum limb = static_cast<LimbEnum>(l);
      LegInfo& info = legInfos_[limb];
      const bool stance = robot_state_->isSupportLeg(limb);
      info.isPartOfForceDistribution_ = stance;
      info.isLoadConstraintActive_ = stance;
      info.indexInStanceLegList_ = stance ? nstance : 0;
      info.startIndexInVectorX_ = 3 * info.indexInStanceLegList_;
      info.desiredContactForce_ = {0, 0, 0};
      info.activeRows_ = 0;
      if (stance) { mask |= (1u << l); nstance++; }
    }
    return mask;
  }

  // What a solve leaves behind in the reference: LegInfo forces, joint efforts in the shared State, the net wrench
  // and the computed flag (CFD.cpp:496-514,516-578,614-625).  Also used by VirtualModelController::compute, whose
  // reference version calls computeForceDistribution itself (VMC.cpp:99).
  bool applyResult(const double* grf, const double* tau, const double* net, uint32_t flags) {
    const unsigned status = (flags & QLB_FLAG_STATUS_MASK) >> QLB_FLAG_STATUS_SHIFT;
    lastFlags_ = flags;
    // the reference returns false (and keeps stale efforts) when the solver fails (CFD.cpp:490-494)
    if (status != QLB_STATE_OK && status != QLB_STATE_NO_STANCE) return false;
    for (int l = 0; l < 4; l++) {
      const LimbEnum limb = static_cast<LimbEnum>(l);
      LegInfo& info = legInfos_[limb];
      info.activeRows_ = (flags >> (QLB_FLAG_ACTIVE_SHIFT + 5 * l)) & 31u;
      if (!info.isPartOfForceDistribution_) continue;  // swing legs: efforts untouched (CFD.cpp:530)
      info.desiredContactForce_ = {-grf[3 * l], -grf[3 * l + 1], -grf[3 * l + 2]};  // CFD.cpp:502-503
      robot_state_->setJointEffortsForLimb(limb, {tau[3 * l], tau[3 * l + 1], tau[3 * l + 2]});
    }
    for (int a = 0; a < 3; a++) { netForce_[a] = net[a]; netTorque_[a] = net[3 + a]; }
    isForceDistributionComputed_ = true;
    return true;
  }

  // ContactForceDistribution::getNetForceAndTorqueOnBase (ContactForceDistribution.cpp:614-625)
  bool getNetForceAndTorqueOnBase(Force& netForce, Torque& netTorque) override {
    if (!isForceDistributionComputed_) return false;
    netForce = netForce_;
    netTorque = netTorque_;
    return true;
  }
  const LegInfo& getLegInfo(LimbEnum leg) const { return legInfos_.at(leg); }  // ContactForceDistribution.hpp:150
  uint32_t getLastFlags() const { return lastFlags_; }

  std::map<LimbEnum, LegInfo> legInfos_;  // public in the reference too (ContactForceDistribution.hpp:200)

 private:
  std::shared_ptr<Device> device_;
  std::shared_ptr<State> robot_state_;
  bool isParametersLoaded_ = false, isForceDistributionComputed_ = false;
  Force netForce_{{0, 0, 0}};
  Torque netTorque_{{0, 0, 0}};
  uint32_t lastFlags_ = 0;
};

class MotionControllerBase {
 public:
  virtual ~MotionControllerBase() = default;
  virtual bool loadParameters() = 0;
  virtual bool compute() = 0;  // MotionControllerBase.hpp:94
};

// VirtualModelController::compute (VirtualModelController.cpp:89-102): errors, gravity compensation,
// virtual force / torque and the contact force distribution run in the same fused kernels (qlb_solve_state).
class VirtualModelController : public MotionControllerBase {
 public:
  VirtualModelController(std::shared_ptr<Device> device, std::shared_ptr<State> robot_state,
                         std::shared_ptr<ContactForceDistribution> cfd)
      : device_(std::move(device)), robot_state_(std::move(robot_state)), cfd_(std::move(cfd)) {}

  // VirtualModelController::loadParameters (VMC.cpp:429-548): the eighteen gains under /balance_controller/virtual_model_controller
  bool loadParameters() override {
    loaded_ = false;
    if (!device_->loadKeys("/balance_controller/virtual_model_controller/")) return false;
    loaded_ = device_->commit();
    return loaded_;
  }
  void setProportionalGainTranslation(const Vector3& k) { setGains("kp", {"heading", "lateral", "vertical"}, k); }
  void setDerivativeGainTranslation(const Vector3& k) { setGains("kd", {"heading", "lateral", "vertical"}, k); }
  void setFeedforwardGainTranslation(const Vector3& k) { setGains("kff", {"heading", "lateral", "vertical"}, k); }
  void setProportionalGainRotation(const Vector3& k) { setGains("kp", {"roll", "pitch", "yaw"}, k); }
  void setDerivativeGainRotation(const Vector3& k) { setGains("kd", {"roll", "pitch", "yaw"}, k); }
  void setFeedforwardGainRotation(const Vector3& k) { setGains("kff", {"roll", "pitch", "yaw"}, k); }
  void setGravityCompensationForcePercentage(double p) { device_->params().gravity_compensation_percentage = p; }  // VMC.cpp:655

  bool compute() override {
    if (!loaded_) return false;  // isParametersLoaded
    const State& s = *robot_state_;
    double q[12], pose[7], twist[6], tpose[7], ttwist[6], mu[4], normals[12];
    uint8_t mask = 0;
    for (int i = 0; i < 12; i++) q[i] = s.getJointPositionFeedback()[i];
    for (int a = 0; a < 3; a++) {
      pose[a] = s.getPositionWorldToBaseInWorldFrame()[a]; tpose[a] = s.getTargetPositionWorldToBaseInWorldFrame()[a];
      twist[a] = s.getLinearVelocityBaseInWorldFrame()[a]; twist[3 + a] = s.getAngularVelocityBaseInBaseFrame()[a];
      ttwist[a] = s.getTargetLinearVelocityBaseInWorldFrame()[a]; ttwist[3 + a] = s.getTargetAngularVelocityBaseInBaseFrame()[a];
    }
    for (int i = 0; i < 4; i++) { pose[3 + i] = s.getOrientationBaseToWorld()[i]; tpose[3 + i] = s.getTargetOrientationBaseToWorld()[i]; }
    mask = cfd_->prepareLegLoading();   // also resets the distribution's state before anything can fail
    for (int l = 0; l < 4; l++) {
      const LimbEnum limb = static_cast<LimbEnum>(l);
      mu[l] = cfd_->getFrictionCoefficient(limb);
      for (int a = 0; a < 3; a++) normals[3 * l + a] = s.getSurfaceNormal(limb)[a];
    }
    double grf[12], tau[12], net[6], wrench[6];
    uint32_t flags = 0;
    const int rc = qlb_solve_state_host(device_->ctx(), 1, q, pose, twist, tpose, ttwist, &mask, mu, normals, grf, tau,
                                        &flags, net, wrench);
    if (rc != QLB_OK) return false;
    for (int a = 0; a < 3; a++) { virtualForceInBaseFrame_[a] = wrench[a]; virtualTorqueInBaseFrame_[a] = wrench[3 + a]; }
    // the reference's compute() ends in contactForceDistribution_->computeForceDistribution(F, T) (VMC.cpp:99): the
    // shared distribution object sees the result exactly as if it had been called
    return cfd_->applyResult(grf, tau, net, flags);
  }
  // VMC.cpp:288-300: what the distribution actually achieved
  bool getDistributedVirtualForceAndTorqueInBaseFrame(Force& netForce, Torque& netTorque) const {
    return cfd_->getNetForceAndTorqueOnBase(netForce, netTorque);
  }
  void setGains(const char* gain, const std::array<const char*, 3>& axes, const Vector3& k) {   // `rosparam set`, see loadParameters
    for (int i = 0; i < 3; i++)
      device_->parameters().setParam(std::string("/balance_controller/virtual_model_controller/") + axes[i] + "/" + gain, k[i]);
  }
  const Force& getDesiredVirtualForceInBaseFrame() const { return virtualForceInBaseFrame_; }
  const Torque& getDesiredVirtualTorqueInBaseFrame() const { return virtualTorqueInBaseFrame_; }

 private:
  std::shared_ptr<Device> device_;
  std::shared_ptr<State> robot_state_;
  std::shared_ptr<ContactForceDistribution> cfd_;
  bool loaded_ = false;
  Force virtualForceInBaseFrame_{{0, 0, 0}};
  Torque virtualTorqueInBaseFrame_{{0, 0, 0}};
};

// ---------------------------------------------------------------- MyRobotSolver
// Swing-leg torque solver (single_leg_test/lib/model_test_header.cpp): limb inverse dynamics + Cartesian PD for
// one limb per update(), written into the shared State like RosBalanceController::update does for every leg that
// is not in stance (ros_balance_controller.cpp:472-603).  The reference differentiates queues of measured joint
// velocities itself (:421-457); here the caller hands in the joint velocity and acceleration it wants used.
class MyRobotSolver {
 public:
  MyRobotSolver(std::shared_ptr<Device> device, std::shared_ptr<State> state,
                const qlb_limb_dynamics* limbs = QLB_LIMB_DYNAMICS_QUADRUPED_MODEL)
      : device_(std::move(device)), robot_state_(std::move(state)), limbs_(limbs) {
    qlb_default_swing_params(&params_);
  }

  bool loadLimbModelFromURDF() {  // :224-247 - the tables were generated from those URDF files
    loaded_ = qlb_set_limb_dynamics(device_->ctx(), limbs_) == QLB_OK;
    return loaded_;
  }
  void setGains(const Vector3& kp, const Vector3& kd) {  // :347-351
    for (int i = 0; i < 3; i++) { params_.kp[i] = kp[i]; params_.kd[i] = kd[i]; }
  }
  void setDesiredPositionAndVelocity(LimbEnum limb, const Vector3& position, const Vector3& velocity) {  // :398-403
    const int l = static_cast<int>(limb);
    for (int i = 0; i < 3; i++) { ptarget_[3 * l + i] = position[i]; vtarget_[3 * l + i] = velocity[i]; }
  }
  void setJointVelocityAndAcceleration(LimbEnum limb, const Vector3& qd, const Vector3& qdd) {
    const int l = static_cast<int>(limb);
    for (int i = 0; i < 3; i++) { qd_[3 * l + i] = qd[i]; qdd_[3 * l + i] = qdd[i]; }
  }
  qlb_swing_params& params() { return params_; }

  bool update(LimbEnum limb) {  // :412-502
    if (!loaded_) return false;
    const JointPositions& jq = robot_state_->getJointPositionFeedback();
    double q[12], tau[12];
    for (int i = 0; i < 12; i++) q[i] = jq[i];
    if (qlb_swing_leg_torques_host(device_->ctx(), 1, q, qd_, qdd_, ptarget_, vtarget_, &params_, tau) != QLB_OK) return false;
    const int l = static_cast<int>(limb);
    tau_ = {{tau[3 * l], tau[3 * l + 1], tau[3 * l + 2]}};
    robot_state_->setJointEffortsForLimb(limb, tau_);
    return true;
  }
  const JointEffortsLeg& getVecTauAct() const { return tau_; }

 private:
  std::shared_ptr<Device> device_;
  std::shared_ptr<State> robot_state_;
  const qlb_limb_dynamics* limbs_;
  qlb_swing_params params_;
  double qd_[12] = {0}, qdd_[12] = {0}, ptarget_[12] = {0}, vtarget_[12] = {0};
  JointEffortsLeg tau_{{0, 0, 0}};
  bool loaded_ = false;
};

// ---------------------------------------------------------------- RosBalanceController
// The whole controller tick of one robot (ros_balance_controller.cpp:198-716 update, starting) over
// qlb_controller_update_host with B = 1: contact state machine, virtual model + force distribution for the stance legs,
// swing-leg dynamics with the joint-velocity history, stale efforts on a failed solve and the +-300 N m command clamp.
// Measured and desired base state, joint positions and surface normals come from the shared State; the per-leg plan and
// contact inputs, the joint velocities and the swing targets are set on the controller.  The joint efforts that survive
// between ticks stay on the device (qlb_controller_get_state); update() returns the clamped command.
class RosBalanceController {
 public:
  RosBalanceController(std::shared_ptr<Device> device, std::shared_ptr<State> state,
                       const qlb_limb_dynamics* limbs = QLB_LIMB_DYNAMICS_QUADRUPED_MODEL)
      : device_(std::move(device)), robot_state_(std::move(state)), limbs_(limbs) {
    qlb_default_tick_params(&params_);
    phase_.fill(0.0);
  }
  ~RosBalanceController() { qlb_controller_destroy(ctrl_); }
  RosBalanceController(const RosBalanceController&) = delete;
  RosBalanceController& operator=(const RosBalanceController&) = delete;

  qlb_tick_params& params() { return params_; }   // period, effort limit and swing gains; read by init()
  // ros_balance_controller.cpp init(): limb models and the controller state for one robot
  bool init() {
    if (ctrl_) return false;
    if (qlb_set_limb_dynamics(device_->ctx(), limbs_) != QLB_OK) return false;
    return qlb_controller_create(device_->ctx(), 1, &params_, &ctrl_) == QLB_OK;
  }
  // RosBalanceController::starting: limb states INIT, efforts zero, velocity history restarted
  bool starting() { return ctrl_ && qlb_controller_reset(ctrl_, nullptr, nullptr) == QLB_OK; }

  // limbs_desired_state_ / is_footstep_ / FootContacts.is_contact / st_phase, sw_phase of one leg
  void setLimbInput(LimbEnum limb, bool desired_stance, bool is_footstep, bool is_contact, double phase) {
    const int l = static_cast<int>(limb);
    const uint8_t bit = static_cast<uint8_t>(1u << l);
    desired_ = desired_stance ? (desired_ | bit) : (desired_ & ~bit);
    footstep_ = is_footstep ? (footstep_ | bit) : (footstep_ & ~bit);
    contact_ = is_contact ? (contact_ | bit) : (contact_ & ~bit);
    phase_[l] = phase;
  }
  void setJointVelocities(const JointEfforts& qd) { qd_ = qd; }   // measured joint velocities, LF..LH x 3
  void setSwingTarget(LimbEnum limb, const Position& position, const LinearVelocity& velocity) {   // base frame
    const int l = static_cast<int>(limb);
    for (int i = 0; i < 3; i++) { ptarget_[3 * l + i] = position[i]; vtarget_[3 * l + i] = velocity[i]; }
  }

  // RosBalanceController::update(time, period).  The period is fixed when the controller is created (the velocity
  // history spans ten of them): a different one is refused.
  bool update(double /*time*/, double period) {
    if (!ctrl_ || period != params_.period) return false;
    const State& s = *robot_state_;
    double q[12], qd[12], pose[7], twist[6], tpose[7], ttwist[6], normals[12], phase[4];
    for (int i = 0; i < 12; i++) { q[i] = s.getJointPositionFeedback()[i]; qd[i] = qd_[i]; }
    for (int a = 0; a < 3; a++) {
      pose[a] = s.getPositionWorldToBaseInWorldFrame()[a]; tpose[a] = s.getTargetPositionWorldToBaseInWorldFrame()[a];
      twist[a] = s.getLinearVelocityBaseInWorldFrame()[a]; twist[3 + a] = s.getAngularVelocityBaseInBaseFrame()[a];
      ttwist[a] = s.getTargetLinearVelocityBaseInWorldFrame()[a]; ttwist[3 + a] = s.getTargetAngularVelocityBaseInBaseFrame()[a];
    }
    for (int i = 0; i < 4; i++) { pose[3 + i] = s.getOrientationBaseToWorld()[i]; tpose[3 + i] = s.getTargetOrientationBaseToWorld()[i]; }
    for (int l = 0; l < 4; l++) {
      phase[l] = phase_[l];
      for (int a = 0; a < 3; a++) normals[3 * l + a] = s.getSurfaceNormal(static_cast<LimbEnum>(l))[a];
    }
    return qlb_controller_update_host(ctrl_, q, qd, pose, twist, tpose, ttwist, &desired_, &footstep_, &contact_, phase, nullptr,
                                      normals, ptarget_, vtarget_, command_.data(), &flags_, grf_) == QLB_OK;
  }
  const JointEfforts& getCommand() const { return command_; }   // clamped to +-effort_limit
  uint32_t getFlags() const { return flags_; }                  // result word of the tick's solve
  Force getGroundReactionForce(LimbEnum limb) const {
    const int l = static_cast<int>(limb);
    return {{grf_[3 * l], grf_[3 * l + 1], grf_[3 * l + 2]}};
  }

 private:
  std::shared_ptr<Device> device_;
  std::shared_ptr<State> robot_state_;
  const qlb_limb_dynamics* limbs_;
  qlb_tick_params params_;
  qlb_controller* ctrl_ = nullptr;
  uint8_t desired_ = 0xF, footstep_ = 0xF, contact_ = 0xF;
  std::array<double, 4> phase_;
  JointEfforts qd_{}, command_{};
  double ptarget_[12] = {0}, vtarget_[12] = {0}, grf_[12] = {0};
  uint32_t flags_ = 0;
};

}  // namespace qlb_host
