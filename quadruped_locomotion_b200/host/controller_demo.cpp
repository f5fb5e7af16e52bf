// controller_demo.cpp - a short trot of one robot through RosBalanceController (qlb_adapter.hpp): init, starting, then
// one update(time, period) per 2.5 ms tick.  LF+RH and RF+LH alternate every 8 ticks; the swing feet touch down early
// in the last quarter of some swings, and one stance foot loses contact for two ticks.
// Prints one JSON object for the run (gains), then one per tick with its inputs and the command, flags and forces, so
// that tests/test_controller.py can replay the ticks through the numpy restatement.
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <memory>

#include "qlb_adapter.hpp"

using namespace qlb_host;

static void print_array(const char* name, const double* v, int n) {
  std::printf(", \"%s\": [", name);
  for (int i = 0; i < n; i++) std::printf("%s%.17g", i ? ", " : "", v[i]);
  std::printf("]");
}

int main(int argc, char** argv) {
  const int ticks = argc > 1 ? std::atoi(argv[1]) : 40;
  try {
    auto device = std::make_shared<Device>(QLB_MODEL_QUADRUPED_MODEL, 0);
    auto state = std::make_shared<State>();
    RosBalanceController ctrl(device, state);
    const Vector3 kp{{300.0, 250.0, 400.0}}, kd{{10.0, 12.0, 8.0}};
    for (int i = 0; i < 3; i++) { ctrl.params().swing.kp[i] = kp[i]; ctrl.params().swing.kd[i] = kd[i]; }
    if (!ctrl.init() || !ctrl.starting()) return 3;
    const double period = ctrl.params().period;
    std::printf("{\"period\": %.17g, \"effort_limit\": %.17g", period, ctrl.params().effort_limit);
    print_array("kp", kp.data(), 3);
    print_array("kd", kd.data(), 3);
    std::printf("}\n");
    const double q0[12] = {0, 0.7, -1.4, 0, -0.7, 1.4, 0, 0.7, -1.4, 0, -0.7, 1.4};
    for (int k = 0; k < ticks; k++) {
      const double t = k * period;
      const int half = (k / 8) % 2;            // 0: LF+RH in stance, 1: RF+LH
      const double ph = (k % 8) / 8.0;
      JointPositions q;
      JointEfforts qd;
      for (int j = 0; j < 12; j++) {
        const double w = 2.0 * M_PI * (1.5 + 0.1 * j);
        q[j] = q0[j] + 0.05 * std::sin(w * t + j);
        qd[j] = 0.05 * w * std::cos(w * t + j);
      }
      state->setCurrentLimbJoints(q);
      ctrl.setJointVelocities(qd);
      const double z = 0.45 + 0.004 * std::sin(2.0 * M_PI * 2.5 * t);
      const double yaw = 0.02 * std::sin(2.0 * M_PI * 1.0 * t);
      state->setPoseBaseToWorld({{0.1 * t, 0.0, z}}, {{std::cos(0.5 * yaw), 0.0, 0.0, std::sin(0.5 * yaw)}});
      state->setBaseStateFromFeedback({{0.1, 0.0, 0.004 * 2.0 * M_PI * 2.5 * std::cos(2.0 * M_PI * 2.5 * t)}}, {{0.0, 0.0, 0.01}});
      state->setTargetPoseBaseToWorld({{0.1 * t + 0.002, 0.0, 0.45}}, {{1, 0, 0, 0}});
      state->setTargetBaseTwist({{0.1, 0.0, 0.0}}, {{0.0, 0.0, 0.0}});
      double phase[4], ptarget[12], vtarget[12];
      uint8_t desired = 0, contact = 0;
      for (int l = 0; l < 4; l++) {
        const bool stance = ((l == 0 || l == 2) ? 0 : 1) == half;
        bool touch = stance;
        if (!stance && ph >= 0.75 && (k / 16) % 2 == 0) touch = true;   // early touchdown
        if (stance && l == 1 && (k == 20 || k == 21)) touch = false;   // lost contact
        phase[l] = ph;
        desired |= stance ? (1u << l) : 0u;
        contact |= touch ? (1u << l) : 0u;
        ctrl.setLimbInput(static_cast<LimbEnum>(l), stance, true, touch, ph);
        const double sx = (l == 0 || l == 1) ? 0.42 : -0.42, sy = (l == 0 || l == 3) ? 0.15 : -0.15;
        for (int a = 0; a < 3; a++) vtarget[3 * l + a] = 0.0;
        ptarget[3 * l] = sx + 0.03 * (ph - 0.5); ptarget[3 * l + 1] = sy; ptarget[3 * l + 2] = -0.40 + 0.06 * std::sin(M_PI * ph);
        vtarget[3 * l] = 0.03 / (8 * period); vtarget[3 * l + 2] = 0.06 * M_PI * std::cos(M_PI * ph) / (8 * period);
        ctrl.setSwingTarget(static_cast<LimbEnum>(l), {{ptarget[3 * l], ptarget[3 * l + 1], ptarget[3 * l + 2]}},
                            {{vtarget[3 * l], vtarget[3 * l + 1], vtarget[3 * l + 2]}});
      }
      if (!ctrl.update(t, period)) return 4;
      double pose[7], twist[6], tpose[7], ttwist[6], grf[12];
      for (int a = 0; a < 3; a++) {
        pose[a] = state->getPositionWorldToBaseInWorldFrame()[a]; tpose[a] = state->getTargetPositionWorldToBaseInWorldFrame()[a];
        twist[a] = state->getLinearVelocityBaseInWorldFrame()[a]; twist[3 + a] = state->getAngularVelocityBaseInBaseFrame()[a];
        ttwist[a] = state->getTargetLinearVelocityBaseInWorldFrame()[a]; ttwist[3 + a] = state->getTargetAngularVelocityBaseInBaseFrame()[a];
      }
      for (int i = 0; i < 4; i++) { pose[3 + i] = state->getOrientationBaseToWorld()[i]; tpose[3 + i] = state->getTargetOrientationBaseToWorld()[i]; }
      for (int l = 0; l < 4; l++)
        for (int a = 0; a < 3; a++) grf[3 * l + a] = ctrl.getGroundReactionForce(static_cast<LimbEnum>(l))[a];
      std::printf("{\"tick\": %d, \"desired\": %u, \"contact\": %u, \"flags\": %u", k, (unsigned)desired, (unsigned)contact,
                  (unsigned)ctrl.getFlags());
      print_array("q", q.data(), 12);
      print_array("qd", qd.data(), 12);
      print_array("pose", pose, 7);
      print_array("twist", twist, 6);
      print_array("tpose", tpose, 7);
      print_array("ttwist", ttwist, 6);
      print_array("phase", phase, 4);
      print_array("ptarget", ptarget, 12);
      print_array("vtarget", vtarget, 12);
      print_array("command", ctrl.getCommand().data(), 12);
      print_array("grf", grf, 12);
      std::printf("}\n");
    }
  } catch (const std::exception& e) {
    std::fprintf(stderr, "error: %s\n", e.what());
    return 1;
  }
  return 0;
}
