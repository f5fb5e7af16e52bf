/*
 * qlb.h - C ABI of the B200-native batched contact-force-distribution solver.
 *
 * One call solves B independent robot states.  For every state the library runs, fused in
 * sm_100a kernels that keep everything between the input state and the outputs on chip
 * (one persistent kernel per call - inputs staged by TMA, the states that need active-set rounds
 * parked in shared memory - plus a fallback kernel that normally finds nothing to do),
 * the hot path of the reference's balance_controller:
 *
 *   leg forward kinematics + foot Jacobians + gravity torques
 *        (reference: quadruped_model/src/quadrupedkinematics.cpp:143-278,485-552)
 *   -> assembly of the virtual-model contact-force QP
 *        (reference: balance_controller/src/contact_force_distribution/
 *                    ContactForceDistribution.cpp:138-336)
 *   -> its solution (reference: ...ContactForceDistribution.cpp:385-514, the call
 *        ooqpei::QuadraticProblemFormulation::solve at :490)
 *   -> joint torques tau = J^T(-x) + G(q)      (reference: ...:516-578)
 *   -> achieved net wrench A x                  (reference: ...:614-625)
 *
 * Plain pointers and sizes only; no C++ or torch types.  Every function returns
 * QLB_OK (0) or a negative qlb_status and never throws.  There is no CPU fallback:
 * if no CUDA device is usable the calls fail with QLB_ERR_CUDA.
 *
 * Conventions (all fixed by the reference):
 *   - legs and joints are ordered LF(0), RF(1), RH(2), LH(3); joint slot = 3*leg + j
 *     (reference: quadruped_model/include/quadruped_model/QuadrupedModel.hpp:47-53,97-109)
 *   - quaternions are (w, x, y, z), Hamilton, rotating base-frame coordinates into the
 *     world frame (reference: balance_controller/src/ros_controller/
 *     gazebo_state_hardware_interface.cpp:327-330; quadruped_state.cpp:127)
 *   - wrench = desired net force (3) and torque (3) on the base, in base frame
 *   - batch arrays are SoA, component-major / batch-minor: element (c, i) of an array
 *     with C components lives at ptr[c * B + i]
 */
#ifndef QLB_H
#define QLB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QLB_NUM_LEGS 4
#define QLB_NUM_JOINTS 12
#define QLB_ABI_VERSION 2

typedef enum qlb_status {
  QLB_OK = 0,
  QLB_ERR_INVALID_ARGUMENT = -1,
  QLB_ERR_CUDA = -2,
  QLB_ERR_BATCH_TOO_LARGE = -3,
  QLB_ERR_NOT_INITIALISED = -4,
  QLB_ERR_ALLOC = -5
} qlb_status;

/* One leg: base_link -> (joint1) link1 -> (joint2) link2 -> (joint3) link3 -> (fixed) foot link.
 * Row k of joint_xyz / joint_rpy is the URDF <origin xyz rpy> of joint k (k = 3: the fixed foot
 * joint); all revolute axes are the local z axis.  link_mass / link_com are the <inertial> mass and
 * origin xyz of the child link of joint k.  Replaces the KDL chains built in
 * quadrupedkinematics.cpp:54-108.  Ready-made tables: include/qlb_models.h. */
typedef struct qlb_leg_model {
  double joint_xyz[4][3];
  double joint_rpy[4][3];
  double link_mass[4];
  double link_com[4][3];
} qlb_leg_model;

/* Controller parameters; defaults (qlb_default_params) are the reference's
 * balance_controller/config/controller_gains.yaml:2-41 and quadruped_state.cpp:28-41,83-97. */
typedef struct qlb_params {
  double wrench_weights[6];   /* S: virtualForceWeights_ (heading, lateral, vertical, roll, pitch, yaw) */
  double ground_force_weight; /* W: groundForceWeight_ (1e-4) */
  double min_normal_force;    /* F_min: minimalNormalGroundForce_ (10 N).  A negative value acts as 0: with mu > 0 the
                                 friction rows already imply n.f >= 0 */
  double friction_default;    /* mu used where the per-leg mu array is NULL (0.6) */
  double gravity;             /* |g|, 9.8 (ContactForceDistribution.cpp:518) */
  /* virtual-model controller (VirtualModelController.cpp:104-268) */
  double kp_translation[3], kd_translation[3], kff_translation[3];
  double kp_rotation[3], kd_rotation[3], kff_rotation[3];
  double torso_mass;                   /* 27.0 */
  double leg_mass[QLB_NUM_LEGS];       /* 6.0 each */
  double leg_base_position[QLB_NUM_LEGS][3]; /* (+-0.42, +-0.075, 0) */
  double com_in_base[3];               /* (0,0,0) */
  double gravity_compensation_percentage; /* 1.0 */
  /* interior-point solver */
  double ipm_tolerance;       /* stop when complementarity gap and residuals <= tol * scale (1e-9) */
  int32_t ipm_max_iterations; /* 40 */
  int32_t reserved;
} qlb_params;

/* Per-state result word, written to flags[i].
 *   bits 0..3   contact bit per leg = leg was part of the force distribution
 *               (isPartOfForceDistribution_, ContactForceDistribution.cpp:147)
 *   bits 4..23  active-set bits, 5 per leg at bit 4 + 5*leg + r, rows r in the reference's
 *               order: 0 = n.f >= F_min (ContactForceDistribution.cpp:241-247),
 *               1 = (mu n + t1).f >= 0, 2 = (mu n - t1).f >= 0, 3 = (mu n + t2).f >= 0,
 *               4 = (mu n - t2).f >= 0 (:315-325); set when the row is tight at the optimum
 *               with a positive multiplier
 *   bits 24..26 status code (qlb_state_status)
 *   bits 27..31 iterations of the stage that finished the state (saturates at 31): active-set rounds, or
 *               interior-point iterations for a state that needed that fallback; 0 = the unconstrained minimiser
 */
#define QLB_FLAG_CONTACT_MASK 0x0000000Fu
#define QLB_FLAG_ACTIVE_SHIFT 4
#define QLB_FLAG_ACTIVE_MASK 0x00FFFFF0u
#define QLB_FLAG_STATUS_SHIFT 24
#define QLB_FLAG_STATUS_MASK 0x07000000u
#define QLB_FLAG_ITER_SHIFT 27
#define QLB_FLAG_PARITY_MASK 0x00FFFFFFu /* contact + active bits: what is compared with the oracle */

typedef enum qlb_state_status {
  QLB_STATE_OK = 0,            /* optimum found, KKT-verified active set */
  QLB_STATE_NO_STANCE = 1,     /* no leg in stance: nothing solved, outputs zero (CFD.cpp:127-132) */
  QLB_STATE_MAX_ITER = 2,      /* iteration limit hit; forces are the last iterate */
  QLB_STATE_UNVERIFIED = 3,    /* converged, but the active-set polish failed its KKT check.  Both come only from the
                                  interior point (the three-pass pipeline's second stage, the fused kernel's fallback),
                                  whose start and stopping rule keep absolute scales: with forces far below 1 N or
                                  weights far below the defaults it ends here more often (0.5 % of C3/C5 states at
                                  (S, W) or (wrench, F_min) scaled by 2^-26 / 2^-30, three-pass pipeline) */
  QLB_STATE_BAD_INPUT = 4,     /* NaN/Inf input, degenerate surface normal, a joint angle beyond 1e6 rad, or a base
                                  quaternion / stance-leg surface normal that is not a unit vector (|v|^2 off by more than
                                  1e-5; smaller deviations - FP32 rounding - are renormalised); outputs zero */
  QLB_STATE_INFEASIBLE = 5     /* a stance leg has a negative friction coefficient while F_min > 0: no force satisfies
                                  mu n.f >= |t.f| and n.f >= F_min; outputs zero (QuadProg++ returns +inf, QuadProg++.cc:340-344) */
} qlb_state_status;

/* Batch statistics (device-side reduction; all-reduced over ranks by the caller, sum / max as noted). */
typedef struct qlb_stats {
  double count;              /* sum: states */
  double count_status[5];    /* sum: per qlb_state_status */
  double sum_iterations;     /* sum */
  double sum_wrench_err;     /* sum of sqrt((Ax-b)' S (Ax-b)) */
  double active_hist[20];    /* sum: how often each (leg,row) was active */
  double count_infeasible;   /* sum: states with QLB_STATE_INFEASIBLE */
  double max_wrench_err;     /* max */
  double max_iterations;     /* max */
} qlb_stats;
#define QLB_STATS_NUM_SUM 29 /* leading doubles that all-reduce with SUM; the rest with MAX */
#define QLB_STATS_NUM 31

/* Parameters under the reference's own names.  `key` is the ROS parameter path that
 * ContactForceDistribution::loadParameters (ContactForceDistribution.cpp:818-886) and
 * VirtualModelController::loadParameters (VirtualModelController.cpp:429-548) read, e.g.
 * "/balance_controller/contact_force_distribution/weights/force/heading".  Returns the index of the key (>= 0) or
 * QLB_ERR_INVALID_ARGUMENT for a path that is none of the qlb_params_num_keys() known ones. */
int qlb_params_set_key(qlb_params* p, const char* key, double value);
int qlb_params_get_key(const qlb_params* p, const char* key, double* value);
int qlb_params_num_keys(void);
const char* qlb_params_key(int index);
/* Fill *p from the text of a parameter file in the layout of balance_controller/config/controller_gains.yaml:2-41
 * (nested mappings, `key: number` leaves; other entries are ignored).  Returns how many of the known keys were
 * found; *first_missing (NULL ok) = the first key the file lacks, or NULL when all are there - the reference's
 * loadParameters() refuses to run with a key missing. */
int qlb_params_from_yaml(qlb_params* p, const char* yaml_text, const char** first_missing);

typedef struct qlb_context qlb_context;

/* Fill *p with the reference's gains, weights and solver defaults. */
int qlb_default_params(qlb_params* p);

/* Create a solver context on CUDA device `device`; max_batch sizes the staging buffers that the
 * *_host entry points use (0 = grow on demand).  Replaces the construction of
 * ContactForceDistribution + QuadrupedKinematics (ros_balance_controller.cpp:73-74). */
int qlb_create(qlb_context** ctx, const qlb_leg_model legs[QLB_NUM_LEGS], const qlb_params* params,
               int device, size_t max_batch);
int qlb_destroy(qlb_context* ctx);
/* Replaces ContactForceDistribution::loadParameters / VirtualModelController::loadParameters
 * (ContactForceDistribution.cpp:818-886, VirtualModelController.cpp:429-548).  Accepted (else
 * QLB_ERR_INVALID_ARGUMENT, and the context keeps its parameters): W and every S_i in [1e-12, 1e12] with
 * S_i / W <= 1e11, |F_min| <= 1e9, finite gravity, friction_default >= 0, ipm_tolerance > 0, ipm_max_iterations >= 1.
 * The bound on S_i / W keeps the FP64 dual solve within ~1e-6 of the exact minimiser on every stance (qlb_api.cu). */
int qlb_set_params(qlb_context* ctx, const qlb_params* params);
int qlb_get_params(const qlb_context* ctx, qlb_params* params);

/* Wrench mode, DEVICE pointers, asynchronous on `stream` (a cudaStream_t, NULL = default stream).
 * Replaces ContactForceDistribution::computeForceDistribution(Force, Torque)
 * (ContactForceDistribution.cpp:99-136) for B states at once.
 *   in : q[12][B] joint positions; quat_wxyz[4][B]; wrench[6][B] (F then T, base frame);
 *        stance_mask[B] bit k = leg k is a support leg (State::isSupportLeg);
 *        mu[4][B] per-leg friction coefficient, or NULL -> params.friction_default;
 *        normals_world[12][B] per-leg surface normal (leg-major), or NULL -> (0,0,1)
 *   out: grf[12][B] ground-reaction forces x in base frame, zero for swing legs
 *        (the reference's desiredContactForce_ is -x, CFD.cpp:502-503);
 *        tau[12][B] joint torques J^T(-x) + G(q) for stance legs, zero for swing legs
 *        (the reference leaves swing slots unwritten, CFD.cpp:530);
 *        flags[B] result word (see above);
 *        netwrench[6][B] achieved A x (getNetForceAndTorqueOnBase), or NULL.
 * Calls of one context may be in flight on different streams at the same time (the context keeps eight
 * sets of work counters and index lists and orders a ninth call behind the first).  A context may be shared by
 * several host threads: every entry point holds the context's lock while it enqueues its work (the *_host entry
 * points until they return), so concurrent calls are serialised on the host and overlap on the device. */
int qlb_solve_wrench(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz,
                     const double* wrench, const uint8_t* stance_mask, const double* mu,
                     const double* normals_world, double* grf, double* tau, uint32_t* flags,
                     double* netwrench, void* stream);

/* Same, HOST pointers: copies in, solves, copies out, synchronises.  This is what a batch-of-1
 * controller tick calls.  Every *_host entry point synchronises all the streams it used before it returns, on
 * failure too, so no copy still reads or writes the caller's arrays. */
int qlb_solve_wrench_host(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz,
                          const double* wrench, const uint8_t* stance_mask, const double* mu,
                          const double* normals_world, double* grf, double* tau, uint32_t* flags,
                          double* netwrench);

/* State mode: the virtual-model-controller prologue (VirtualModelController::compute,
 * VirtualModelController.cpp:89-268) runs in the same kernel and produces the wrench.
 *   base_pose[7][B]  = position world->base (3) + quat_wxyz (4), feedback
 *   base_twist[6][B] = linear velocity in world (3) + angular velocity in base (3), feedback
 *   target_pose[7][B], target_twist[6][B] = the desired counterparts
 *   wrench_out[6][B] = the virtual force/torque that was distributed, or NULL */
int qlb_solve_state(qlb_context* ctx, size_t B, const double* q, const double* base_pose,
                    const double* base_twist, const double* target_pose, const double* target_twist,
                    const uint8_t* stance_mask, const double* mu, const double* normals_world,
                    double* grf, double* tau, uint32_t* flags, double* netwrench, double* wrench_out,
                    void* stream);
int qlb_solve_state_host(qlb_context* ctx, size_t B, const double* q, const double* base_pose,
                         const double* base_twist, const double* target_pose,
                         const double* target_twist, const uint8_t* stance_mask, const double* mu,
                         const double* normals_world, double* grf, double* tau, uint32_t* flags,
                         double* netwrench, double* wrench_out);

/* FP32 twins (SURVEY 8b "_f32 suffix", BASELINE config C4): the same entry points with float arrays -
 * half the HBM / PCIe bytes.  Two solver cores, chosen per context with qlb_set_f32_core:
 *   QLB_F32_CORE_FP64 (default): FP32 arrays and leg kinematics (sincos, chain product, Jacobian, gravity torques);
 *     the friction frame is built in FP64 from the FP32 quaternion and normal (renormalised) and the QP is solved in
 *     FP64.  The only error left is the rounding of inputs, kinematics and outputs.  STATED TOLERANCE: forces within
 *     5e-4 relative of the FP64 result (scale max(1,|f|_inf); measured 8e-5 on C3, 9e-7 on C2, 5e-6 on C5), torques
 *     within 1e-3 (measured 1.5e-4); status and contact bits exact; active-row bits exact on states whose active set
 *     is decided by a margin above 1e-3 (measured: exact on every test state).  Device-resident throughput as FP64
 *     (both kernels are bound by the FP64 solve), 1.55x end to end (half the PCIe bytes).
 *   QLB_F32_CORE_FP32: FP32 arithmetic throughout (the round-1 three-pass kernels: 6x6 systems with one step of
 *     iterative refinement, active-set rounds, interior point; states the FP32 core cannot verify are solved again by
 *     the FP64 core inside the same kernel, so every status is the FP64 one).  Kept for comparison: since round 2 it is
 *     both slower and less accurate than the default.  STATED TOLERANCE (tests/test_gpu_parity.py, measured on C2/C3):
 *     the QP Hessian has condition number ~1e5 (W = 1e-4 against S|a|^2 ~ 10), so the weakly determined internal-force
 *     directions carry errors of order cond * eps: relative force error median 2e-7 on full-rank stances and 2e-4 on
 *     two-leg stances, 99 % of states below 2e-2, worst observed 5e-2; the achieved wrench A x agrees to 1e-2, every
 *     constraint holds to 1e-4 of the force scale, the objective is within 1e-4 relative of the optimum; contact bits
 *     exact, active-row bits equal on >= 95 % of states.
 * Status values and layouts are unchanged. */
int qlb_solve_wrench_f32(qlb_context* ctx, size_t B, const float* q, const float* quat_wxyz,
                         const float* wrench, const uint8_t* stance_mask, const float* mu,
                         const float* normals_world, float* grf, float* tau, uint32_t* flags,
                         float* netwrench, void* stream);
int qlb_solve_wrench_f32_host(qlb_context* ctx, size_t B, const float* q, const float* quat_wxyz,
                              const float* wrench, const uint8_t* stance_mask, const float* mu,
                              const float* normals_world, float* grf, float* tau, uint32_t* flags,
                              float* netwrench);
int qlb_solve_state_f32(qlb_context* ctx, size_t B, const float* q, const float* base_pose,
                        const float* base_twist, const float* target_pose, const float* target_twist,
                        const uint8_t* stance_mask, const float* mu, const float* normals_world,
                        float* grf, float* tau, uint32_t* flags, float* netwrench, float* wrench_out,
                        void* stream);
int qlb_solve_state_f32_host(qlb_context* ctx, size_t B, const float* q, const float* base_pose,
                             const float* base_twist, const float* target_pose,
                             const float* target_twist, const uint8_t* stance_mask, const float* mu,
                             const float* normals_world, float* grf, float* tau, uint32_t* flags,
                             float* netwrench, float* wrench_out);

/* Kernel organisation of the solve entry points (the results are the same optimum either way):
 *   QLB_PIPELINE_FUSED (default): one persistent kernel - inputs staged through shared memory by the TMA unit,
 *     kinematics + QP data + unconstrained minimiser per state, the states that need active-set rounds parked in
 *     shared memory and solved by a dual block active-set method in the same kernel (every quad of a warp refills
 *     itself from the stash) - followed by the interior-point kernel for states the rounds could not verify
 *     (normally none).
 *   QLB_PIPELINE_THREE_PASS: the round-1 organisation (first / active-set / interior-point kernels over
 *     compacted index lists in HBM), kept for comparison.  Always used by the FP32 solver core. */
#define QLB_PIPELINE_FUSED 0
#define QLB_PIPELINE_THREE_PASS 1
int qlb_set_pipeline(qlb_context* ctx, int pipeline);

#define QLB_F32_CORE_FP32 0
#define QLB_F32_CORE_FP64 1
int qlb_set_f32_core(qlb_context* ctx, int core);

/* Kinematics only (DEVICE pointers): foot positions, translational Jacobians (row-major 3x3 per leg)
 * and gravity torques for all four legs.  Replaces QuadrupedKinematics::FowardKinematicsSolve /
 * AnalysticJacobian / getGravityCompensationForLimb (quadrupedkinematics.cpp:143-278,485-552).
 *   foot[12][B], jac[36][B] (slot = 9*leg + 3*row + col), gravity_tau[12][B]; any output may be NULL.
 *   quat_wxyz may be NULL (identity: gravity along -z of the base frame). */
int qlb_leg_kinematics(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz,
                       double* foot, double* jac, double* gravity_tau, void* stream);

/* One sample of the desired robot state as RosBalanceController::baseCommandCallback reads it from a
 * free_gait_msgs/RobotState message (ros_balance_controller.cpp:761-811: base_pose.pose.pose,
 * base_pose.twist.twist, {lf,rf,rh,lh}_leg_joints.position[0..2], {..}_leg_mode.support_leg and
 * .surface_normal.vector).  Fixed layout, 304 bytes, 16-byte aligned; a planner fills an array of these (one per
 * robot, or one per time sample of a planned motion, StateBatch.hpp / BatchExecutor.cpp:69-83). */
typedef struct qlb_robot_state_record {
  double base_position[3];          /* geometry_msgs/Point x, y, z (world) */
  double base_orientation_xyzw[4];  /* geometry_msgs/Quaternion field order x, y, z, w */
  double base_linear_velocity[3];   /* twist.linear, world frame */
  double base_angular_velocity[3];  /* twist.angular, base frame */
  double joint_position[12];        /* LF, RF, RH, LH x (HAA, HFE, KFE) */
  double surface_normal[12];        /* per leg, world frame */
  uint8_t support_leg[4];           /* LegMode.support_leg per leg */
  uint8_t reserved[4];
} qlb_robot_state_record;

/* records[B] (DEVICE, array of structs) -> the solver's SoA arrays (any output may be NULL):
 * q[12][B], base_pose[7][B] (position + quat w,x,y,z), base_twist[6][B], stance_mask[B], normals_world[12][B].
 * Byte movement only; bit-exact.  SURVEY 8f rank 1 ("RobotState message -> SoA packer"). */
int qlb_pack_robot_states(qlb_context* ctx, size_t B, const qlb_robot_state_record* records, double* q,
                          double* base_pose, double* base_twist, uint8_t* stance_mask,
                          double* normals_world, void* stream);

/* Foot positions in the WORLD frame for every state of a batch, feet_world[12][B] (leg-major):
 * position + R_bw * FK(q).  Replaces the per-state loop of StateBatchComputer::computeEndEffectorTrajectories
 * (free_gait_core/src/executor/StateBatchComputer.cpp:64-77).  DEVICE pointers. */
int qlb_feet_in_world(qlb_context* ctx, size_t B, const double* q, const double* base_pose,
                      double* feet_world, void* stream);

/* ---- preview of a planned motion (SURVEY 8f rank 2) --------------------------------------------------------
 * One sample of the preview: what StateBatchComputer::computeEndEffectorTrajectories collects
 * (free_gait_core/src/executor/StateBatchComputer.cpp:64-77) plus what the controller would command at that sample. */
typedef struct qlb_preview_record {
  double feet_world[12];   /* foot positions in the world frame, leg-major */
  double grf[12];          /* ground-reaction forces in base frame (zero for swing legs) */
  double tau[12];          /* joint torques of the stance legs */
  double netwrench[6];     /* achieved net wrench */
  double wrench[6];        /* the virtual wrench that was distributed (gravity compensation + feed-forward terms) */
  double friction_margin;  /* qlb_friction_margins */
  double min_normal_slack; /* min over stance legs of n.f - F_min */
  uint32_t flags;          /* result word of the solve */
  uint32_t reserved;
} qlb_preview_record;      /* 408 bytes */

/* The whole plan in one call, HOST pointers: records[B] = the states of a StateBatch (one per time sample, as
 * BatchExecutor::processInThread collects them at 10 ms steps, BatchExecutor.cpp:69-83) -> preview[B].
 * Each sample is taken as both feedback and target of the virtual model controller (perfect tracking), so the
 * distributed wrench is the controller's gravity compensation plus its feed-forward terms.  mu[4] = friction
 * coefficient per leg for every sample, or NULL -> params.friction_default.  Device work per chunk: record packer,
 * feet-in-world kernel, fused solve (state mode), friction-margin kernel, result packer.  Synchronises. */
int qlb_preview_plan_host(qlb_context* ctx, size_t B, const qlb_robot_state_record* records, const double mu[4],
                          qlb_preview_record* preview);

/* ---- swing-leg torques (SURVEY 8f rank 4) ----------------------------------------------------------
 * Rigid-body table of one limb: three bodies on z-axis revolute joints (the link behind the fixed foot
 * joint merged into the third), as a rigid-body-dynamics URDF reader builds it from the per-leg URDFs that
 * MyRobotSolver::loadLimbModelFromURDF loads (single_leg_test/lib/model_test_header.cpp:224-247). */
typedef struct qlb_limb_dynamics {
  double joint_xyz[3][3];     /* <origin xyz> of the three revolute joints */
  double joint_rpy[3][3];     /* <origin rpy> */
  double body_mass[3];
  double body_com[3][3];      /* centre of mass in the link frame */
  double body_inertia[3][6];  /* Ixx, Ixy, Ixz, Iyy, Iyz, Izz about the centre of mass, link axes */
} qlb_limb_dynamics;

typedef struct qlb_swing_params {
  double gravity[3];          /* in the base frame.  The reference never sets it on its limb models, so they run with
                                 the dynamics library's default (0, -9.81, 0) (model_test_header.cpp:36 vs :193) */
  double acceleration_scale;  /* the reference feeds 0.5 * qdd to the inverse dynamics (model_test_header.cpp:460) */
  double kp[3], kd[3];        /* Cartesian gains on the foot position / velocity error in the base frame (:497-498) */
} qlb_swing_params;

int qlb_default_swing_params(qlb_swing_params* p);                     /* the reference's values; kp = kd = 0 */
int qlb_set_limb_dynamics(qlb_context* ctx, const qlb_limb_dynamics legs[QLB_NUM_LEGS]);

/* MyRobotSolver::update for every leg of every state (model_test_header.cpp:412-502): inverse dynamics of the limb
 * (recursive Newton-Euler, fixed base) at (q, qd, acceleration_scale * qdd) plus the Cartesian PD term
 * J^T (kp .* (p* - p) + kd .* (v* - J qd)).  DEVICE pointers, SoA: q, qd, qdd[12][B]; foot_target_position,
 * foot_target_velocity[12][B] in the base frame (either may be NULL: that error term is zero); tau[12][B].
 * The caller keeps the rows of its swing legs (the stance rows come from qlb_solve_*). */
int qlb_swing_leg_torques(qlb_context* ctx, size_t B, const double* q, const double* qd, const double* qdd,
                          const double* foot_target_position, const double* foot_target_velocity,
                          const qlb_swing_params* params, double* tau, void* stream);
/* Same, HOST pointers: copies in, computes, copies out, synchronises (a batch-of-1 controller tick). */
int qlb_swing_leg_torques_host(qlb_context* ctx, size_t B, const double* q, const double* qd, const double* qdd,
                               const double* foot_target_position, const double* foot_target_velocity,
                               const qlb_swing_params* params, double* tau);

/* The same with the joint acceleration estimated the way the reference does it (model_test_header.cpp:421-429):
 * the caller keeps a queue of joint-velocity samples per leg; qd_back is its newest entry (also the velocity fed to
 * the dynamics), qd_front its oldest, and qdd = (qd_back - qd_front) / (10 * period).  DEVICE pointers. */
int qlb_swing_leg_torques_from_queue(qlb_context* ctx, size_t B, const double* q, const double* qd_back,
                                     const double* qd_front, double period, const double* foot_target_position,
                                     const double* foot_target_velocity, const qlb_swing_params* params,
                                     double* tau, void* stream);

/* ---- per-leg contact state machine (SURVEY 8f rank 4) ----------------------------------------------------
 * Limb states in the order of StateSwitcher::States (balance_controller/include/state_switcher/StateSwitcher.hpp:62-72). */
typedef enum qlb_limb_state {
  QLB_LIMB_INIT = 0,
  QLB_LIMB_STANCE_NORMAL = 1,
  QLB_LIMB_STANCE_SLIPPING = 2,
  QLB_LIMB_STANCE_LOST_CONTACT = 3,
  QLB_LIMB_SWING_NORMAL = 4,
  QLB_LIMB_SWING_LATE_LIFTOFF = 5,
  QLB_LIMB_SWING_EARLY_TOUCHDOWN = 6,
  QLB_LIMB_SWING_BUMPED_INTO_OBSTACLE = 7,
  QLB_LIMB_SWING_LATELY_TOUCHDOWN = 8
} qlb_limb_state;

/* RosBalanceController::footContactsCallback (ros_balance_controller.cpp:1086-1140) for B robots at once, plus the
 * support-leg decision update() takes from the limb state (:242-366: StanceNormal, SwingEarlyTouchDown and Init are
 * support legs).  DEVICE pointers.
 *   desired_stance_mask[B]  bit k = the plan has leg k in stance (limbs_desired_state_, :968-1080)
 *   footstep_mask[B]        bit k = is_footstep_ (contact supervision on); NULL = all legs
 *   contact_mask[B]         bit k = measured contact (sim_assiants/FootContacts.is_contact)
 *   phase[4][B]             phase in [0,1] of the leg's current stance or swing (st_phase / sw_phase)
 *   limb_state[4][B]        in: previous qlb_limb_state per leg, out: new one
 *   stance_mask[B]          out (NULL ok): the stance mask to hand to qlb_solve_* */
int qlb_contact_fsm(qlb_context* ctx, size_t B, const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                    const uint8_t* contact_mask, const double* phase, uint8_t* limb_state, uint8_t* stance_mask,
                    void* stream);

/* ---- the controller tick for B robots (RosBalanceController::update / starting) --------------------------------
 * One qlb_controller_update = one 2.5 ms tick of ros_balance_controller.cpp:198-716 for every robot of the batch:
 * contact state machine (as qlb_contact_fsm) -> state-mode solve of the stance legs (as qlb_solve_state) -> swing-leg
 * torques with the velocity-queue acceleration (as qlb_swing_leg_torques_from_queue) -> merge into the robot's joint
 * efforts -> clamped command.  The state that lives from tick to tick is kept on the device, per robot:
 *   limb_state[4][B]  qlb_limb_state per leg; QLB_LIMB_INIT after create / reset
 *   efforts[12][B]    the reference's State joint efforts: unclamped, zero after create / reset, never non-finite.
 *                     Stance rows take the solve's torques when its status is QLB_STATE_OK or QLB_STATE_NO_STANCE and
 *                     keep their previous value otherwise (stale efforts, RBC.cpp:418,455-458); swing rows take the
 *                     swing-leg torques unless one of the leg's three is non-finite, in which case the row is kept
 *   a ring of the last 11 joint-velocity samples qd: the newest is this tick's sample, the oldest the one 10 ticks
 *                     earlier, so the swing legs use qdd = (qd_newest - qd_oldest) / (10 period), the reference's
 *                     Time_derta divisor over a true 10-period span.  Start-up rule: the first tick after create or
 *                     reset fills all 11 samples of the robot with its qd, so that tick has qdd = 0; a non-finite qd
 *                     sample makes that robot's swing rows stale until it has left the ring (10 ticks).
 * A controller and its arrays belong to one context: destroy the controller before the context.  Updates of one
 * controller must be ordered (one stream, or the caller orders them); every update is ordered after the controller's
 * last reset, whatever stream that ran on; different controllers of one context may run on different streams at the
 * same time.  Every update launches the kernels of qlb_solve_state plus two.  After an update that returned an error the
 * robots' state is unspecified until they are reset. */
typedef struct qlb_tick_params {
  double period;           /* control period in s: 0.0025 (400 Hz, balance_controller_manager.cpp:48,70) */
  double effort_limit;     /* |command| clamp in N m: 300 (RBC.cpp:450-454); the stored efforts are not clamped */
  qlb_swing_params swing;  /* swing-leg gains and gravity, as qlb_default_swing_params */
} qlb_tick_params;         /* 96 bytes */
int qlb_default_tick_params(qlb_tick_params* p);

typedef struct qlb_controller qlb_controller;
/* Allocates the per-robot state for B robots on ctx's device (limb states INIT, efforts zero, rings marked for refill)
 * and synchronises.  The swing legs need the limb tables: qlb_set_limb_dynamics before the first update.
 * QLB_ERR_CUDA when no CUDA device is usable. */
int qlb_controller_create(qlb_context* ctx, size_t B, const qlb_tick_params* params, qlb_controller** out);
int qlb_controller_destroy(qlb_controller* c);
/* RosBalanceController::starting for the robots with reset_mask[i] != 0 (DEVICE [B]; NULL = all): limb states INIT,
 * efforts zero, ring refilled by the next sample.  Other robots are untouched.  Asynchronous on `stream`. */
int qlb_controller_reset(qlb_controller* c, const uint8_t* reset_mask, void* stream);
/* One tick for all B robots, DEVICE pointers, asynchronous on `stream`.
 *   q[12][B], qd[12][B]           measured joint positions and velocities
 *   base_pose .. target_twist     as qlb_solve_state
 *   desired_stance_mask, footstep_mask (NULL = all legs), contact_mask, phase[4][B]   as qlb_contact_fsm
 *   mu, normals_world             as qlb_solve_state (NULL ok)
 *   foot_target_position, foot_target_velocity   as qlb_swing_leg_torques (NULL ok: that error term is zero)
 *   command[12][B]                out: clamp(efforts, +-effort_limit)
 *   flags[B]                      out: result word of the solve
 *   grf[12][B]                    out (NULL ok): ground-reaction forces of the solve */
int qlb_controller_update(qlb_controller* c, const double* q, const double* qd, const double* base_pose,
                          const double* base_twist, const double* target_pose, const double* target_twist,
                          const uint8_t* desired_stance_mask, const uint8_t* footstep_mask, const uint8_t* contact_mask,
                          const double* phase, const double* mu, const double* normals_world,
                          const double* foot_target_position, const double* foot_target_velocity, double* command,
                          uint32_t* flags, double* grf, void* stream);
/* Same, HOST pointers: staged through the context's buffers, synchronises (a batch-of-1 controller tick). */
int qlb_controller_update_host(qlb_controller* c, const double* q, const double* qd, const double* base_pose,
                               const double* base_twist, const double* target_pose, const double* target_twist,
                               const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                               const uint8_t* contact_mask, const double* phase, const double* mu,
                               const double* normals_world, const double* foot_target_position,
                               const double* foot_target_velocity, double* command, uint32_t* flags, double* grf);
/* FP32 twins of the tick, for a caller that keeps its state in float: the same arguments, NULL rules, errors, ordering
 * and launches as above, with float arrays.  They act on the same controller, whose state stays FP64 (limb states,
 * efforts, the ring of qd samples: a float sample is stored exactly), so the FP64 and FP32 updates may be mixed from
 * tick to tick; qlb_controller_get_state is unchanged.
 *   contact state machine: the float phase is widened to double before the comparisons, so the limb states are those
 *     of the FP64 tick on the same values, bit for bit
 *   stance legs: qlb_solve_state_f32 (the solver core follows qlb_set_f32_core; the default FP64 core)
 *   swing legs: FP32 arithmetic on FP32 copies of the limb tables and the kinematic model; qdd differenced in FP32
 *     from the float sample and the oldest ring slot rounded to float (exact when only FP32 updates wrote it)
 *   command: the FP64 efforts clamped to +-effort_limit in double, then rounded to float
 * Stale rows, the clamp and the reset behave as in FP64.  One difference: FP32 overflows earlier, so a huge but finite
 * qd can make a swing row stale (non-finite FP32 torque) where the FP64 tick would not.
 * STATED TOLERANCE against the FP64 tick on the same values widened to double (tests/test_controller_f32.py, 40-tick
 * trot): limb states and the status and contact bits of flags exact; active-row bits equal on >= 99.9 % of robot-ticks;
 * stance rows of command and efforts within 1e-3 per robot (scale max(1, |x|_inf)), grf within 5e-4 (the bars of the
 * solve twin); swing rows within 1e-4.  Measured on one B200 (1000 W power limit, 4099 robots over 40 ticks): limb states,
 * status and contact bits exact; active-row bits equal on every robot-tick; stance rows 1.1e-4, grf 7.2e-5, swing rows
 * 4.4e-6.  Speed on the same card: 2^20 robots 1.52 ms per tick against 1.86 ms for the FP64 tick (DESIGN.md section 5). */
int qlb_controller_update_f32(qlb_controller* c, const float* q, const float* qd, const float* base_pose,
                              const float* base_twist, const float* target_pose, const float* target_twist,
                              const uint8_t* desired_stance_mask, const uint8_t* footstep_mask, const uint8_t* contact_mask,
                              const float* phase, const float* mu, const float* normals_world,
                              const float* foot_target_position, const float* foot_target_velocity, float* command,
                              uint32_t* flags, float* grf, void* stream);
int qlb_controller_update_f32_host(qlb_controller* c, const float* q, const float* qd, const float* base_pose,
                                   const float* base_twist, const float* target_pose, const float* target_twist,
                                   const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                                   const uint8_t* contact_mask, const float* phase, const float* mu,
                                   const float* normals_world, const float* foot_target_position,
                                   const float* foot_target_velocity, float* command, uint32_t* flags, float* grf);
/* DEVICE copies of the persistent state, asynchronous on `stream`: limb_state[4][B], efforts[12][B] (either NULL ok). */
int qlb_controller_get_state(const qlb_controller* c, uint8_t* limb_state, double* efforts, void* stream);

/* Friction margins of a solved batch (DEVICE pointers): margin[i] = min over stance legs and the four friction rows of
 * slack / (mu n.f) - 1 = unloaded tangentially, 0 = a friction row is active; min_normal[i] (NULL ok) = min over
 * stance legs of n.f - F_min.  What a preview of a planned motion reports next to forces and torques
 * (StateBatchComputer / BatchExecutor consumers, SURVEY 8f rank 2).  mu / normals_world as in qlb_solve_wrench. */
int qlb_friction_margins(qlb_context* ctx, size_t B, const double* grf, const double* quat_wxyz,
                         const uint8_t* stance_mask, const double* mu, const double* normals_world, double* margin,
                         double* min_normal, void* stream);

/* Generic small dense QP (DEVICE pointers), B problems of the same shape, in the argument convention of
 * the reference's in-repo backend quadprogpp::solve_quadprog (qp_solver/include/qp_solver/QuadProg++.h:
 * 8-30), which qp_solver::QuadraticProblemSolver::minimize forwards to
 * (qp_solver/src/quadraticproblemsolver.cpp:65-97):
 *     min 1/2 x'Gx + g0'x   s.t.   CE' x + ce0 = 0,   CI' x + ci0 >= 0
 * G[n*n][B], g0[n][B], CE[n*p][B] (element (i,j) of the n x p matrix at slot i*p+j), ce0[p][B],
 * CI[n*m][B], ci0[m][B]; n <= 12, m <= 24, p <= 12; CE/ce0 may be NULL when p == 0, CI/ci0 when m == 0.
 * An all-zero equality column is treated as absent (the reference's callers pass one).
 * Out: x[n][B]; cost[B] (NULL ok; +inf when infeasible); status[B]: 0 ok, 1 infeasible, 2 G not positive
 * definite or non-finite input, 3 iteration limit; active[B] (NULL ok): bit i = inequality i is in the
 * final working set.  One warp per problem: a dual active-set iteration on the Gram matrix of the whitened
 * constraint normals (csrc/qlb_qp_dense.cuh); it brings in the most violated constraint first, like the reference,
 * so optimum and working set agree with the reference's solver on non-degenerate problems. */
int qlb_qp_dense(qlb_context* ctx, size_t B, int n, int m, int p, const double* G, const double* g0,
                 const double* CE, const double* ce0, const double* CI, const double* ci0, double* x,
                 double* cost, uint32_t* status, uint32_t* active, void* stream);
/* Same, HOST pointers; copies in, solves, copies out, synchronises. */
int qlb_qp_dense_host(qlb_context* ctx, size_t B, int n, int m, int p, const double* G, const double* g0,
                      const double* CE, const double* ce0, const double* CI, const double* ci0, double* x,
                      double* cost, uint32_t* status, uint32_t* active);

/* ---- array-of-structs face of the wrench-mode solve ------------------------------------------------------
 * One robot state as ContactForceDistribution::computeForceDistribution consumes it (the State accessors of
 * free_gait_core/src/executor/State.cpp:59-235 plus the Force / Torque arguments), and its result (LegInfo::
 * desiredContactForce_ = -grf, State::getAllJointEfforts, getNetForceAndTorqueOnBase).  Fixed layouts, 8-byte
 * aligned.  A host caller moves one contiguous block per direction over PCIe; the transposition to the solver's
 * SoA arrays is a device kernel. */
typedef struct qlb_wrench_record {
  double q[12];           /* LF, RF, RH, LH x (HAA, HFE, KFE) */
  double quat_wxyz[4];
  double wrench[6];       /* desired net force (3) and torque (3) on the base, base frame */
  double mu[4];           /* friction coefficient per leg */
  uint8_t stance_mask;    /* bit k = leg k is a support leg */
  uint8_t reserved[7];
} qlb_wrench_record;      /* 216 bytes */
typedef struct qlb_result_record {
  double grf[12];
  double tau[12];
  double netwrench[6];
  uint32_t flags;
  uint32_t reserved;
} qlb_result_record;      /* 248 bytes */

/* DEVICE pointers, asynchronous on `stream`: unpack -> qlb_solve_wrench -> pack, in chunks that reuse the
 * context's staging buffers.  Surface normals are the default (0, 0, 1).  The staging is shared with the other calls
 * of the context: a later call, on any stream, does not write it before this one has finished with it. */
int qlb_solve_records(qlb_context* ctx, size_t B, const qlb_wrench_record* records, qlb_result_record* results,
                      void* stream);
/* HOST pointers (pinned memory recommended): chunks flow through the context's copy / compute pipeline with one
 * 1-D copy per chunk and direction; synchronises. */
int qlb_solve_records_host(qlb_context* ctx, size_t B, const qlb_wrench_record* records,
                           qlb_result_record* results);

/* Synthetic robot states on the device (DEVICE pointers, asynchronous on `stream`): the counter-based generator of
 * SURVEY.md 8d, BIT-IDENTICAL to the host generator (quadruped_locomotion_b200/synth.py: splitmix64 streams, elementary
 * functions from IEEE-exact operations), so a sweep of perturbed states - the batch-of-states consumer shape of
 * free_gait_core/src/executor/BatchExecutor.cpp:40-83 and BASELINE config C5 - needs no input staging from the host.
 *   config 1..5 = BASELINE configs C1..C5 (4 = the C3 states); states start .. start + B - 1 of the stream;
 *   seed 0 = the config's default seed (0x5EED0000 + config).  Any output may be NULL.
 * The _f32 twin rounds each value to float on store (what the host generator's .astype(float32) gives). */
int qlb_generate_states(qlb_context* ctx, int config, size_t B, uint64_t start, uint64_t seed, double* q,
                        double* quat_wxyz, double* wrench, uint8_t* stance_mask, double* mu,
                        double* normals_world, void* stream);
int qlb_generate_states_f32(qlb_context* ctx, int config, size_t B, uint64_t start, uint64_t seed, float* q,
                            float* quat_wxyz, float* wrench, uint8_t* stance_mask, float* mu,
                            float* normals_world, void* stream);

/* Device-side statistics over a solved batch (DEVICE pointers; stats_out is a HOST pointer,
 * the call synchronises the stream).  wrench/netwrench may be NULL (error terms then zero). */
int qlb_batch_stats(qlb_context* ctx, size_t B, const uint32_t* flags, const double* wrench,
                    const double* netwrench, qlb_stats* stats_out, void* stream);

/* The one collective of the design (SURVEY 8e): all-reduce *stats over the ranks of an NCCL communicator - the
 * leading QLB_STATS_NUM_SUM doubles with SUM, the rest with MAX - on `stream`; synchronises.  nccl_comm is an
 * ncclComm_t created by the caller (one rank per GPU); stats is a HOST pointer, reduced in place.  NCCL is resolved
 * at run time (dlopen of libnccl.so.2), so linking against libqlb.so does not need NCCL.  No data-path traffic
 * crosses GPUs: instances are sharded, only these 31 numbers are exchanged. */
int qlb_stats_allreduce(qlb_context* ctx, void* nccl_comm, qlb_stats* stats, void* stream);

/* Measure the FP64 FMA throughput of the context's device (TFLOP/s, best of 4 runs of a register-only
 * DFMA kernel): the denominator of the FP64-pipe roofline this path is bound by.  Synchronous. */
int qlb_measure_fp64_peak(qlb_context* ctx, double* tflops_out);

/* How many kernels this context has launched so far (bench.py reports it as gpu_launches). */
uint64_t qlb_launch_count(const qlb_context* ctx);

const char* qlb_strerror(int status);
/* Text of the last CUDA error seen by this context ("" if none). */
const char* qlb_last_cuda_error(const qlb_context* ctx);
int qlb_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* QLB_H */
