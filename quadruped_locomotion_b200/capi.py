"""ctypes binding of the C ABI in include/qlb.h (libqlb.so, built in-tree by build.py).

This is harness plumbing: torch supplies device memory and streams, the product is the shared
library.  There is no fallback: if libqlb.so is missing or CUDA is unavailable the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np

from . import legmodel

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("QLB_LIB", os.path.join(PKG, "libqlb.so"))  # QLB_LIB: kernel-variant experiments only

NUM_LEGS = 4
STATS_NUM = 31
STATS_NUM_SUM = 29
FLAG_PARITY_MASK = 0x00FFFFFF
PIPELINE_FUSED, PIPELINE_THREE_PASS = 0, 1
STATUS_NAMES = ("ok", "no_stance", "max_iter", "unverified", "bad_input", "infeasible")


class LegModel(C.Structure):
    _fields_ = [("joint_xyz", (C.c_double * 3) * 4), ("joint_rpy", (C.c_double * 3) * 4),
                ("link_mass", C.c_double * 4), ("link_com", (C.c_double * 3) * 4)]


class Params(C.Structure):
    _fields_ = [("wrench_weights", C.c_double * 6), ("ground_force_weight", C.c_double),
                ("min_normal_force", C.c_double), ("friction_default", C.c_double), ("gravity", C.c_double),
                ("kp_translation", C.c_double * 3), ("kd_translation", C.c_double * 3),
                ("kff_translation", C.c_double * 3), ("kp_rotation", C.c_double * 3),
                ("kd_rotation", C.c_double * 3), ("kff_rotation", C.c_double * 3),
                ("torso_mass", C.c_double), ("leg_mass", C.c_double * 4),
                ("leg_base_position", (C.c_double * 3) * 4), ("com_in_base", C.c_double * 3),
                ("gravity_compensation_percentage", C.c_double), ("ipm_tolerance", C.c_double),
                ("ipm_max_iterations", C.c_int32), ("reserved", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("count", C.c_double), ("count_status", C.c_double * 5), ("sum_iterations", C.c_double),
                ("sum_wrench_err", C.c_double), ("active_hist", C.c_double * 20),
                ("count_infeasible", C.c_double), ("max_wrench_err", C.c_double), ("max_iterations", C.c_double)]


EXPORTS = (
    "qlb_default_params", "qlb_create", "qlb_destroy", "qlb_set_params", "qlb_get_params",
    "qlb_solve_wrench", "qlb_solve_wrench_host", "qlb_solve_state", "qlb_solve_state_host",
    "qlb_solve_wrench_f32", "qlb_solve_wrench_f32_host", "qlb_solve_state_f32", "qlb_solve_state_f32_host",
    "qlb_default_swing_params", "qlb_set_limb_dynamics", "qlb_swing_leg_torques", "qlb_swing_leg_torques_host",
    "qlb_set_f32_core", "qlb_set_pipeline", "qlb_generate_states", "qlb_generate_states_f32", "qlb_solve_records", "qlb_solve_records_host", "qlb_stats_allreduce", "qlb_preview_plan_host", "qlb_params_set_key", "qlb_params_get_key", "qlb_params_num_keys", "qlb_params_key", "qlb_params_from_yaml", "qlb_swing_leg_torques_from_queue", "qlb_contact_fsm", "qlb_friction_margins", "qlb_leg_kinematics", "qlb_pack_robot_states", "qlb_feet_in_world", "qlb_qp_dense", "qlb_qp_dense_host", "qlb_batch_stats", "qlb_measure_fp64_peak", "qlb_launch_count", "qlb_strerror",
    "qlb_last_cuda_error", "qlb_abi_version",
    "qlb_default_tick_params", "qlb_controller_create", "qlb_controller_destroy", "qlb_controller_reset",
    "qlb_controller_update", "qlb_controller_update_host", "qlb_controller_get_state",
    "qlb_controller_update_f32", "qlb_controller_update_f32_host",
)

class LimbDynamics(C.Structure):
    _fields_ = [("joint_xyz", (C.c_double * 3) * 3), ("joint_rpy", (C.c_double * 3) * 3), ("body_mass", C.c_double * 3),
                ("body_com", (C.c_double * 3) * 3), ("body_inertia", (C.c_double * 6) * 3)]


class SwingParams(C.Structure):
    _fields_ = [("gravity", C.c_double * 3), ("acceleration_scale", C.c_double), ("kp", C.c_double * 3), ("kd", C.c_double * 3)]


class TickParams(C.Structure):
    _fields_ = [("period", C.c_double), ("effort_limit", C.c_double), ("swing", SwingParams)]


# numpy mirror of qlb_robot_state_record (include/qlb.h)
RECORD_DTYPE = np.dtype([("base_position", "<f8", 3), ("base_orientation_xyzw", "<f8", 4),
                         ("base_linear_velocity", "<f8", 3), ("base_angular_velocity", "<f8", 3),
                         ("joint_position", "<f8", 12), ("surface_normal", "<f8", 12),
                         ("support_leg", "u1", 4), ("reserved", "u1", 4)])
assert RECORD_DTYPE.itemsize == 304

# numpy mirrors of qlb_wrench_record / qlb_result_record (include/qlb.h)
WRENCH_RECORD_DTYPE = np.dtype([("q", "<f8", 12), ("quat_wxyz", "<f8", 4), ("wrench", "<f8", 6), ("mu", "<f8", 4),
                                ("stance_mask", "u1"), ("reserved", "u1", 7)])
RESULT_RECORD_DTYPE = np.dtype([("grf", "<f8", 12), ("tau", "<f8", 12), ("netwrench", "<f8", 6), ("flags", "<u4"),
                                ("reserved", "<u4")])
assert WRENCH_RECORD_DTYPE.itemsize == 216 and RESULT_RECORD_DTYPE.itemsize == 248


PREVIEW_RECORD_DTYPE = np.dtype([("feet_world", "<f8", 12), ("grf", "<f8", 12), ("tau", "<f8", 12), ("netwrench", "<f8", 6),
                                 ("wrench", "<f8", 6), ("friction_margin", "<f8"), ("min_normal_slack", "<f8"), ("flags", "<u4"),
                                 ("reserved", "<u4")])
assert PREVIEW_RECORD_DTYPE.itemsize == 408


def wrench_records(states: dict) -> np.ndarray:
    """SoA state dict (synth.make_states) -> array of qlb_wrench_record."""
    B = states["q"].shape[1]
    rec = np.zeros(B, dtype=WRENCH_RECORD_DTYPE)
    rec["q"] = states["q"].T; rec["quat_wxyz"] = states["quat"].T; rec["wrench"] = states["wrench"].T
    rec["mu"] = states["mu"].T; rec["stance_mask"] = states["mask"]
    return rec


_lib = None
_vp = C.c_void_p


def load() -> C.CDLL:
    """dlopen libqlb.so and declare the signatures.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not found: run `python -m quadruped_locomotion_b200.build` "
                           "(or __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    lib.qlb_default_params.argtypes = [C.POINTER(Params)]
    lib.qlb_create.argtypes = [C.POINTER(_vp), C.POINTER(LegModel), C.POINTER(Params), C.c_int, C.c_size_t]
    lib.qlb_destroy.argtypes = [_vp]
    lib.qlb_set_params.argtypes = [_vp, C.POINTER(Params)]
    lib.qlb_get_params.argtypes = [_vp, C.POINTER(Params)]
    lib.qlb_solve_wrench.argtypes = [_vp, C.c_size_t] + [_vp] * 11
    lib.qlb_solve_wrench_host.argtypes = [_vp, C.c_size_t] + [_vp] * 10
    lib.qlb_solve_state.argtypes = [_vp, C.c_size_t] + [_vp] * 14
    lib.qlb_solve_state_host.argtypes = [_vp, C.c_size_t] + [_vp] * 13
    lib.qlb_solve_wrench_f32.argtypes = [_vp, C.c_size_t] + [_vp] * 11
    lib.qlb_solve_wrench_f32_host.argtypes = [_vp, C.c_size_t] + [_vp] * 10
    lib.qlb_solve_state_f32.argtypes = [_vp, C.c_size_t] + [_vp] * 14
    lib.qlb_solve_state_f32_host.argtypes = [_vp, C.c_size_t] + [_vp] * 13
    lib.qlb_set_f32_core.argtypes = [_vp, C.c_int]
    lib.qlb_set_pipeline.argtypes = [_vp, C.c_int]
    lib.qlb_preview_plan_host.argtypes = [_vp, C.c_size_t, _vp, C.POINTER(C.c_double * 4), _vp]
    lib.qlb_params_set_key.argtypes = [C.POINTER(Params), C.c_char_p, C.c_double]
    lib.qlb_params_get_key.argtypes = [C.POINTER(Params), C.c_char_p, C.POINTER(C.c_double)]
    lib.qlb_params_key.argtypes = [C.c_int]
    lib.qlb_params_key.restype = C.c_char_p
    lib.qlb_params_from_yaml.argtypes = [C.POINTER(Params), C.c_char_p, C.POINTER(C.c_char_p)]
    lib.qlb_swing_leg_torques_from_queue.argtypes = [_vp, C.c_size_t, _vp, _vp, _vp, C.c_double, _vp, _vp, C.POINTER(SwingParams), _vp, _vp]
    lib.qlb_contact_fsm.argtypes = [_vp, C.c_size_t] + [_vp] * 7
    lib.qlb_friction_margins.argtypes = [_vp, C.c_size_t] + [_vp] * 8
    lib.qlb_stats_allreduce.argtypes = [_vp, _vp, C.POINTER(Stats), _vp]
    lib.qlb_solve_records.argtypes = [_vp, C.c_size_t, _vp, _vp, _vp]
    lib.qlb_solve_records_host.argtypes = [_vp, C.c_size_t, _vp, _vp]
    lib.qlb_generate_states.argtypes = [_vp, C.c_int, C.c_size_t, C.c_uint64, C.c_uint64] + [_vp] * 7
    lib.qlb_generate_states_f32.argtypes = [_vp, C.c_int, C.c_size_t, C.c_uint64, C.c_uint64] + [_vp] * 7
    lib.qlb_pack_robot_states.argtypes = [_vp, C.c_size_t] + [_vp] * 7
    lib.qlb_feet_in_world.argtypes = [_vp, C.c_size_t] + [_vp] * 4
    lib.qlb_default_swing_params.argtypes = [C.POINTER(SwingParams)]
    lib.qlb_set_limb_dynamics.argtypes = [_vp, C.POINTER(LimbDynamics)]
    lib.qlb_swing_leg_torques.argtypes = [_vp, C.c_size_t] + [_vp] * 5 + [C.POINTER(SwingParams), _vp, _vp]
    lib.qlb_swing_leg_torques_host.argtypes = [_vp, C.c_size_t] + [_vp] * 5 + [C.POINTER(SwingParams), _vp]
    lib.qlb_leg_kinematics.argtypes = [_vp, C.c_size_t] + [_vp] * 6
    lib.qlb_qp_dense.argtypes = [_vp, C.c_size_t, C.c_int, C.c_int, C.c_int] + [_vp] * 11
    lib.qlb_qp_dense_host.argtypes = [_vp, C.c_size_t, C.c_int, C.c_int, C.c_int] + [_vp] * 10
    lib.qlb_batch_stats.argtypes = [_vp, C.c_size_t, _vp, _vp, _vp, C.POINTER(Stats), _vp]
    lib.qlb_measure_fp64_peak.argtypes = [_vp, C.POINTER(C.c_double)]
    lib.qlb_launch_count.argtypes = [_vp]
    lib.qlb_launch_count.restype = C.c_uint64
    lib.qlb_strerror.argtypes = [C.c_int]
    lib.qlb_strerror.restype = C.c_char_p
    lib.qlb_last_cuda_error.argtypes = [_vp]
    lib.qlb_last_cuda_error.restype = C.c_char_p
    lib.qlb_abi_version.restype = C.c_int
    lib.qlb_default_tick_params.argtypes = [C.POINTER(TickParams)]
    lib.qlb_controller_create.argtypes = [_vp, C.c_size_t, C.POINTER(TickParams), C.POINTER(_vp)]
    lib.qlb_controller_destroy.argtypes = [_vp]
    lib.qlb_controller_reset.argtypes = [_vp, _vp, _vp]
    lib.qlb_controller_update.argtypes = [_vp] + [_vp] * 18
    lib.qlb_controller_update_host.argtypes = [_vp] + [_vp] * 17
    lib.qlb_controller_update_f32.argtypes = [_vp] + [_vp] * 18
    lib.qlb_controller_update_f32_host.argtypes = [_vp] + [_vp] * 17
    lib.qlb_controller_get_state.argtypes = [_vp, _vp, _vp, _vp]
    _lib = lib
    return lib


def default_params() -> Params:
    p = Params()
    rc = load().qlb_default_params(C.byref(p))
    if rc != 0:
        raise RuntimeError("qlb_default_params failed")
    return p


def params_from_yaml(text: str, base: Params | None = None):
    """(Params, first missing key or None) from the text of a controller_gains.yaml-style file."""
    p = base if base is not None else default_params()
    miss = C.c_char_p()
    n = load().qlb_params_from_yaml(C.byref(p), text.encode(), C.byref(miss))
    if n < 0:
        raise RuntimeError("qlb_params_from_yaml failed")
    return p, (miss.value.decode() if miss.value else None)


def leg_models(model: dict | str = "quadruped_model"):
    if isinstance(model, str):
        model = legmodel.load_model(model)
    arr = (LegModel * NUM_LEGS)()
    for i, leg in enumerate(model["legs"]):
        for k in range(4):
            for a in range(3):
                arr[i].joint_xyz[k][a] = leg["joint_xyz"][k][a]
                arr[i].joint_rpy[k][a] = leg["joint_rpy"][k][a]
                arr[i].link_com[k][a] = leg["link_com"][k][a]
            arr[i].link_mass[k] = leg["link_mass"][k]
    return arr


def _is_f32(t) -> bool:
    """float32 arrays select the _f32 twins of the solve entry points."""
    return str(t.dtype).endswith("float32")


def _ptr(t):
    """device/host pointer of a torch tensor or numpy array, or None."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


class Solver:
    """One context = one GPU.  Mirrors the call shape of ContactForceDistribution
    (computeForceDistribution / getNetForceAndTorqueOnBase) for a whole batch."""

    def __init__(self, model: dict | str = "quadruped_model", params: Params | None = None, device: int = 0,
                 max_batch: int = 0):
        self.lib = load()
        self._ctx = _vp()
        legs = leg_models(model)
        rc = self.lib.qlb_create(C.byref(self._ctx), legs, C.byref(params) if params is not None else None,
                                 int(device), int(max_batch))
        if rc != 0:
            self._ctx = _vp()
            raise RuntimeError(f"qlb_create failed: {self.lib.qlb_strerror(rc).decode()} (no CPU fallback)")
        self.device = int(device)

    def close(self):
        for c in list(getattr(self, "_controllers", ())):   # a controller is destroyed before its context
            c.close()
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.qlb_destroy(self._ctx)
            self._ctx = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            detail = self.lib.qlb_last_cuda_error(self._ctx).decode()
            raise RuntimeError(f"{what} failed: {self.lib.qlb_strerror(rc).decode()} {detail}")

    @property
    def launches(self) -> int:
        return int(self.lib.qlb_launch_count(self._ctx))

    def measure_fp64_peak(self) -> float:
        v = C.c_double(0.0)
        self._check(self.lib.qlb_measure_fp64_peak(self._ctx, C.byref(v)), "qlb_measure_fp64_peak")
        return float(v.value)

    def set_params(self, p: Params):
        self._check(self.lib.qlb_set_params(self._ctx, C.byref(p)), "qlb_set_params")

    def set_f32_core(self, fp64_core: bool):
        """Solver core of the _f32 entry points: FP64 (default; FP32 interface only) or FP32."""
        self._check(self.lib.qlb_set_f32_core(self._ctx, 1 if fp64_core else 0), "qlb_set_f32_core")

    def set_pipeline(self, which: str):
        """Kernel organisation: "fused" (one persistent kernel, default) or "three_pass" (the round-1 kernels)."""
        code = {"fused": PIPELINE_FUSED, "three_pass": PIPELINE_THREE_PASS}[which]
        self._check(self.lib.qlb_set_pipeline(self._ctx, code), "qlb_set_pipeline")

    def generate_states(self, config: str, B: int, start: int = 0, seed: int = 0, q=None, quat=None, wrench=None, mask=None,
                        mu=None, normals=None, stream=None):
        """Fill CUDA tensors (SoA [C, B]; float64, or float32 for the _f32 twin) with the synthetic states of a
        BASELINE config - the device twin of synth.make_states, bit-identical to it."""
        cid = {"C1": 1, "C2": 2, "C3": 3, "C4": 4, "C5": 5}[config.upper()]
        ref = next(t for t in (q, quat, wrench, mu, normals) if t is not None)
        fn = self.lib.qlb_generate_states_f32 if _is_f32(ref) else self.lib.qlb_generate_states
        rc = fn(self._ctx, cid, B, int(start), int(seed), _ptr(q), _ptr(quat), _ptr(wrench), _ptr(mask), _ptr(mu), _ptr(normals),
                stream if stream is not None else None)
        self._check(rc, "qlb_generate_states")

    def get_params(self) -> Params:
        p = Params()
        self._check(self.lib.qlb_get_params(self._ctx, C.byref(p)), "qlb_get_params")
        return p

    # -- device-pointer entry points (torch CUDA tensors, SoA [C, B] contiguous; float64, or float32 for the
    #    _f32 twins - every floating-point array of one call must have the same dtype)
    def solve_wrench(self, q, quat, wrench, mask, mu=None, normals=None, grf=None, tau=None, flags=None,
                     netwrench=None, stream=None):
        B = q.shape[1]
        fn = self.lib.qlb_solve_wrench_f32 if _is_f32(q) else self.lib.qlb_solve_wrench
        rc = fn(self._ctx, B, _ptr(q), _ptr(quat), _ptr(wrench), _ptr(mask), _ptr(mu),
                _ptr(normals), _ptr(grf), _ptr(tau), _ptr(flags), _ptr(netwrench),
                stream if stream is not None else None)
        self._check(rc, "qlb_solve_wrench")

    def solve_state(self, q, pose, twist, tpose, ttwist, mask, mu=None, normals=None, grf=None, tau=None,
                    flags=None, netwrench=None, wrench_out=None, stream=None):
        B = q.shape[1]
        fn = self.lib.qlb_solve_state_f32 if _is_f32(q) else self.lib.qlb_solve_state
        rc = fn(self._ctx, B, _ptr(q), _ptr(pose), _ptr(twist), _ptr(tpose), _ptr(ttwist),
                _ptr(mask), _ptr(mu), _ptr(normals), _ptr(grf), _ptr(tau), _ptr(flags),
                _ptr(netwrench), _ptr(wrench_out), stream if stream is not None else None)
        self._check(rc, "qlb_solve_state")

    def leg_kinematics(self, q, quat=None, foot=None, jac=None, gtau=None, stream=None):
        B = q.shape[1]
        rc = self.lib.qlb_leg_kinematics(self._ctx, B, _ptr(q), _ptr(quat), _ptr(foot), _ptr(jac), _ptr(gtau),
                stream if stream is not None else None)
        self._check(rc, "qlb_leg_kinematics")

    def pack_robot_states(self, records, q=None, pose=None, twist=None, mask=None, normals=None, stream=None):
        """records: CUDA uint8 tensor holding B qlb_robot_state_record structs (RECORD_DTYPE)."""
        B = records.numel() // RECORD_DTYPE.itemsize
        rc = self.lib.qlb_pack_robot_states(self._ctx, B, _ptr(records), _ptr(q), _ptr(pose), _ptr(twist), _ptr(mask),
                                            _ptr(normals), stream if stream is not None else None)
        self._check(rc, "qlb_pack_robot_states")

    def feet_in_world(self, q, pose, feet_world, stream=None):
        rc = self.lib.qlb_feet_in_world(self._ctx, q.shape[1], _ptr(q), _ptr(pose), _ptr(feet_world),
                                        stream if stream is not None else None)
        self._check(rc, "qlb_feet_in_world")

    def set_limb_dynamics(self, model: dict | str = "quadruped_model"):
        """Upload the rigid-body tables of the four limbs (models/<name>.json, key "limb_dynamics")."""
        if isinstance(model, str):
            model = legmodel.load_model(model)
        arr = (LimbDynamics * NUM_LEGS)()
        for i, leg in enumerate(model["limb_dynamics"]):
            for k in range(3):
                for a in range(3):
                    arr[i].joint_xyz[k][a] = leg["joint_xyz"][k][a]
                    arr[i].joint_rpy[k][a] = leg["joint_rpy"][k][a]
                    arr[i].body_com[k][a] = leg["body_com"][k][a]
                arr[i].body_mass[k] = leg["body_mass"][k]
                for a in range(6):
                    arr[i].body_inertia[k][a] = leg["body_inertia"][k][a]
        self._check(self.lib.qlb_set_limb_dynamics(self._ctx, arr), "qlb_set_limb_dynamics")

    def default_swing_params(self) -> SwingParams:
        p = SwingParams()
        self._check(self.lib.qlb_default_swing_params(C.byref(p)), "qlb_default_swing_params")
        return p

    def swing_leg_torques(self, q, qd, qdd, ptarget, vtarget, params: SwingParams, tau, stream=None):
        rc = self.lib.qlb_swing_leg_torques(self._ctx, q.shape[1], _ptr(q), _ptr(qd), _ptr(qdd), _ptr(ptarget), _ptr(vtarget),
                                            C.byref(params), _ptr(tau), stream if stream is not None else None)
        self._check(rc, "qlb_swing_leg_torques")

    def swing_leg_torques_from_queue(self, q, qd_back, qd_front, period, ptarget, vtarget, params: SwingParams, tau, stream=None):
        rc = self.lib.qlb_swing_leg_torques_from_queue(self._ctx, q.shape[1], _ptr(q), _ptr(qd_back), _ptr(qd_front), float(period),
                                                       _ptr(ptarget), _ptr(vtarget), C.byref(params), _ptr(tau),
                                                       stream if stream is not None else None)
        self._check(rc, "qlb_swing_leg_torques_from_queue")

    def contact_fsm(self, desired, footstep, contact, phase, limb_state, stance=None, stream=None):
        rc = self.lib.qlb_contact_fsm(self._ctx, desired.shape[0], _ptr(desired), _ptr(footstep), _ptr(contact), _ptr(phase),
                                      _ptr(limb_state), _ptr(stance), stream if stream is not None else None)
        self._check(rc, "qlb_contact_fsm")

    def friction_margins(self, grf, quat, mask, mu, normals, margin, min_normal=None, stream=None):
        rc = self.lib.qlb_friction_margins(self._ctx, grf.shape[1], _ptr(grf), _ptr(quat), _ptr(mask), _ptr(mu), _ptr(normals),
                                           _ptr(margin), _ptr(min_normal), stream if stream is not None else None)
        self._check(rc, "qlb_friction_margins")

    def swing_leg_torques_host(self, q, qd, qdd, ptarget, vtarget, params: SwingParams, tau):
        rc = self.lib.qlb_swing_leg_torques_host(self._ctx, q.shape[1], _ptr(q), _ptr(qd), _ptr(qdd), _ptr(ptarget), _ptr(vtarget),
                                                 C.byref(params), _ptr(tau))
        self._check(rc, "qlb_swing_leg_torques_host")

    def batch_stats(self, flags, wrench=None, netwrench=None, stream=None) -> np.ndarray:
        st = Stats()
        B = flags.shape[0]
        rc = self.lib.qlb_batch_stats(self._ctx, B, _ptr(flags), _ptr(wrench), _ptr(netwrench), C.byref(st),
                stream if stream is not None else None)
        self._check(rc, "qlb_batch_stats")
        return np.frombuffer(bytes(st), dtype=np.float64).copy()

    # -- host-pointer entry points (numpy arrays or pinned torch CPU tensors)
    def solve_wrench_host(self, q, quat, wrench, mask, mu=None, normals=None, grf=None, tau=None, flags=None,
                          netwrench=None):
        B = q.shape[1]
        fn = self.lib.qlb_solve_wrench_f32_host if _is_f32(q) else self.lib.qlb_solve_wrench_host
        rc = fn(self._ctx, B, _ptr(q), _ptr(quat), _ptr(wrench), _ptr(mask), _ptr(mu),
                _ptr(normals), _ptr(grf), _ptr(tau), _ptr(flags), _ptr(netwrench))
        self._check(rc, "qlb_solve_wrench_host")

    def solve_state_host(self, q, pose, twist, tpose, ttwist, mask, mu=None, normals=None, grf=None, tau=None,
                         flags=None, netwrench=None, wrench_out=None):
        B = q.shape[1]
        fn = self.lib.qlb_solve_state_f32_host if _is_f32(q) else self.lib.qlb_solve_state_host
        rc = fn(self._ctx, B, _ptr(q), _ptr(pose), _ptr(twist), _ptr(tpose),
                _ptr(ttwist), _ptr(mask), _ptr(mu), _ptr(normals), _ptr(grf), _ptr(tau),
                _ptr(flags), _ptr(netwrench), _ptr(wrench_out))
        self._check(rc, "qlb_solve_state_host")

    def preview_plan_host(self, records: np.ndarray, mu=None) -> np.ndarray:
        """records: numpy array of RECORD_DTYPE (the states of a planned motion) -> array of PREVIEW_RECORD_DTYPE."""
        B = records.shape[0]
        out = np.zeros(B, dtype=PREVIEW_RECORD_DTYPE)
        mu_arr = (C.c_double * 4)(*[float(v) for v in mu]) if mu is not None else None
        rc = self.lib.qlb_preview_plan_host(self._ctx, B, _ptr(records), C.byref(mu_arr) if mu_arr is not None else None, _ptr(out))
        self._check(rc, "qlb_preview_plan_host")
        return out

    def solve_records_host(self, records, results):
        """records: B qlb_wrench_record (numpy structured array or pinned torch uint8 tensor), results: B
        qlb_result_record, both HOST memory."""
        B = (records.shape[0] if isinstance(records, np.ndarray) else records.numel() // WRENCH_RECORD_DTYPE.itemsize)
        self._check(self.lib.qlb_solve_records_host(self._ctx, B, _ptr(records), _ptr(results)), "qlb_solve_records_host")

    def solve_records(self, records, results, stream=None):
        """DEVICE uint8 tensors holding B qlb_wrench_record / B qlb_result_record."""
        B = records.numel() // WRENCH_RECORD_DTYPE.itemsize
        self._check(self.lib.qlb_solve_records(self._ctx, B, _ptr(records), _ptr(results), stream if stream is not None else None),
                    "qlb_solve_records")

    def qp_dense_numpy(self, G, g0, CI=None, ci0=None, CE=None, ce0=None) -> dict:
        """Batched generic QP through the host entry point.  G[B,n,n], g0[B,n], CI[B,n,m], ci0[B,m],
        CE[B,n,p], ce0[B,p] in QuadProg++ convention (CI' x + ci0 >= 0); returns x[B,n], cost, status, active."""
        G = np.asarray(G, dtype=np.float64); g0 = np.asarray(g0, dtype=np.float64)
        B, n = g0.shape
        m = 0 if CI is None else np.asarray(CI).shape[2]
        p = 0 if CE is None else np.asarray(CE).shape[2]
        soa = lambda a, k: np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(B, k).T)  # noqa: E731
        Gs, gs = soa(G, n * n), soa(g0, n)
        CIs = soa(CI, n * m) if m else None; cis = soa(ci0, m) if m else None
        CEs = soa(CE, n * p) if p else None; ces = soa(ce0, p) if p else None
        x = np.zeros((n, B)); cost = np.zeros(B); status = np.zeros(B, np.uint32); active = np.zeros(B, np.uint32)
        rc = self.lib.qlb_qp_dense_host(self._ctx, B, n, m, p, _ptr(Gs), _ptr(gs), _ptr(CEs), _ptr(ces), _ptr(CIs),
                _ptr(cis), _ptr(x), _ptr(cost), _ptr(status), _ptr(active))
        self._check(rc, "qlb_qp_dense_host")
        return dict(x=np.ascontiguousarray(x.T), cost=cost, status=status, active=active)

    def solve_wrench_numpy(self, states: dict, with_net=True, dtype=np.float64) -> dict:
        """Convenience for tests: numpy SoA in, numpy SoA out, through the host entry point
        (dtype=np.float32: the _f32 twin)."""
        B = states["q"].shape[1]
        f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=dtype)  # noqa: E731
        q, quat, wr = f64(states["q"]), f64(states["quat"]), f64(states["wrench"])
        mu, nr = f64(states.get("mu")), f64(states.get("normals"))
        mask = np.ascontiguousarray(states["mask"], dtype=np.uint8)
        grf = np.zeros((12, B), dtype); tau = np.zeros((12, B), dtype); flags = np.zeros(B, dtype=np.uint32)
        net = np.zeros((6, B), dtype) if with_net else None
        self.solve_wrench_host(q, quat, wr, mask, mu, nr, grf, tau, flags, net)
        return dict(grf=grf, tau=tau, flags=flags, netwrench=net)


def default_tick_params() -> TickParams:
    p = TickParams()
    if load().qlb_default_tick_params(C.byref(p)) != 0:
        raise RuntimeError("qlb_default_tick_params failed")
    return p


class Controller:
    """RosBalanceController::update for B robots: one update() per control tick, the limb states, joint efforts and
    joint-velocity history of every robot kept on the device between ticks (include/qlb.h, qlb_controller_*).
    Belongs to the Solver's context; Solver.close() closes it first."""

    def __init__(self, solver: Solver, B: int, params: TickParams | None = None):
        self.solver = solver
        self.lib = solver.lib
        self.B = int(B)
        self._c = _vp()
        rc = self.lib.qlb_controller_create(solver._ctx, self.B, C.byref(params) if params is not None else None, C.byref(self._c))
        if rc != 0:
            self._c = _vp()
            solver._check(rc, "qlb_controller_create")
        if not hasattr(solver, "_controllers"):
            solver._controllers = weakref.WeakSet()
        solver._controllers.add(self)

    def close(self):
        if getattr(self, "_c", None) is not None and self._c.value:
            self.lib.qlb_controller_destroy(self._c)
            self._c = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _pick(fn64, fn32, arrays):
        """The FP64 entry point, or its _f32 twin when q is float32.  Every floating-point array of the call must have
        the dtype of q: the library reads each array as that type."""
        dtypes = {str(a.dtype).split(".")[-1] for a in arrays if a is not None}
        if len(dtypes) > 1:
            raise TypeError(f"controller update: floating-point arrays of mixed dtypes {sorted(dtypes)}; "
                            "use float64 throughout, or float32 throughout for the _f32 twin")
        return fn32 if _is_f32(arrays[0]) else fn64

    # -- DEVICE pointers (torch CUDA tensors, SoA [C, B] contiguous float64, or float32 throughout for the _f32 twin;
    #    masks uint8 [B]; flags 32-bit [B])
    def update(self, q, qd, pose, twist, tpose, ttwist, desired, contact, phase, command, flags, footstep=None, mu=None,
               normals=None, ptarget=None, vtarget=None, grf=None, stream=None):
        fn = self._pick(self.lib.qlb_controller_update, self.lib.qlb_controller_update_f32,
                        (q, qd, pose, twist, tpose, ttwist, phase, mu, normals, ptarget, vtarget, command, grf))
        rc = fn(self._c, _ptr(q), _ptr(qd), _ptr(pose), _ptr(twist), _ptr(tpose), _ptr(ttwist),
                _ptr(desired), _ptr(footstep), _ptr(contact), _ptr(phase), _ptr(mu), _ptr(normals),
                _ptr(ptarget), _ptr(vtarget), _ptr(command), _ptr(flags), _ptr(grf),
                stream if stream is not None else None)
        self.solver._check(rc, "qlb_controller_update")

    def reset(self, mask=None, stream=None):
        """RosBalanceController::starting for the robots with mask[i] != 0 (device uint8 [B]; None = all)."""
        self.solver._check(self.lib.qlb_controller_reset(self._c, _ptr(mask), stream if stream is not None else None),
                           "qlb_controller_reset")

    def get_state(self, limb_state=None, efforts=None, stream=None):
        """Device copies of the persistent state: limb_state uint8 [4, B], efforts float64 [12, B]."""
        self.solver._check(self.lib.qlb_controller_get_state(self._c, _ptr(limb_state), _ptr(efforts),
                                                             stream if stream is not None else None), "qlb_controller_get_state")

    # -- HOST pointers (numpy arrays or pinned torch CPU tensors); synchronises
    def update_host(self, q, qd, pose, twist, tpose, ttwist, desired, contact, phase, command, flags, footstep=None, mu=None,
                    normals=None, ptarget=None, vtarget=None, grf=None):
        fn = self._pick(self.lib.qlb_controller_update_host, self.lib.qlb_controller_update_f32_host,
                        (q, qd, pose, twist, tpose, ttwist, phase, mu, normals, ptarget, vtarget, command, grf))
        rc = fn(self._c, _ptr(q), _ptr(qd), _ptr(pose), _ptr(twist), _ptr(tpose), _ptr(ttwist), _ptr(desired), _ptr(footstep),
                _ptr(contact), _ptr(phase), _ptr(mu), _ptr(normals), _ptr(ptarget), _ptr(vtarget), _ptr(command), _ptr(flags),
                _ptr(grf))
        self.solver._check(rc, "qlb_controller_update_host")
