"""FP32 twins of the controller tick (qlb_controller_update_f32[_host], include/qlb.h): float arrays in and out, the
controller's state FP64.  The reference is the FP64 controller with the same parameters, fed the float32 inputs widened
to float64: the contact state machine and the status and contact bits must match it exactly, forces and torques within
the stated tolerances, and stale rows must keep their previous values bit for bit."""
import ctypes as C
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from quadruped_locomotion_b200 import capi

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_controller import _rel_state, _robots, _tick  # noqa: E402

KP, KD = (300.0, 250.0, 400.0), (10.0, 12.0, 8.0)
FLOAT_KEYS = ("q", "qd", "pose", "twist", "tpose", "ttwist", "phase", "mu", "pt", "vt")
STATUS = lambda f: (f >> 24) & 7  # noqa: E731
BAD_INPUT = 4
TOL_STANCE, TOL_GRF, TOL_SWING = 1e-3, 5e-4, 1e-4


def _f32(inp):
    """float32 copy of a tick's inputs (masks unchanged) and the same values widened back to float64."""
    lo = {k: (v.astype(np.float32) if k in FLOAT_KEYS else v) for k, v in inp.items()}
    wide = {k: (v.astype(np.float64) if k in FLOAT_KEYS else v) for k, v in lo.items()}
    return lo, wide


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _params(kp=KP, kd=KD):
    p = capi.default_tick_params()
    for c in range(3):
        p.swing.kp[c] = kp[c]; p.swing.kd[c] = kd[c]
    return p


class _Outs:
    def __init__(self, B, dtype):
        self.command = torch.zeros((12, B), dtype=dtype, device="cuda")
        self.flags = torch.zeros(B, dtype=torch.int32, device="cuda")
        self.grf = torch.zeros((12, B), dtype=dtype, device="cuda")


def _update(ctrl, inp, out):
    d = {k: _dev(v) for k, v in inp.items()}
    ctrl.update(d["q"], d["qd"], d["pose"], d["twist"], d["tpose"], d["ttwist"], d["desired"], d["contact"], d["phase"],
                out.command, out.flags, footstep=d["footstep"], mu=d["mu"], ptarget=d["pt"], vtarget=d["vt"], grf=out.grf)


def _state(ctrl):
    limb = torch.zeros((4, ctrl.B), dtype=torch.uint8, device="cuda")
    eff = torch.zeros((12, ctrl.B), dtype=torch.float64, device="cuda")
    ctrl.get_state(limb, eff)
    torch.cuda.synchronize()
    return limb.cpu().numpy(), eff.cpu().numpy()


def _support_rows(limb):
    """[12, B] bool: the joint rows of the support legs (StanceNormal, SwingEarlyTouchDown, Init)."""
    return np.repeat(np.isin(limb, (0, 1, 6)), 3, axis=0)


def _rel_rows(a, b, rows):
    """_rel_state over the selected rows only (other rows count as zero in both)."""
    return _rel_state(np.where(rows, a, 0.0), np.where(rows, b, 0.0)) if rows.any() else 0.0


class _Compare:
    """Checks of one tick of the FP32 controller against the FP64 reference; counts the active-row bits."""

    def __init__(self):
        self.robot_ticks = 0
        self.active_equal = 0
        self.worst = dict(stance=0.0, grf=0.0, swing=0.0)

    def tick(self, k, got, ref, prev_got, prev_ref):
        (limb, eff, cmd, fl, grf), (limb_r, eff_r, cmd_r, fl_r, grf_r) = got, ref
        assert np.array_equal(limb, limb_r), k
        assert np.array_equal(fl & 0x0700000F, fl_r & 0x0700000F), k                # status and contact bits
        self.robot_ticks += fl.size
        self.active_equal += int(((fl & 0x00FFFFF0) == (fl_r & 0x00FFFFF0)).sum())
        stance = _support_rows(limb_r)
        e_st = max(_rel_rows(eff, eff_r, stance), _rel_rows(cmd.astype(np.float64), cmd_r, stance))
        ok = STATUS(fl_r) != BAD_INPUT
        e_grf = _rel_state(grf[:, ok].astype(np.float64), grf_r[:, ok]) if ok.any() else 0.0
        e_sw = max(_rel_rows(eff, eff_r, ~stance), _rel_rows(cmd.astype(np.float64), cmd_r, ~stance))
        assert e_st <= TOL_STANCE and e_grf <= TOL_GRF and e_sw <= TOL_SWING, (k, e_st, e_grf, e_sw)
        for key, v in (("stance", e_st), ("grf", e_grf), ("swing", e_sw)):
            self.worst[key] = max(self.worst[key], v)
        # rows the reference kept are kept here, bit for bit, and no other row is
        if prev_got is not None:
            stale_r = eff_r == prev_ref
            assert np.array_equal(eff[stale_r], prev_got[stale_r]), k
            assert np.array_equal(eff == prev_got, stale_r), k
        assert np.array_equal(cmd, np.clip(eff, -300.0, 300.0).astype(np.float32)), k
        assert np.isfinite(eff).all(), k
        return stance


def _outputs(ctrl, out):
    limb, eff = _state(ctrl)
    return limb, eff, out.command.cpu().numpy(), out.flags.cpu().numpy().view(np.uint32), out.grf.cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_f32_symbols_exported(qlb_built):
    lib = capi.load()
    for name in ("qlb_controller_update_f32", "qlb_controller_update_f32_host"):
        assert name in capi.EXPORTS and hasattr(lib, name), name


def test_f32_update_without_controller(qlb_built):
    lib = capi.load()
    assert lib.qlb_controller_update_f32(None, *([None] * 18)) == -4        # QLB_ERR_NOT_INITIALISED
    assert lib.qlb_controller_update_f32_host(None, *([None] * 17)) == -4


def test_f32_epilogue_is_fp32_without_local_memory(qlb_built):
    """Build check (no GPU): the float instantiation of the tick epilogue exists, keeps everything in registers and
    does no FP64 arithmetic (the clamp of the FP64 efforts is compares and selects, the rest conversions)."""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    txt = subprocess.run(["cuobjdump", "-sass", capi.LIB_PATH], capture_output=True, text=True).stdout
    body, name = {}, None
    for ln in txt.split("\n"):
        m = re.search(r"Function : (\S+)", ln)
        if m:
            name = m.group(1)
            body[name] = []
        elif name:
            body[name].append(ln)
    epi = [k for k in body if "qlb_tick_epilogue_kernel" in k and "IfE" in k]
    assert len(epi) == 1, [k for k in body if "tick" in k]
    sass = "\n".join(body[epi[0]])
    for op in ("STL", "LDL", "DFMA", "DMUL", "DADD"):
        assert not re.search(r"\b" + op + r"\b", sass), op


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def solver(qlb_built):
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device")
    s = capi.Solver("quadruped_model")
    s.set_limb_dynamics("quadruped_model")
    yield s
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("B", [4099, 1])
def test_f32_tick_matches_the_fp64_tick(solver, B):
    """40-tick trot with poisoned robots (NaN base pose: BAD_INPUT; an inf qd sample) and a reset at tick 20."""
    T, R = 40, 20
    rob = _robots(B, seed=31)
    c32, c64 = capi.Controller(solver, B, _params()), capi.Controller(solver, B, _params())
    o32, o64 = _Outs(B, torch.float32), _Outs(B, torch.float64)
    nan_pose = np.arange(3, B, 211) if B > 1 else np.array([], int)
    inf_qd = np.arange(7, B, 307) if B > 1 else np.array([], int)
    reset = (np.random.default_rng(2).random(B) < 0.25).astype(np.uint8)
    cmp = _Compare()
    prev32 = prev64 = None
    inf_ticks = []
    for k in range(T):
        lo, wide = _f32(_tick(rob, k, seed=31))
        if k in (6, 7, 8):
            lo["pose"][2, nan_pose] = np.nan
        if k == 9:
            lo["qd"][4, inf_qd] = np.inf                                     # joint 4 = leg 1: one sample in the ring
        wide = {key: (v.astype(np.float64) if key in FLOAT_KEYS else v) for key, v in lo.items()}
        if k == R:
            c32.reset(_dev(reset)); c64.reset(_dev(reset))
        _update(c32, lo, o32)
        _update(c64, wide, o64)
        got, ref = _outputs(c32, o32), _outputs(c64, o64)
        assert got[2].dtype == np.float32 and got[4].dtype == np.float32
        stance = cmp.tick(k, got, ref, prev32, prev64)
        if k in (6, 7, 8) and nan_pose.size:
            has = stance[:, nan_pose].any(axis=0)
            assert has.any() and (STATUS(got[3][nan_pose[has]]) == BAD_INPUT).all(), k
        if inf_qd.size and prev32 is not None:
            # the inf sample is the newest at tick 9 and the ring's oldest 10 ticks later (read in FP32 from the rounded
            # slot): every poisoned robot whose leg 1 swings is stale on exactly those two ticks
            swing = ~stance[3, inf_qd]
            kept = (got[1][3:6, inf_qd] == prev32[3:6, inf_qd]).all(axis=0)
            if k in (9, 19):
                assert swing.any() and kept[swing].all(), (k, swing, kept)
                inf_ticks.append(k)
            else:
                assert not kept[swing].any(), (k, swing, kept)
        prev32, prev64 = got[1], ref[1]
    if inf_qd.size:
        assert inf_ticks == [9, 19], inf_ticks
    share = cmp.active_equal / cmp.robot_ticks
    print(f"B={B}: active-row bits equal on {cmp.active_equal}/{cmp.robot_ticks} robot-ticks ({share:.5f}); "
          f"worst stance {cmp.worst['stance']:.2e}, grf {cmp.worst['grf']:.2e}, swing {cmp.worst['swing']:.2e}")
    assert share >= 0.999
    c32.close(); c64.close()


@pytest.mark.gpu
def test_f32_phase_is_compared_in_double(solver, oracle):
    """Phases at float32(0.1), float32(0.2), float32(0.5) and their float neighbours: the limb states equal the FP64
    tick's on the widened phase.  Compared against float thresholds instead (0.2f < float32(0.2) > 0.2), some robots
    would land in another state; the restatement shows that this input tells the two apart."""
    from oracle import oracle as O
    marks = [np.float32(x) for x in (0.1, 0.2, 0.5)]
    vals = np.array([v for m in marks for v in (np.nextafter(m, np.float32(0)), m, np.nextafter(m, np.float32(1)))],
                    np.float32)
    B = 16 * 16 * vals.size                                                  # every desired x contact pattern per phase
    rob = _robots(B, seed=9)
    lo, _ = _f32(_tick(rob, 0, seed=9))
    i = np.arange(B)
    lo["phase"] = np.tile(vals[i % vals.size], (4, 1)).astype(np.float32)
    lo["desired"] = ((i // vals.size) % 16).astype(np.uint8)
    lo["contact"] = ((i // (16 * vals.size)) % 16).astype(np.uint8)
    lo["footstep"] = np.full(B, 0xF, np.uint8)
    wide = {key: (v.astype(np.float64) if key in FLOAT_KEYS else v) for key, v in lo.items()}
    c32, c64 = capi.Controller(solver, B, _params()), capi.Controller(solver, B, _params())
    _update(c32, lo, _Outs(B, torch.float32))
    _update(c64, wide, _Outs(B, torch.float64))
    limb32, _ = _state(c32)
    limb64, _ = _state(c64)
    init = np.zeros((4, B), np.uint8)
    want, _ = O.contact_fsm(lo["desired"], lo["footstep"], lo["contact"], wide["phase"], init)
    as_float, _ = O.contact_fsm(lo["desired"], lo["footstep"], lo["contact"], lo["phase"], init)
    assert np.array_equal(limb64, want)
    assert np.array_equal(limb32, want)
    assert not np.array_equal(as_float, want)                                # the input separates the two rules
    c32.close(); c64.close()


@pytest.mark.gpu
def test_f32_command_is_the_rounded_clamp(solver):
    B = 4096
    rob = _robots(B, seed=3)
    ctrl = capi.Controller(solver, B, _params(kp=(1e5, 1e5, 1e5), kd=(1e3, 1e3, 1e3)))
    out = _Outs(B, torch.float32)
    lo, _ = _f32(_tick(rob, 0, seed=3))
    lo["pt"] = lo["pt"] + np.float32(0.5)
    _update(ctrl, lo, out)
    _, eff = _state(ctrl)
    cmd = out.command.cpu().numpy()
    assert (np.abs(eff) > 300.0).sum() > 1000                               # the stored efforts are not clamped
    assert np.array_equal(cmd, np.clip(eff, -300.0, 300.0).astype(np.float32))
    ctrl.close()


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 37])
def test_f32_host_entry_matches_device_entry_and_launch_count(solver, B):
    rob = _robots(B, seed=17)
    dev_c, host_c = capi.Controller(solver, B, _params()), capi.Controller(solver, B, _params())
    out = _Outs(B, torch.float32)
    for k in range(6):
        lo, _ = _f32(_tick(rob, k, seed=17))
        n0 = solver.launches
        _update(dev_c, lo, out)
        n1 = solver.launches
        c = lambda a: np.ascontiguousarray(a)  # noqa: E731
        cmd = np.zeros((12, B), np.float32); fl = np.zeros(B, np.uint32); grf = np.zeros((12, B), np.float32)
        host_c.update_host(c(lo["q"]), c(lo["qd"]), c(lo["pose"]), c(lo["twist"]), c(lo["tpose"]), c(lo["ttwist"]),
                           c(lo["desired"]), c(lo["contact"]), c(lo["phase"]), cmd, fl, footstep=c(lo["footstep"]),
                           mu=c(lo["mu"]), ptarget=c(lo["pt"]), vtarget=c(lo["vt"]), grf=grf)
        n2 = solver.launches
        torch.cuda.synchronize()
        assert n2 - n1 == n1 - n0, (n0, n1, n2)
        assert np.array_equal(cmd, out.command.cpu().numpy()), k
        assert np.array_equal(fl, out.flags.cpu().numpy().view(np.uint32)), k
        assert np.array_equal(grf, out.grf.cpu().numpy()), k
        assert all(np.array_equal(x, y) for x, y in zip(_state(dev_c), _state(host_c))), k
    dev_c.close(); host_c.close()


@pytest.mark.gpu
def test_f32_and_fp64_updates_mix_on_one_controller(solver):
    B, T = 3001, 20
    rob = _robots(B, seed=41)
    mixed, ref = capi.Controller(solver, B, _params()), capi.Controller(solver, B, _params())
    o32, o64, oref = _Outs(B, torch.float32), _Outs(B, torch.float64), _Outs(B, torch.float64)
    cmp = _Compare()
    prev_m = prev_r = None
    for k in range(T):
        lo, wide = _f32(_tick(rob, k, seed=41))
        if k % 2 == 0:
            _update(mixed, lo, o32)
            got = _outputs(mixed, o32)
        else:
            _update(mixed, wide, o64)
            got = _outputs(mixed, o64)
            got = got[:2] + (got[2].astype(np.float32),) + got[3:]          # FP64 command: compare as the clamp check does
        _update(ref, wide, oref)
        r = _outputs(ref, oref)
        cmp.tick(k, got, r, prev_m, prev_r)
        prev_m, prev_r = got[1], r[1]
    assert cmp.active_equal / cmp.robot_ticks >= 0.999
    mixed.close(); ref.close()


@pytest.mark.gpu
def test_capi_picks_the_twin_by_dtype_and_refuses_mixed_arrays(solver):
    B = 257
    rob = _robots(B, seed=5)
    lo, _ = _f32(_tick(rob, 0, seed=5))
    a, b = capi.Controller(solver, B, _params()), capi.Controller(solver, B, _params())
    out = _Outs(B, torch.float32)
    _update(a, lo, out)
    # the same call straight through the FP32 entry point
    d = {k: _dev(v) for k, v in lo.items()}
    cmd = torch.zeros((12, B), dtype=torch.float32, device="cuda")
    fl = torch.zeros(B, dtype=torch.int32, device="cuda")
    grf = torch.zeros((12, B), dtype=torch.float32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    rc = solver.lib.qlb_controller_update_f32(b._c, p(d["q"]), p(d["qd"]), p(d["pose"]), p(d["twist"]), p(d["tpose"]),
                                              p(d["ttwist"]), p(d["desired"]), p(d["footstep"]), p(d["contact"]),
                                              p(d["phase"]), p(d["mu"]), None, p(d["pt"]), p(d["vt"]), p(cmd), p(fl), p(grf),
                                              None)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(out.command, cmd) and torch.equal(out.flags, fl) and torch.equal(out.grf, grf)
    # one float64 array among float32 ones (and the reverse): refused before anything is launched
    n0 = solver.launches
    for key in ("qd", "phase", "pt"):
        bad = dict(lo)
        bad[key] = lo[key].astype(np.float64)
        with pytest.raises(TypeError):
            _update(a, bad, out)
    with pytest.raises(TypeError):
        _update(a, _f32(_tick(rob, 1, seed=5))[1], out)                      # float64 inputs, float32 outputs
    c = np.ascontiguousarray
    with pytest.raises(TypeError):
        a.update_host(c(lo["q"]), c(lo["qd"]), c(lo["pose"]), c(lo["twist"]), c(lo["tpose"]), c(lo["ttwist"]), c(lo["desired"]),
                      c(lo["contact"]), c(lo["phase"]), np.zeros((12, B)), np.zeros(B, np.uint32))
    assert solver.launches == n0
    a.close(); b.close()
