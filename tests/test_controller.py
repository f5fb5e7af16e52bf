"""The controller tick (qlb_controller_*, include/qlb.h): RosBalanceController::update for B robots in one call, with
the limb states, joint efforts and joint-velocity history of every robot kept on the device.  Checked against the
existing entry points called one after another, against the numpy restatement (tests/controller_oracle.py), and for the
rules the tick adds: stale efforts on a failed solve, the command clamp and the reset."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from quadruped_locomotion_b200 import build, capi, legmodel, synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import controller_oracle as CO  # noqa: E402

PERIOD = 0.0025
KP, KD = (300.0, 250.0, 400.0), (10.0, 12.0, 8.0)
NEW_SYMBOLS = ("qlb_default_tick_params", "qlb_controller_create", "qlb_controller_destroy", "qlb_controller_reset",
               "qlb_controller_update", "qlb_controller_update_host", "qlb_controller_get_state")


def _robots(B, seed=11):
    """Per-robot constants: trot phase offset, friction coefficients, footstep masks, nominal base height."""
    rng = np.random.default_rng(seed)
    fs = np.full(B, 0xF, np.uint8)
    fs[rng.random(B) < 0.1] = 0b0111
    return dict(offset=rng.integers(0, 8, B), mu=rng.uniform(0.4, 1.0, (4, B)), footstep=fs, z=0.45 + rng.normal(0, 0.01, B))


def _tick(rob, k, seed=11):
    """Inputs of tick k for a trot: LF+RH and RF+LH alternate every 8 ticks (per-robot offset), with early, late and lost
    touchdowns drawn at random."""
    B = rob["offset"].shape[0]
    rng = np.random.default_rng([seed, k])
    kk = k + rob["offset"]
    half = (kk // 8) % 2
    ph = (kk % 8) / 8.0
    desired = np.where(half == 0, 0b0101, 0b1010).astype(np.uint8)
    contact = desired.copy()
    for leg in range(4):
        bit = np.uint8(1 << leg)
        st = (desired & bit) != 0
        early = ~st & (ph > 0.5) & (rng.random(B) < 0.3)
        late = st & (ph < 0.1) & (rng.random(B) < 0.3)
        lost = st & (ph > 0.5) & (rng.random(B) < 0.1)
        contact = np.where(early, contact | bit, contact)
        contact = np.where(late | lost, contact & ~bit, contact).astype(np.uint8)
    s = np.array([1, -1, 1, -1])[:, None]
    q = np.zeros((12, B))
    q[0::3] = rng.uniform(-0.2, 0.2, (4, B))
    q[1::3] = s * (0.7 + rng.uniform(-0.2, 0.2, (4, B)))
    q[2::3] = -s * (1.4 + rng.uniform(-0.3, 0.3, (4, B)))
    qd = rng.normal(0, 1.0, (12, B))
    quat = synth.quat_from_ypr(rng.normal(0, 0.3, B), rng.normal(0, 0.03, B), rng.normal(0, 0.03, B))
    pose = np.concatenate([rng.normal(0, 0.01, (3, B)) + np.stack([np.zeros(B), np.zeros(B), rob["z"]]), quat])
    twist = rng.normal(0, 0.05, (6, B))
    tpose = np.concatenate([pose[:3] + rng.normal(0, 0.004, (3, B)), quat])
    ttwist = rng.normal(0, 0.05, (6, B))
    foot = np.array([[0.42, 0.15, -0.4], [0.42, -0.15, -0.4], [-0.42, -0.15, -0.4], [-0.42, 0.15, -0.4]]).reshape(12, 1)
    pt = foot + rng.normal(0, 0.03, (12, B))
    vt = rng.normal(0, 0.2, (12, B))
    return dict(q=q, qd=qd, pose=pose, twist=twist, tpose=tpose, ttwist=ttwist, desired=desired, footstep=rob["footstep"],
                contact=contact, phase=np.tile(ph, (4, 1)), mu=rob["mu"], pt=pt, vt=vt)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _params(kp=KP, kd=KD):
    p = capi.default_tick_params()
    for c in range(3):
        p.swing.kp[c] = kp[c]; p.swing.kd[c] = kd[c]
    return p


class _Outs:
    def __init__(self, B):
        self.command = torch.zeros((12, B), dtype=torch.float64, device="cuda")
        self.flags = torch.zeros(B, dtype=torch.int32, device="cuda")
        self.grf = torch.zeros((12, B), dtype=torch.float64, device="cuda")


def _update(ctrl, inp, out, stream=None, d=None):
    d = d or {k: _dev(v) for k, v in inp.items()}
    ctrl.update(d["q"], d["qd"], d["pose"], d["twist"], d["tpose"], d["ttwist"], d["desired"], d["contact"], d["phase"],
                out.command, out.flags, footstep=d["footstep"], mu=d["mu"], ptarget=d["pt"], vtarget=d["vt"], grf=out.grf,
                stream=stream)


def _state(ctrl):
    limb = torch.zeros((4, ctrl.B), dtype=torch.uint8, device="cuda")
    eff = torch.zeros((12, ctrl.B), dtype=torch.float64, device="cuda")
    ctrl.get_state(limb, eff)
    torch.cuda.synchronize()
    return limb.cpu().numpy(), eff.cpu().numpy()


def _support(limb):
    """Support legs of a limb state array (StanceNormal, SwingEarlyTouchDown, Init)."""
    m = np.zeros(limb.shape[1], np.uint8)
    for leg in range(4):
        m |= (np.isin(limb[leg], (0, 1, 6)).astype(np.uint8) << leg).astype(np.uint8)
    return m


def _rel(a, b):
    """Largest elementwise |a - b| / max(1, |b|)."""
    return float((np.abs(a - b) / np.maximum(1.0, np.abs(b))).max()) if a.size else 0.0


def _rel_state(a, b):
    """Largest per-robot |a - b|_inf / max(1, |b|_inf) (the metric of the solver's parity tests)."""
    return float((np.abs(a - b).max(axis=0) / np.maximum(1.0, np.abs(b).max(axis=0))).max())


def _stance_rows(mask):
    """[12, B] bool: the joint rows of the stance legs."""
    return np.repeat(np.stack([((mask >> leg) & 1).astype(bool) for leg in range(4)]), 3, axis=0)


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_new_symbols_exported(qlb_built):
    lib = capi.load()
    for name in NEW_SYMBOLS:
        assert name in capi.EXPORTS and hasattr(lib, name), name


def test_tick_params_layout(qlb_built):
    assert C.sizeof(capi.TickParams) == 96 == 2 * 8 + C.sizeof(capi.SwingParams)
    p = capi.default_tick_params()
    assert p.period == 0.0025 and p.effort_limit == 300.0
    assert list(p.swing.gravity) == [0.0, -9.81, 0.0] and p.swing.acceleration_scale == 0.5


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_controller_create_needs_a_device(qlb_built):
    out = C.c_void_p()
    assert capi.load().qlb_controller_create(None, 16, None, C.byref(out)) == -2   # QLB_ERR_CUDA
    assert not out.value


def test_controller_demo_compiles_and_links(qlb_built):
    demo = build.build_host_demo(which="controller_demo")
    out = subprocess.run(["ldd", demo], capture_output=True, text=True).stdout
    assert "libqlb.so" in out and "not found" not in out


def test_restatement_ring_rule():
    B = 3
    st = CO.controller_init(B)
    samples = [np.full((12, B), float(k + 1)) for k in range(14)]
    ring, front = CO.ring_push(st, samples[0])
    assert np.array_equal(front, samples[0])                       # first tick after create: qdd = 0
    st = dict(st, ring=ring, refill=np.zeros(B, bool))
    for k in range(1, 14):
        ring, front = CO.ring_push(st, samples[k])
        st = dict(st, ring=ring)
        want = samples[max(k - 10, 0)]                             # 10 ticks back; the start-up fill before that
        assert np.array_equal(front, want), k
    st = CO.controller_reset(st, np.array([0, 1, 0], np.uint8))
    ring, front = CO.ring_push(st, samples[0])
    assert np.array_equal(front[:, 1], samples[0][:, 1]) and np.array_equal(front[:, 0], samples[4][:, 0])
    assert (st["efforts"][:, 1] == 0).all() and (st["limb_state"][:, 1] == 0).all()


def test_restatement_stale_and_clamp_rules():
    B = 4
    prev = np.arange(48, dtype=np.float64).reshape(12, B) + 1.0
    tau = -np.ones((12, B)); swing = np.full((12, B), 7.0)
    swing[0, 3] = np.nan                                           # leg 0 of robot 3: one non-finite joint
    stance = np.array([0b0011, 0b0011, 0b0000, 0b1100], np.uint8)
    flags = (np.array([0, 4, 1, 2], np.uint32) << 24)              # OK, BAD_INPUT, NO_STANCE, MAX_ITER
    eff = CO.merge(prev, stance, flags, tau, swing)
    want = prev.copy()
    want[0:6, 0] = -1.0; want[6:12, 0] = 7.0                      # solved: the solve's torques; swing legs: swing torques
    want[6:12, 1] = 7.0                                            # failed (BAD_INPUT): stance rows stale
    want[:, 2] = 7.0                                               # no stance leg
    want[3:6, 3] = 7.0                                             # MAX_ITER: stance rows 6..11 stale; leg 0 non-finite: kept
    assert np.array_equal(eff, want)
    big = np.array([[-1e4, -300.0, 299.0, 1e4]])
    assert np.array_equal(np.clip(big, -300.0, 300.0), [[-300.0, -300.0, 299.0, 300.0]])


def test_restatement_tick_keeps_efforts_of_bad_input(oracle):
    """controller_tick end to end on the CPU: a NaN joint angle makes the solve BAD_INPUT and every row of that robot
    keeps its previous efforts; the clamp limits the command only."""
    m = legmodel.load_model("quadruped_model")
    M = oracle.model_array(m)
    rob = _robots(3)
    inp = _tick(rob, 0)
    st = CO.controller_init(3)
    st["efforts"][:] = 400.0
    inp["contact"] = inp["desired"].copy()                         # every planned stance leg in contact
    inp["q"][4, 1] = np.nan
    new, out = CO.controller_tick(oracle, m, M, st, inp["q"], inp["qd"], inp["pose"], inp["twist"], inp["tpose"], inp["ttwist"],
                                  inp["desired"], inp["footstep"], inp["contact"], inp["phase"], mu=inp["mu"], ptarget=inp["pt"],
                                  vtarget=inp["vt"], kp=KP, kd=KD)
    assert (out["flags"][1] >> 24) & 7 == 4
    kept = _stance_rows(out["stance"])[:, 1]
    kept[3:6] = True                                               # leg 1 holds the NaN: its swing row is kept too
    assert (new["efforts"][kept, 1] == 400.0).all() and (out["command"][kept, 1] == 300.0).all()
    assert not (new["efforts"][~kept, 1] == 400.0).any()
    assert np.abs(out["qdd"]).max() == 0.0                         # start-up fill
    assert np.isfinite(new["efforts"]).all() and not (new["efforts"][:, 0] == 400.0).any()


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
def test_tick_is_the_composition_of_the_entry_points(solver):
    B, T = 20011, 40
    rob = _robots(B)
    ctrl = capi.Controller(solver, B, _params())
    out = _Outs(B)
    prm = solver.default_swing_params()
    for c in range(3):
        prm.kp[c] = KP[c]; prm.kd[c] = KD[c]
    limb = torch.zeros((4, B), dtype=torch.uint8, device="cuda")
    stance = torch.zeros(B, dtype=torch.uint8, device="cuda")
    grf = torch.zeros((12, B), dtype=torch.float64, device="cuda"); tau = torch.zeros_like(grf); swing = torch.zeros_like(grf)
    flags = torch.zeros(B, dtype=torch.int32, device="cuda")
    ref = CO.controller_init(B)
    seen = set()
    for k in range(T):
        inp = _tick(rob, k)
        d = {key: _dev(v) for key, v in inp.items()}
        _update(ctrl, inp, out, d=d)
        solver.contact_fsm(d["desired"], d["footstep"], d["contact"], d["phase"], limb, stance)
        solver.solve_state(d["q"], d["pose"], d["twist"], d["tpose"], d["ttwist"], stance, d["mu"], None, grf, tau, flags)
        ring, front = CO.ring_push(ref, inp["qd"])
        solver.swing_leg_torques_from_queue(d["q"], d["qd"], _dev(front), PERIOD, d["pt"], d["vt"], prm, swing)
        torch.cuda.synchronize()
        st_ref, fl_ref = stance.cpu().numpy(), flags.cpu().numpy().view(np.uint32)
        eff_ref = CO.merge(ref["efforts"], st_ref, fl_ref, tau.cpu().numpy(), swing.cpu().numpy())
        ref = dict(limb_state=limb.cpu().numpy(), efforts=eff_ref, ring=ring, refill=np.zeros(B, bool))
        got_limb, got_eff = _state(ctrl)
        assert np.array_equal(got_limb, ref["limb_state"]), k
        assert np.array_equal(_support(got_limb), st_ref), k
        assert np.array_equal(out.flags.cpu().numpy().view(np.uint32), fl_ref), k
        assert np.array_equal(out.grf.cpu().numpy(), grf.cpu().numpy()), k
        rows = _stance_rows(st_ref)
        assert np.array_equal(got_eff[rows], eff_ref[rows]), k
        assert _rel(got_eff[~rows], eff_ref[~rows]) <= 1e-12, k
        assert np.array_equal(out.command.cpu().numpy(), np.clip(got_eff, -300.0, 300.0)), k
        assert np.isfinite(got_eff).all()
        seen |= set(np.unique(got_limb).tolist())
    # the trot went through early, late and lost touchdowns
    assert {1, 3, 4, 6, 8} <= seen, seen
    ctrl.close()


@pytest.mark.gpu
def test_tick_matches_the_restatement(solver, oracle):
    B, T = 64, 10
    m = legmodel.load_model("quadruped_model")
    M = oracle.model_array(m)
    rob = _robots(B, seed=5)
    ctrl = capi.Controller(solver, B, _params())
    out = _Outs(B)
    st = CO.controller_init(B)
    for k in range(T):
        inp = _tick(rob, k, seed=5)
        _update(ctrl, inp, out)
        st, want = CO.controller_tick(oracle, m, M, st, inp["q"], inp["qd"], inp["pose"], inp["twist"], inp["tpose"],
                                      inp["ttwist"], inp["desired"], inp["footstep"], inp["contact"], inp["phase"], mu=inp["mu"],
                                      ptarget=inp["pt"], vtarget=inp["vt"], kp=KP, kd=KD)
        limb, eff = _state(ctrl)
        fl = out.flags.cpu().numpy().view(np.uint32)
        assert np.array_equal(limb, want["limb_state"]), k
        assert np.array_equal(fl & capi.FLAG_PARITY_MASK, want["flags"] & capi.FLAG_PARITY_MASK), k
        assert _rel_state(out.grf.cpu().numpy(), want["grf"]) <= 1e-9, k
        assert _rel_state(eff, want["efforts"]) <= 1e-9, k
        assert _rel_state(out.command.cpu().numpy(), want["command"]) <= 1e-9, k
    ctrl.close()


@pytest.mark.gpu
def test_failed_solves_keep_stale_efforts(solver):
    B, T, K = 2000, 6, 3
    rob = _robots(B, seed=7)
    clean, dirty = capi.Controller(solver, B, _params()), capi.Controller(solver, B, _params())
    oc, od = _Outs(B), _Outs(B)
    nan_q, bad_quat, first = np.arange(0, B, 17), np.arange(5, B, 23), np.arange(9, B, 29)
    hit = np.zeros(B, bool); hit[nan_q] = hit[bad_quat] = True
    hit0 = np.zeros(B, bool); hit0[first] = True
    prev = None
    for k in range(T):
        inp = _tick(rob, k, seed=7)
        _update(clean, inp, oc)
        bad = {key: v.copy() for key, v in inp.items()}
        sel = hit if k == K else (hit0 if k == 0 else np.zeros(B, bool))
        if k == K:
            bad["q"][7, nan_q] = np.nan
            bad["pose"][3:, bad_quat] *= 1.01                      # |q|^2 off by 2e-2: not a unit quaternion
        if k == 0:
            bad["q"][2, first] = np.nan
        _update(dirty, bad, od)
        torch.cuda.synchronize()
        _, ec = _state(clean)
        _, ed = _state(dirty)
        cmd = od.command.cpu().numpy()
        fl = od.flags.cpu().numpy().view(np.uint32)
        assert np.isfinite(cmd).all() and np.isfinite(ed).all()
        has_stance = _support(_state(dirty)[0]) != 0
        assert ((fl[sel & has_stance] >> 24) & 7 == 4).all()
        rows = _stance_rows(_support(_state(dirty)[0]))
        before = prev if k > 0 else np.zeros((12, B))
        for i in np.flatnonzero(sel):
            assert np.array_equal(ed[rows[:, i], i], before[rows[:, i], i]), (k, i)
        if k == K:
            # the NaN is joint 7 (leg 2): that leg's row is kept whether it stands or swings; the other swing legs only
            # use their own joints and are recomputed
            assert np.array_equal(ed[6:9, nan_q], before[6:9, nan_q])
        # other robots are unaffected (robots hit at tick 0 restart from zero efforts, as the clean run does at tick 0)
        other = ~hit & ~hit0 if k >= K else ~hit0
        assert np.array_equal(ed[:, other], ec[:, other]), k
        assert np.array_equal(cmd[:, other], oc.command.cpu().numpy()[:, other]), k
        prev = ed
    clean.close(); dirty.close()


@pytest.mark.gpu
def test_command_is_clamped_not_the_efforts(solver):
    B = 4096
    rob = _robots(B, seed=3)
    ctrl = capi.Controller(solver, B, _params(kp=(1e5, 1e5, 1e5), kd=(1e3, 1e3, 1e3)))
    out = _Outs(B)
    inp = _tick(rob, 0, seed=3)
    inp["pt"] = inp["pt"] + 0.5
    _update(ctrl, inp, out)
    _, eff = _state(ctrl)
    cmd = out.command.cpu().numpy()
    big = np.abs(eff) > 300.0
    assert big.sum() > 1000
    assert np.array_equal(np.abs(cmd[big]), np.full(big.sum(), 300.0)) and np.array_equal(np.sign(cmd[big]), np.sign(eff[big]))
    assert np.array_equal(cmd[~big], eff[~big])
    ctrl.close()


@pytest.mark.gpu
def test_reset_of_a_subset(solver):
    B, T, R = 3001, 12, 6
    rob = _robots(B, seed=13)
    a, b = capi.Controller(solver, B, _params()), capi.Controller(solver, B, _params())
    oa, ob = _Outs(B), _Outs(B)
    mask = (np.random.default_rng(1).random(B) < 0.3).astype(np.uint8)
    sel = mask != 0
    prm = solver.default_swing_params()
    for c in range(3):
        prm.kp[c] = KP[c]; prm.kd[c] = KD[c]
    for k in range(T):
        inp = _tick(rob, k, seed=13)
        if k == R:
            a.reset(_dev(mask))
            limb, eff = _state(a)
            assert (limb[:, sel] == 0).all() and (eff[:, sel] == 0).all()
            lb, eb = _state(b)
            assert np.array_equal(limb[:, ~sel], lb[:, ~sel]) and np.array_equal(eff[:, ~sel], eb[:, ~sel])
        _update(a, inp, oa)
        _update(b, inp, ob)
        torch.cuda.synchronize()
        la, ea = _state(a)
        lb, eb = _state(b)
        if k < R:
            assert np.array_equal(ea, eb) and np.array_equal(la, lb)
        else:
            assert np.array_equal(ea[:, ~sel], eb[:, ~sel]) and np.array_equal(la[:, ~sel], lb[:, ~sel]), k
            assert np.array_equal(oa.command.cpu().numpy()[:, ~sel], ob.command.cpu().numpy()[:, ~sel]), k
        if k == R:
            # first tick after the reset: the limb states evolve from INIT and the swing legs see qdd = 0
            from oracle import oracle as O
            want, _ = O.contact_fsm(inp["desired"], inp["footstep"], inp["contact"], inp["phase"], np.zeros((4, B), np.uint8))
            assert np.array_equal(la[:, sel], want[:, sel])
            d = {key: _dev(v) for key, v in inp.items()}
            swing = torch.zeros((12, B), dtype=torch.float64, device="cuda")
            solver.swing_leg_torques(d["q"], d["qd"], torch.zeros_like(d["qd"]), d["pt"], d["vt"], prm, swing)
            torch.cuda.synchronize()
            rows = ~_stance_rows(_support(la))
            rows[:, ~sel] = False
            assert rows.any() and _rel(ea[rows], swing.cpu().numpy()[rows]) <= 1e-12
    a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 37])
def test_host_entry_matches_device_entry_and_launch_count(solver, B):
    rob = _robots(B, seed=17)
    dev_c, host_c = capi.Controller(solver, B, _params()), capi.Controller(solver, B, _params())
    out = _Outs(B)
    for k in range(6):
        inp = _tick(rob, k, seed=17)
        d = {key: _dev(v) for key, v in inp.items()}
        n0 = solver.launches
        solver.solve_state(d["q"], d["pose"], d["twist"], d["tpose"], d["ttwist"], d["desired"], d["mu"], None, out.grf,
                           out.command, out.flags)
        n1 = solver.launches
        _update(dev_c, inp, out, d=d)
        n2 = solver.launches
        assert n2 - n1 == (n1 - n0) + 2
        c = lambda a: np.ascontiguousarray(a)  # noqa: E731
        cmd = np.zeros((12, B)); fl = np.zeros(B, np.uint32); grf = np.zeros((12, B))
        host_c.update_host(c(inp["q"]), c(inp["qd"]), c(inp["pose"]), c(inp["twist"]), c(inp["tpose"]), c(inp["ttwist"]),
                           c(inp["desired"]), c(inp["contact"]), c(inp["phase"]), cmd, fl, footstep=c(inp["footstep"]),
                           mu=c(inp["mu"]), ptarget=c(inp["pt"]), vtarget=c(inp["vt"]), grf=grf)
        torch.cuda.synchronize()
        assert np.array_equal(cmd, out.command.cpu().numpy()), k
        assert np.array_equal(fl, out.flags.cpu().numpy().view(np.uint32)), k
        assert np.array_equal(grf, out.grf.cpu().numpy()), k
        assert all(np.array_equal(x, y) for x, y in zip(_state(dev_c), _state(host_c))), k
    dev_c.close(); host_c.close()


@pytest.mark.gpu
def test_ros_balance_controller_demo_matches_the_restatement(qlb_built, oracle):
    demo = build.build_host_demo(which="controller_demo")
    r = subprocess.run([demo, "40"], capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [json.loads(x) for x in r.stdout.strip().splitlines()]
    head, ticks = lines[0], lines[1:]
    assert len(ticks) == 40
    m = legmodel.load_model("quadruped_model")
    M = oracle.model_array(m)
    st = CO.controller_init(1)
    col = lambda t, key: np.array(t[key], dtype=np.float64)[:, None]  # noqa: E731
    stances = set()
    for t in ticks:
        st, want = CO.controller_tick(oracle, m, M, st, col(t, "q"), col(t, "qd"), col(t, "pose"), col(t, "twist"), col(t, "tpose"),
                                      col(t, "ttwist"), np.array([t["desired"]], np.uint8), None, np.array([t["contact"]], np.uint8),
                                      col(t, "phase"), ptarget=col(t, "ptarget"), vtarget=col(t, "vtarget"), period=head["period"],
                                      effort_limit=head["effort_limit"], kp=head["kp"], kd=head["kd"])
        assert (t["flags"] & capi.FLAG_PARITY_MASK) == (int(want["flags"][0]) & capi.FLAG_PARITY_MASK), t["tick"]
        assert _rel_state(col(t, "command"), want["command"]) <= 1e-9, t["tick"]
        assert _rel_state(col(t, "grf"), want["grf"]) <= 1e-9, t["tick"]
        stances.add(int(want["stance"][0]))
    assert {0b0101, 0b1010} <= stances


@pytest.mark.gpu
def test_two_controllers_on_two_streams(solver):
    Bs, T = (20011, 9000), 8
    robs = [_robots(B, seed=21 + j) for j, B in enumerate(Bs)]
    inputs = [[{key: _dev(v) for key, v in _tick(robs[j], k, seed=21 + j).items()} for k in range(T)] for j in range(2)]

    def run(concurrent):
        ctrls = [capi.Controller(solver, B, _params()) for B in Bs]
        outs = [_Outs(B) for B in Bs]
        streams = [torch.cuda.Stream(), torch.cuda.Stream()] if concurrent else [None, None]
        torch.cuda.synchronize()
        res = [[], []]
        for k in range(T):
            for j in range(2):
                s = streams[j]
                if s is not None:
                    with torch.cuda.stream(s):
                        _update(ctrls[j], None, outs[j], stream=s.cuda_stream, d=inputs[j][k])
                        res[j].append((outs[j].command.clone(), outs[j].flags.clone(), outs[j].grf.clone()))
                else:
                    _update(ctrls[j], None, outs[j], d=inputs[j][k])
                    torch.cuda.synchronize()
                    res[j].append((outs[j].command.clone(), outs[j].flags.clone(), outs[j].grf.clone()))
        torch.cuda.synchronize()
        states = [_state(c) for c in ctrls]
        for c in ctrls:
            c.close()
        return [[tuple(x.cpu().numpy() for x in r) for r in res[j]] for j in range(2)], states

    serial, s_states = run(False)
    conc, c_states = run(True)
    for j in range(2):
        for k in range(T):
            assert all(np.array_equal(x, y) for x, y in zip(serial[j][k], conc[j][k])), (j, k)
        assert all(np.array_equal(x, y) for x, y in zip(s_states[j], c_states[j])), j
