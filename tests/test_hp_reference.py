"""The 50-digit reference of tests/hp_reference.py against the CPU oracle, where the oracle is accurate (CPU tests).

At the default parameters (W = 1e-4) the oracle's FP64 Goldfarb-Idnani solve is accurate to ~1e-11, so there the two
must agree: this pins the restatement (frame, kinematics, QP, outputs, status rules) to the oracle's.  Away from the
defaults the oracle is not the judge.  Its primal Hessian A'SA + W I has condition number ~S|A|^2 / W, and its relative
force error against the certified 50-digit optimum of the same inputs grows as W goes down (300 C3 states, default S,
quadruped_model; the kernels solve the dual 6x6 system S^-1 + A W^-1 A' instead and are not limited by this):

    W                oracle median    oracle max
    1e-4 (default)   2.8e-12          9.2e-12
    1e-8             2.8e-8           9.4e-8
    1e-10            2.8e-6           1.2e-5
    1e-12            2.7e-4           1.0e-3

`sens` - the largest relative change of x* when every input is perturbed by a random relative +-2^-53 (four draws) - is
what a backward-stable solve may miss by.  Measured on the 96 C3 states of test_sensitivity_by_stance_count (largest
value per stance count; the FP32 column perturbs by 2^-24):

    stance legs   W = 1e-4: forces   torques    W = 1e-12: forces   torques    W = 1e-4, 2^-24: forces
    2             4.3e-16            1.3e-15    4.3e-16             1.3e-15    2.0e-7
    3             5.6e-16            2.1e-15    5.6e-16             2.1e-15    3.5e-7
    4             6.4e-16            2.0e-15    6.4e-16             2.0e-15    2.7e-7

It stays at rounding level on every stance count and does not grow on 2-leg stances as W goes down: the wrench map of
a diagonal pair has rank 5 for every input (two point forces exert no moment about the line through the feet), so
perturbed inputs keep that structure and the minimiser stays well conditioned.  The 1e-3 error of the oracle at
W = 1e-12 is its method, not the problem.  (What does grow as W goes down is the error of a method that rounds the
wrench map entry by entry, which breaks the rank-5 structure, and of the kernels' dual 6x6 solve: see
tests/test_solve_edges.py.)
"""
import numpy as np
import pytest

import hp_reference as H
from quadruped_locomotion_b200 import synth

STATE_KEYS = ("q", "quat", "wrench", "mask", "mu", "normals")


def _rel(a, b):
    """|a - b|_inf / |b|_inf per state (columns); 0 where both are zero."""
    d = np.abs(a - b).max(axis=0)
    n = np.abs(b).max(axis=0)
    return np.where(n > 0, d / np.where(n > 0, n, 1.0), d)


def _stack(refs, key):
    return np.stack([r[key] for r in refs], axis=1)


def _check_against_oracle(refs, orc, tol):
    status = np.array([r["status"] for r in refs])
    assert np.array_equal(status, (orc["flags"] >> 24) & 7)
    assert all(r["certified"] for r in refs)
    ok = status == 0
    for key in H.OUT_KEYS:
        assert _rel(orc[key][:, ok], _stack(refs, key)[:, ok]).max() <= tol, key
    bits = np.array([r["bits"] for r in refs])
    margin = np.array([r["margin"] for r in refs])
    mism = ((orc["flags"] & 0xFFFFF0) != bits) & ok
    assert not (mism & (margin > 1e-6)).any()


@pytest.mark.parametrize("name", ["quadruped_model", "simpledog"])
def test_frame_and_kinematics_match_the_oracle(oracle, models, name):
    """Foot position, Jacobian and gravity torques of every leg, and the friction frame of every stance leg, to 1e-14."""
    M = models[name]
    st = synth.make_states("C5", 24, start=5 << 10)
    st["q"][:, :8] += np.linspace(-3.0, 3.0, 8)       # joint angles over a full turn, not only the synthetic range
    for i in range(st["q"].shape[1]):
        raw = H._exact_inputs(st, i, H.Params(), M, np.float64)
        r, p, model = H._to_mp(raw, H.Params(), M)
        su = H.setup(r, p, model)
        assert su["status"] == 0
        qn = H._unit(r["quat"])
        R = H._quat_rot(*qn)
        gb = [float(-p["gravity"] * R[6 + c]) for c in range(3)]
        for leg in range(4):
            foot, jac, gt = oracle.leg_kinematics(M, leg, st["q"][3 * leg:3 * leg + 3, i], grav=gb)
            f2, J2, g2 = H.leg_kinematics(model[leg], r["q"][3 * leg:3 * leg + 3], [H._F(v) for v in gb])
            assert np.abs(np.array([float(v) for v in f2]) - foot).max() <= 1e-14 * max(1.0, np.abs(foot).max())
            assert np.abs(np.array([[float(v) for v in row] for row in J2]) - jac).max() <= 1e-14 * max(1.0, np.abs(jac).max())
            assert np.abs(np.array([float(v) for v in g2]) - gt).max() <= 1e-14 * max(1.0, np.abs(gt).max())
        qp = oracle.assemble(M, st["q"][:, i], st["quat"][:, i], st["wrench"][:, i], st["mask"][i], st["mu"][:, i], st["normals"][:, i])
        ns = qp["ns"]
        for k in range(ns):
            D = qp["D"]
            n_o = D[k, 3 * k:3 * k + 3]
            t1_o = (D[ns + 4 * k, 3 * k:3 * k + 3] - D[ns + 4 * k + 1, 3 * k:3 * k + 3]) / 2
            t2_o = (D[ns + 4 * k + 2, 3 * k:3 * k + 3] - D[ns + 4 * k + 3, 3 * k:3 * k + 3]) / 2
            E = np.array([[float(v) for v in e] for e in su["E"][k]])
            assert np.abs(E - np.array([n_o, t1_o, t2_o])).max() <= 1e-14


@pytest.mark.parametrize("name", ["quadruped_model", "simpledog"])
def test_matches_the_oracle_at_the_defaults_golden(golden, models, name):
    """The golden fixture (465 states of every kind: stance masks, bad inputs, friction-limited) against the oracle's
    committed outputs: status, certified KKT, forces / torques / net wrench to 1e-10, active rows where not degenerate."""
    st = {k: golden[k] for k in STATE_KEYS}
    refs = H.solve_batch(st, H.Params(), models[name], units=(), workers=H.default_workers())
    orc = dict(grf=golden[name + "_grf"], tau=golden[name + "_tau"], netwrench=golden[name + "_net"], flags=golden[name + "_flags"])
    _check_against_oracle(refs, orc, 1e-10)


@pytest.mark.parametrize("name", ["quadruped_model", "simpledog"])
def test_matches_the_oracle_at_the_defaults_c5(oracle, models, name):
    st = synth.make_states("C5", 96, start=77 << 10)
    refs = H.solve_batch(st, H.Params(), models[name], units=(), workers=H.default_workers())
    orc = oracle.solve_wrench_batch(models[name], st["q"], st["quat"], st["wrench"], st["mask"], mu=st["mu"], normals=st["normals"])
    _check_against_oracle(refs, orc, 1e-10)


def test_certificates(models):
    """Every OK result carries a KKT certificate at 1e-35 of its scale - also where no candidate was right and the
    reference's own active-set loop found the active set (here: no candidate at all, and a wrong one)."""
    st = synth.make_states("C3", 48, start=901)
    prm = H.Params(W=1e-12, fmin=25.0)
    work = H.jobs(st, prm, models["quadruped_model"], units=())
    wrong = np.full(48, sum(11 << (4 + 5 * leg) for leg in range(4)), np.uint32)   # F_min row and one friction row of each leg
    plain = [H.solve_state(st, i, prm, models["quadruped_model"], candidates=(), units=()) for i in range(48)]
    forced = [H.solve_state(st, i, prm, models["quadruped_model"], candidates=[("kernel", wrong[i])], units=()) for i in range(48)]
    cand = [r for part in H.run_jobs(work) for r in part]
    for a, b, c in zip(plain, forced, cand):
        assert a["certified"] and b["certified"] and c["certified"]
        assert a["how"] in ("loop", "status")
        assert a["bits"] == b["bits"] == c["bits"]
        if a["status"] == 0:
            assert a["margin"] >= -1e-35
            for key in H.OUT_KEYS:
                assert np.abs(a[key] - c[key]).max() <= 1e-15 * max(1e-300, np.abs(c[key]).max())


def test_sensitivity_by_stance_count(models):
    """The sens table of the module docstring: at rounding level for every stance count at W = 1e-4 and W = 1e-12."""
    st = synth.make_states("C3", 96, start=11)
    ns = np.array([bin(int(m)).count("1") for m in st["mask"]])
    rows = {}
    for W in (1e-4, 1e-12):
        refs = H.solve_batch(st, H.Params(W=W), models["quadruped_model"], units=(H.U64, H.U32), workers=H.default_workers())
        for n in (2, 3, 4):
            sel = [r for r, k in zip(refs, ns) if k == n]
            assert sel
            rows[W, n] = (max(r["sens"][H.U64]["grf"] for r in sel), max(r["sens"][H.U64]["tau"] for r in sel),
                          max(r["sens"][H.U32]["grf"] for r in sel))
    for (W, n), (sf, stq, sf32) in sorted(rows.items()):
        print(f"W = {W:g}, {n} stance legs: sens forces {sf:.1e}, torques {stq:.1e}; 2^-24: forces {sf32:.1e}")
        assert sf <= 1e-14 and stq <= 1e-14 and sf32 <= 1e-5


def test_the_oracle_is_not_the_judge_at_small_w(oracle, models):
    """Why the kernels are not held to the oracle at W = 1e-12: the oracle itself misses the certified optimum by more
    than 1e-5 (the W table of the module docstring)."""
    st = synth.make_states("C3", 64, start=11)
    prm = H.Params(W=1e-12)
    refs = H.solve_batch(st, prm, models["quadruped_model"], units=(), workers=H.default_workers())
    orc = oracle.solve_wrench_batch(models["quadruped_model"], st["q"], st["quat"], st["wrench"], st["mask"], mu=st["mu"],
                                    normals=st["normals"], params=prm.oracle(oracle))
    assert all(r["certified"] for r in refs)
    err = _rel(orc["grf"], _stack(refs, "grf"))
    print(f"oracle at W = 1e-12: median {np.median(err):.1e}, max {err.max():.1e}")
    assert err.max() > 1e-5
