"""GPU parity tests (run on the B200 box): the fused sm_100a path, called through the C ABI, against the
CPU oracle on identical inputs.

Bars (BASELINE.json north_star / SURVEY.md 8d):
  forces and torques: max_i |x_gpu - x_oracle|_inf / max(1, |x_oracle|_inf) <= 1e-6 in FP64
  contact + active-set bits: bit-exact on non-degenerate instances; degenerate ones counted
"""
import numpy as np
import pytest
import torch

from conftest import rel_err
from quadruped_locomotion_b200 import capi, synth

pytestmark = pytest.mark.gpu

TOL = 1e-6          # the north-star bar
TIGHT = 1e-9        # what the kernel actually delivers; a regression guard
STATE_KEYS = ("q", "quat", "wrench", "mask", "mu", "normals")


@pytest.fixture(scope="module", params=["fused", "three_pass"])
def solver(qlb_built, request):
    """Every parity test runs on both kernel organisations (qlb_set_pipeline)."""
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device: the product path has no CPU fallback")
    s = capi.Solver("quadruped_model")
    s.set_pipeline(request.param)
    s.launches_per_call = 2 if request.param == "fused" else 3   # fused kernel + interior-point fallback, or the three passes
    yield s
    s.close()


@pytest.fixture(scope="module")
def solver_sd(qlb_built):
    s = capi.Solver("simpledog")
    yield s
    s.close()


def _oracle(O, M, st, **kw):
    return O.solve_wrench_batch(M, st["q"], st["quat"], st["wrench"], st["mask"], mu=st.get("mu"),
                                normals=st.get("normals"), want_margin=True, **kw)


def _compare(out, ref, tol=TIGHT, max_degenerate=1e-4):
    assert np.isfinite(out["grf"]).all() and np.isfinite(out["tau"]).all()
    assert rel_err(out["grf"], ref["grf"]).max() <= tol
    assert rel_err(out["tau"], ref["tau"]).max() <= tol
    if out.get("netwrench") is not None:
        assert rel_err(out["netwrench"], ref["netwrench"]).max() <= tol
    mism = ((out["flags"] ^ ref["flags"]) & capi.FLAG_PARITY_MASK) != 0
    # contact bits always exact
    assert np.array_equal(out["flags"] & 0xF, ref["flags"] & 0xF)
    # status must agree on ok / no-stance / bad-input
    so, sr = (out["flags"] >> 24) & 7, (ref["flags"] >> 24) & 7
    assert np.array_equal(so == 1, sr == 1) and np.array_equal(so == 4, sr == 4)
    assert (so[(sr == 0)] == 0).all()
    # active bits: exact except on (counted) near-degenerate instances
    assert mism.mean() <= max_degenerate
    if mism.any():
        assert (ref["margin"][mism] < 1e-6).all(), "active-set mismatch on a non-degenerate instance"
    return int(mism.sum())


def test_survey_known_answers(solver, oracle, models, kats):
    for k in kats["kats"]:
        st = dict(q=np.array(k["q"], float)[:, None], quat=np.array(k["quat"], float)[:, None],
                  wrench=np.array(k["wrench"], float)[:, None], mask=np.array([k["mask"]], np.uint8),
                  mu=np.full((4, 1), k["mu"]), normals=None)
        out = solver.solve_wrench_numpy(st)
        legs = [l for l in range(4) if (k["mask"] >> l) & 1]
        x = np.concatenate([out["grf"][3 * l:3 * l + 3, 0] for l in legs])
        np.testing.assert_allclose(x, k["x"], rtol=0, atol=1e-9 * max(1.0, np.abs(k["x"]).max()))
        np.testing.assert_allclose(x, k["survey_x"], rtol=0, atol=5e-8)
        # active rows in the reference's D-row numbering: ns F_min rows, then 4 per stance leg
        ns = len(legs)
        rows = []
        for slot, l in enumerate(legs):
            bits = (int(out["flags"][0]) >> (4 + 5 * l)) & 31
            if bits & 1:
                rows.append(slot)
            rows += [ns + 4 * slot + r for r in range(4) if bits & (2 << r)]
        assert sorted(rows) == k["survey_active_rows"]
        assert (int(out["flags"][0]) >> 24) & 7 == 0


def test_golden_fixture(solver, solver_sd, golden):
    st = {k: golden[k] for k in STATE_KEYS}
    for name, s in (("quadruped_model", solver), ("simpledog", solver_sd)):
        out = s.solve_wrench_numpy(st)
        assert rel_err(out["grf"], golden[name + "_grf"]).max() <= TIGHT
        assert rel_err(out["tau"], golden[name + "_tau"]).max() <= TIGHT
        assert rel_err(out["netwrench"], golden[name + "_net"]).max() <= TIGHT
        assert np.array_equal(out["flags"] & capi.FLAG_PARITY_MASK, golden[name + "_flags"] & capi.FLAG_PARITY_MASK)


@pytest.mark.parametrize("cfg,B", [("C1", 1), ("C2", 65536), ("C3", 131072), ("C5", 131072)])
def test_parity_with_oracle(solver, oracle, models, cfg, B):
    st = synth.make_states(cfg, B)
    ref = _oracle(oracle, models["quadruped_model"], st)
    out = solver.solve_wrench_numpy(st)
    _compare(out, ref)
    assert rel_err(out["grf"], ref["grf"]).max() <= TOL  # the stated bar, for the record


def test_parity_simpledog(solver_sd, oracle, models):
    st = synth.make_states("C3", 32768, start=1 << 21)
    ref = _oracle(oracle, models["simpledog"], st)
    _compare(solver_sd.solve_wrench_numpy(st), ref)


def test_parity_with_reference_solver(solver, oracle, models):
    """Same check against the reference's own QuadProg++ (oracle/_ref), where it was built."""
    if not oracle.have_ref():
        pytest.skip("oracle/_ref not present")
    st = synth.make_states("C5", 32768, start=99)
    ref = oracle.solve_wrench_batch(models["quadruped_model"], st["q"], st["quat"], st["wrench"], st["mask"],
                                    mu=st["mu"], normals=st["normals"], solver=oracle.SOLVER_REF)
    out = solver.solve_wrench_numpy(st)
    assert rel_err(out["grf"], ref["grf"]).max() <= TIGHT
    assert rel_err(out["tau"], ref["tau"]).max() <= TIGHT


@pytest.mark.parametrize("B", [1, 2, 3, 15, 16, 17, 31, 33, 1000, 1001])
def test_ragged_batch_sizes(solver, oracle, models, B):
    st = synth.make_states("C5", B, start=31337)
    _compare(solver.solve_wrench_numpy(st), _oracle(oracle, models["quadruped_model"], st), max_degenerate=0.0)


def test_empty_batch(solver):
    z = np.zeros((12, 0))
    solver.solve_wrench_host(z, np.zeros((4, 0)), np.zeros((6, 0)), np.zeros(0, np.uint8), None, None,
                             z.copy(), z.copy(), np.zeros(0, np.uint32), None)


def test_all_stance_masks_and_defaults(solver, oracle, models):
    st = synth.make_states("C3", 64)
    st["mask"] = (np.arange(64) % 16).astype(np.uint8)
    st["mu"] = None
    st["normals"] = None
    ref = _oracle(oracle, models["quadruped_model"], st)
    out = solver.solve_wrench_numpy(st)
    _compare(out, ref, max_degenerate=0.0)
    nos = st["mask"] == 0
    assert (((out["flags"][nos] >> 24) & 7) == 1).all() and not out["grf"][:, nos].any() and not out["tau"][:, nos].any()
    for leg in range(4):
        swing = ((st["mask"] >> leg) & 1) == 0
        assert not out["grf"][3 * leg:3 * leg + 3, swing].any()
        assert not out["tau"][3 * leg:3 * leg + 3, swing].any()


def test_tilted_normals_and_per_leg_friction(solver, oracle, models):
    st = synth.make_states("C5", 4096, start=777777)
    rng = np.random.default_rng(5)
    n = rng.normal(0, 0.12, (4, 3, 4096))
    n[:, 2] = 1.0
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    st["normals"] = n.reshape(12, 4096)
    _compare(solver.solve_wrench_numpy(st), _oracle(oracle, models["quadruped_model"], st))


def test_friction_limited(solver, oracle, models):
    st = synth.make_states("C3", 8192, start=5)
    st["wrench"][0] += 350.0   # heavy heading force: most legs sit on the friction pyramid
    ref = _oracle(oracle, models["quadruped_model"], st)
    out = solver.solve_wrench_numpy(st)
    _compare(out, ref)
    nact = np.array([bin(int(f) >> 4 & 0xFFFFF).count("1") for f in out["flags"]])
    assert (nact >= 1).mean() > 0.8


def test_bad_inputs_are_flagged_and_isolated(solver, oracle, models):
    st = synth.make_states("C3", 64, start=11)
    clean = solver.solve_wrench_numpy(st)
    st["q"][4, 3] = np.nan
    st["quat"][1, 10] = np.inf
    st["wrench"][5, 20] = np.nan
    st["normals"][:, 30] = np.tile([0.0, 1.0, 0.0], 4)  # normal along base y for identity yaw? degenerate only if parallel
    st["quat"][:, 30] = [1.0, 0.0, 0.0, 0.0]            # identity attitude: n x e_y = 0 -> NaN tangent (CFD.cpp:303)
    ref = _oracle(oracle, models["quadruped_model"], st)
    out = solver.solve_wrench_numpy(st)
    status = (out["flags"] >> 24) & 7
    for i in (3, 10, 20, 30):
        assert status[i] == 4 and ((ref["flags"][i] >> 24) & 7) == 4
        assert not out["grf"][:, i].any() and not out["tau"][:, i].any()
    ok = np.ones(64, bool); ok[[3, 10, 20, 30]] = False
    assert np.array_equal(out["grf"][:, ok], clean["grf"][:, ok])
    assert np.array_equal(out["flags"][ok], clean["flags"][ok])


def test_negative_friction_is_infeasible_and_zero_friction_is_solved(solver, oracle, models):
    """mu < 0 on a stance leg: QLB_STATE_INFEASIBLE (5) like the oracle (the reference's solver returns +inf), outputs
    zero, neighbours untouched.  mu = 0: a frictionless contact is a valid QP (tangential force zero)."""
    st = synth.make_states("C3", 96, start=5)
    st["mask"][:] = 0xF
    clean = solver.solve_wrench_numpy(st)
    st["mu"][1, 7] = -0.2
    st["mu"][:, 40] = -1.0
    st["mu"][3, 60] = 0.0
    ref = _oracle(oracle, models["quadruped_model"], st)
    out = solver.solve_wrench_numpy(st)
    status = (out["flags"] >> 24) & 7
    for i in (7, 40):
        assert status[i] == 5 and ((ref["flags"][i] >> 24) & 7) == 5
        assert not out["grf"][:, i].any() and not out["tau"][:, i].any()
    assert status[60] == 0
    assert rel_err(out["grf"][:, 60:61], ref["grf"][:, 60:61]).max() <= TIGHT
    ok = np.ones(96, bool); ok[[7, 40, 60]] = False
    assert np.array_equal(out["grf"][:, ok], clean["grf"][:, ok]) and np.array_equal(out["flags"][ok], clean["flags"][ok])
    # a swing leg's friction coefficient is never looked at
    st2 = synth.make_states("C2", 64)
    st2["mu"][0] = np.where((st2["mask"] & 1) == 0, -5.0, st2["mu"][0])
    out2 = solver.solve_wrench_numpy(st2)
    assert (((out2["flags"] >> 24) & 7) == 0).all()


@pytest.mark.parametrize("fmin", [0.0, -25.0])
def test_nonpositive_minimal_force(solver, oracle, models, fmin):
    """F_min = 0 and F_min < 0 (which acts as 0: the friction rows imply n.f >= 0).  Forces against the oracle run
    with the same F_min; active bits only where the oracle's margin says the active set is well defined (a leg that
    is unloaded completely sits at the apex of its pyramid, a degenerate vertex)."""
    st = synth.make_states("C5", 8192, start=999)
    p = solver.get_params()
    try:
        p2 = solver.get_params()
        p2.min_normal_force = fmin
        solver.set_params(p2)
        op = oracle.default_params()
        op.fmin = fmin
        ref = _oracle(oracle, models["quadruped_model"], st, params=op)
        out = solver.solve_wrench_numpy(st)
        status = (out["flags"] >> 24) & 7
        if solver.launches_per_call == 2:
            assert (status == 0).all()              # the fused kernel's rounds verify every state, degenerate or not
        else:
            # the three-pass kernels end on their interior point for a leg at the apex of its pyramid (all four
            # friction rows tight at zero force): the forces are right, the active-set check cannot succeed
            assert np.isin(status, (0, 3)).all() and (status == 3).mean() < 0.05
        assert rel_err(out["grf"], ref["grf"]).max() <= 1e-6 and rel_err(out["tau"], ref["tau"]).max() <= 1e-6
        assert rel_err(out["grf"][:, status == 0], ref["grf"][:, status == 0]).max() <= 1e-8
        if fmin == 0.0:
            mism = ((out["flags"] ^ ref["flags"]) & capi.FLAG_PARITY_MASK) != 0
            assert (ref["margin"][mism] < 1e-6).all()
    finally:
        solver.set_params(p)


def test_parameter_bounds_are_enforced(solver):
    """Weights outside [1e-12, 1e12], S_i / W above 1e11, a negative default friction coefficient, NaN: qlb_set_params
    refuses them."""
    for field, val in (("ground_force_weight", 0.0), ("ground_force_weight", 1e13), ("friction_default", -0.1),
                       ("min_normal_force", float("nan")), ("ground_force_weight", float("nan")),
                       ("ground_force_weight", 1e-12), ("ground_force_weight", 9.9e-11)):
        p = solver.get_params()
        setattr(p, field, val)
        with pytest.raises(RuntimeError):
            solver.set_params(p)
    p = solver.get_params()
    p.wrench_weights[2] = 1e-13
    with pytest.raises(RuntimeError):
        solver.set_params(p)
    p = solver.get_params()
    p.wrench_weights[3] = 1e12      # S_i / W = 1e16
    with pytest.raises(RuntimeError):
        solver.set_params(p)
    assert solver.get_params().ground_force_weight == 1e-4   # the context keeps its parameters
    p = solver.get_params()
    p.ground_force_weight = 1e-10   # max S_i / W = 1e11: the bound itself is accepted
    solver.set_params(p)
    p.ground_force_weight = 1e-4
    solver.set_params(p)


def test_huge_joint_angles_are_bad_input(solver):
    st = synth.make_states("C3", 16)
    st["q"][5, 3] = 3e9
    out = solver.solve_wrench_numpy(st)
    status = (out["flags"] >> 24) & 7
    assert status[3] == 4 and (np.delete(status, 3) == 0).all() and np.isfinite(out["grf"]).all()


def test_tma_staging_and_cp_async_staging_agree(qlb_built):
    """The fused kernel stages its input rows with TMA tensor boxes when the arrays are 16-byte aligned and with
    cp.async otherwise (include/qlb.h takes any pointer).  The same states through both paths - the second time from
    arrays that start 8 bytes off a 16-byte boundary, stance masks 1 byte off - give the same bits."""
    B = 4096
    st = synth.make_states("C3", B, start=123)
    dev = torch.device("cuda:0")
    s = capi.Solver("quadruped_model")

    def run(shift):
        def put(a):
            flat = torch.empty(a.size + shift, dtype=torch.from_numpy(a).dtype, device=dev)
            view = flat[shift:].view(a.shape)
            view.copy_(torch.from_numpy(np.ascontiguousarray(a)))
            return view
        d = {k: put(v) for k, v in st.items()}
        assert all((t.data_ptr() % 16 == 0) == (shift == 0) for k, t in d.items() if k != "mask")
        grf = torch.zeros((12, B), dtype=torch.float64, device=dev); tau = torch.zeros_like(grf)
        net = torch.zeros((6, B), dtype=torch.float64, device=dev); flags = torch.zeros(B, dtype=torch.int32, device=dev)
        s.solve_wrench(d["q"], d["quat"], d["wrench"], d["mask"], d["mu"], d["normals"], grf, tau, flags, net)
        torch.cuda.synchronize()
        return grf.cpu().numpy(), tau.cpu().numpy(), flags.cpu().numpy(), net.cpu().numpy()

    a, b = run(0), run(1)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert ((a[2].view(np.uint32) >> 24) & 7 == 0).all()


def test_results_do_not_depend_on_the_launch_geometry(qlb_built, monkeypatch):
    """The fused kernel is persistent: how many boxes a warp takes - and with it how often hard states are parked in
    the shared-memory stash and resumed - depends on the number of resident CTAs.  The optimum does not: one CTA per SM
    (QLB_FUSED_BPS=1, read when the context is created) gives the same forces and the same flags as the default."""
    st = synth.make_states("C5", 65536, start=3)
    ref = capi.Solver("quadruped_model").solve_wrench_numpy(st)
    monkeypatch.setenv("QLB_FUSED_BPS", "1")
    out = capi.Solver("quadruped_model").solve_wrench_numpy(st)
    assert np.array_equal(out["flags"] & 0xFFFFFF, ref["flags"] & 0xFFFFFF)
    sc = np.maximum(1.0, np.abs(ref["grf"]).max(0))
    assert (np.abs(out["grf"] - ref["grf"]).max(0) / sc).max() <= 1e-10


def test_unit_vector_contract_of_quaternion_and_normals(solver, oracle, models):
    """The contact coordinates need a unit base quaternion and unit surface normals (QLB_STATE_BAD_INPUT in
    include/qlb.h): deviations at rounding level are renormalised - the result is the oracle's for the exact unit
    vectors - and anything beyond 1e-5 in |v|^2 is refused, neighbours untouched."""
    st = synth.make_states("C3", 64, start=77)
    st["mask"][:] = 0xF
    ref = _oracle(oracle, models["quadruped_model"], st)
    clean = solver.solve_wrench_numpy(st)
    pert = {k: v.copy() for k, v in st.items()}
    pert["quat"][:, 5] *= 1.0 + 2e-7           # what an FP32 round trip does to a unit quaternion
    pert["normals"][:, 9] *= 1.0 - 1.5e-7
    pert["quat"][:, 20] *= 1.01                # not a rotation any more
    pert["normals"][3:6, 33] *= 0.9            # leg 1's normal is not a unit vector
    out = solver.solve_wrench_numpy(pert)
    status = (out["flags"] >> 24) & 7
    assert status[20] == 4 and status[33] == 4 and not out["grf"][:, [20, 33]].any()
    ok = np.ones(64, bool); ok[[20, 33]] = False
    assert (status[ok] == 0).all()
    sc = np.maximum(1.0, np.abs(ref["grf"]).max(0))
    assert (np.abs(out["grf"] - ref["grf"]).max(0) / sc)[ok].max() <= 1e-9
    assert np.array_equal(out["flags"][ok] & 0xFFFFFF, ref["flags"][ok] & 0xFFFFFF)
    same = ok.copy(); same[[5, 9]] = False
    assert np.array_equal(out["grf"][:, same], clean["grf"][:, same])


def test_full_size_properties(solver, oracle, models):
    """BASELINE size (2^20): size-independent properties on the whole batch + oracle parity on a slice."""
    B = 1 << 20
    st = synth.make_states("C3", B)
    out = solver.solve_wrench_numpy(st)
    flags = out["flags"]
    status = (flags >> 24) & 7
    assert (status == 0).mean() > 0.99999
    ok = status == 0
    # (1) determinism / idempotence: a second run is bit-identical
    again = solver.solve_wrench_numpy(st)
    assert np.array_equal(out["grf"], again["grf"]) and np.array_equal(flags, again["flags"])
    # (2) batch-split invariance: solving a slice alone gives the same bits
    lo, hi = 333333, 333333 + 4097
    part = solver.solve_wrench_numpy({k: (None if v is None else np.ascontiguousarray(v[..., lo:hi])) for k, v in st.items()})
    assert np.array_equal(part["grf"], out["grf"][:, lo:hi]) and np.array_equal(part["flags"], flags[lo:hi])
    # (3) primal feasibility of every constraint in the reference's form, from the outputs alone
    R = synth.rot_from_quat(st["quat"])                 # (3,3,B) base->world
    n = R[2]                                            # R^T e_z : rows of R_bw -> third row
    ey = R[1]
    t1 = np.cross(n, ey, axis=0); t1 /= np.linalg.norm(t1, axis=0)
    t2 = np.cross(n, t1, axis=0); t2 /= np.linalg.norm(t2, axis=0)
    for leg in range(4):
        f = out["grf"][3 * leg:3 * leg + 3]
        stance = ((st["mask"] >> leg) & 1).astype(bool) & ok
        fn = (n * f).sum(0); f1 = (t1 * f).sum(0); f2 = (t2 * f).sum(0)
        scale = np.maximum(1.0, np.abs(out["grf"]).max(0))
        rows = np.stack([fn - 10.0, 0.6 * fn + f1, 0.6 * fn - f1, 0.6 * fn + f2, 0.6 * fn - f2])
        assert (rows[:, stance] >= -1e-9 * scale[stance]).all()
        # (4) an active bit means the row is tight
        for r in range(5):
            bit = ((flags >> (4 + 5 * leg + r)) & 1).astype(bool) & stance
            assert (np.abs(rows[r, bit]) <= 1e-8 * scale[bit]).all()
    # (5) net wrench output equals sum f and sum r x f recomputed from the force output
    net_f = out["grf"][0:3] + out["grf"][3:6] + out["grf"][6:9] + out["grf"][9:12]
    assert np.abs(net_f - out["netwrench"][:3]).max() <= 1e-9 * np.abs(net_f).max()
    # (6) oracle parity on a slice of the same batch
    sl = slice(500000, 500000 + 65536)
    sub = {k: (None if v is None else np.ascontiguousarray(v[..., sl])) for k, v in st.items()}
    ref = _oracle(oracle, models["quadruped_model"], sub)
    _compare({k: (None if v is None else v[..., sl]) for k, v in out.items()}, ref)


def test_device_pointer_api_and_stream(solver, oracle, models):
    B = 50000
    st = synth.make_states("C3", B, start=42)
    dev = torch.device("cuda:0")
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in st.items()}
    grf = torch.full((12, B), float("nan"), dtype=torch.float64, device=dev)
    tau = torch.full((12, B), float("nan"), dtype=torch.float64, device=dev)
    flags = torch.zeros(B, dtype=torch.int32, device=dev)
    net = torch.zeros((6, B), dtype=torch.float64, device=dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    before = solver.launches
    with torch.cuda.stream(side):
        solver.solve_wrench(d["q"], d["quat"], d["wrench"], d["mask"], d["mu"], d["normals"], grf, tau, flags, net,
                            stream=side.cuda_stream)
    side.synchronize()
    assert solver.launches == before + solver.launches_per_call
    out = dict(grf=grf.cpu().numpy(), tau=tau.cpu().numpy(), flags=flags.cpu().numpy().view(np.uint32),
               netwrench=net.cpu().numpy())
    ref = _oracle(oracle, models["quadruped_model"], st)
    _compare(out, ref)
    # statistics kernel against numpy
    s = solver.batch_stats(flags, d["wrench"], net)
    assert s[0] == B and s[1] == ((out["flags"] >> 24) & 7 == 0).sum()
    err = np.sqrt((np.array([1, 5, 1, 10, 10, 5.])[:, None] * (out["netwrench"] - st["wrench"]) ** 2).sum(0))
    assert abs(s[7] - err.sum()) <= 1e-9 * err.sum() and abs(s[29] - err.max()) <= 1e-12 * err.max()
    assert s[6] == (out["flags"] >> 27).sum() and s[30] == (out["flags"] >> 27).max()
    for leg in range(4):
        for r in range(5):
            assert s[8 + 5 * leg + r] == ((out["flags"] >> (4 + 5 * leg + r)) & 1).sum()


def test_leg_kinematics_kernel(solver, solver_sd, oracle, models):
    B = 4097
    st = synth.make_states("C3", B, start=9)
    dev = torch.device("cuda:0")
    q = torch.from_numpy(st["q"]).to(dev); quat = torch.from_numpy(st["quat"]).to(dev)
    for name, s in (("quadruped_model", solver), ("simpledog", solver_sd)):
        foot = torch.empty((12, B), dtype=torch.float64, device=dev)
        jac = torch.empty((36, B), dtype=torch.float64, device=dev)
        gt = torch.empty((12, B), dtype=torch.float64, device=dev)
        s.leg_kinematics(q, quat, foot, jac, gt)
        torch.cuda.synchronize()
        foot, jac, gt = foot.cpu().numpy(), jac.cpu().numpy(), gt.cpu().numpy()
        for i in range(0, B, 97):
            R = synth.rot_from_quat(st["quat"][:, i])
            g = R.T @ np.array([0, 0, -9.8])
            for leg in range(4):
                f, J, G = oracle.leg_kinematics(models[name], leg, st["q"][3 * leg:3 * leg + 3, i], grav=g)
                np.testing.assert_allclose(foot[3 * leg:3 * leg + 3, i], f, atol=1e-13)
                np.testing.assert_allclose(jac[9 * leg:9 * leg + 9, i].reshape(3, 3), J, atol=1e-13)
                np.testing.assert_allclose(gt[3 * leg:3 * leg + 3, i], G, atol=1e-11)


def test_state_mode_runs_the_vmc_prologue(solver, oracle, models):
    """qlb_solve_state = VirtualModelController::compute + computeForceDistribution in one kernel."""
    B = 20000
    st = synth.make_states("C3", B, start=2024)
    rng = np.random.default_rng(3)
    pose = np.concatenate([rng.normal(0, 0.05, (3, B)) + np.array([[0], [0], [0.45]]), st["quat"]])
    twist = rng.normal(0, 0.05, (6, B))
    tq = synth.quat_from_ypr(*(rng.normal(0, 0.02, (3, B)) + np.stack([
        np.arctan2(2 * (st["quat"][0] * st["quat"][3] + st["quat"][1] * st["quat"][2]),
                   1 - 2 * (st["quat"][2] ** 2 + st["quat"][3] ** 2)), np.zeros(B), np.zeros(B)])))
    tpose = np.concatenate([pose[:3] + rng.normal(0, 0.004, (3, B)), tq])
    ttwist = rng.normal(0, 0.05, (6, B))
    wref = np.stack([oracle.vmc_wrench(pose[:, i], twist[:, i], tpose[:, i], ttwist[:, i]) for i in range(B)], axis=1)
    grf = np.zeros((12, B)); tau = np.zeros((12, B)); flags = np.zeros(B, np.uint32); net = np.zeros((6, B)); wout = np.zeros((6, B))
    solver.solve_state_host(st["q"], pose, twist, tpose, ttwist, st["mask"], st["mu"], st["normals"], grf, tau, flags, net, wout)
    assert rel_err(wout, wref).max() <= 1e-11
    st2 = dict(st); st2["wrench"] = wref
    ref = _oracle(oracle, models["quadruped_model"], st2)
    _compare(dict(grf=grf, tau=tau, flags=flags, netwrench=net), ref)


def test_parameters_can_be_changed(solver, oracle, models):
    st = synth.make_states("C3", 4096, start=77)
    p = solver.get_params()
    try:
        p2 = solver.get_params()
        p2.min_normal_force = 25.0
        p2.ground_force_weight = 1e-3
        for i, v in enumerate((2, 3, 1, 8, 12, 4)):
            p2.wrench_weights[i] = v
        solver.set_params(p2)
        op = oracle.default_params()
        op.fmin = 25.0; op.W = 1e-3
        for i, v in enumerate((2, 3, 1, 8, 12, 4)):
            op.S[i] = v
        ref = _oracle(oracle, models["quadruped_model"], st, params=op)
        _compare(solver.solve_wrench_numpy(st), ref)
    finally:
        solver.set_params(p)


# ---------------------------------------------------------------- FP32 twins (BASELINE config C4)
# Stated tolerance of the _f32 entry points with the FP32 core (include/qlb.h).  FP32 arithmetic on a QP whose
# Hessian has condition number ~1e5 (W = 1e-4 against S |a|^2 ~ 10) cannot resolve the weakly determined
# internal-force directions better than cond * eps ~ 5e-3; the error lives in those directions only, so the
# achieved wrench, the feasibility and the objective value stay at FP32 rounding level.  Measured relative
# force error (65 536 states each):   median    90 %     99 %     99.9 %   max
#     C3 (60 % four-stance)           1.6e-7    3.2e-4   2.5e-3   2.3e-2   5.0e-2
#     C2 (two-leg stances only)       1.8e-4    5.4e-4   1.1e-3   1.7e-3   4.3e-3
#     C5 (perturbed pose / friction)  1.4e-7    3.0e-4   1.1e-2   3.6e-2   9.0e-2
F32_MEDIAN, F32_P90, F32_P99, F32_MAX = 5e-4, 2e-3, 2e-2, 0.2
F32_NET = 1e-2          # achieved wrench A x, relative
F32_FEAS = 1e-4         # constraint violation / force scale
F32_OBJ = 1e-4          # (f(x32) - f(x*)) / max(1, |f(x*)|); measured 9e-6
F32_SAME_FLAGS = 0.95   # fraction of states with identical active-row bits
MIXED_TOL = 5e-4        # FP32 arrays + kinematics, frame and QP in FP64: rounding of inputs, kinematics, outputs (measured 8e-5 forces,
                        # 1.5e-4 torques on C3; round 1, with the frame in FP32: 5e-4 / 1.2e-3)


def _f32_checks(out, ref, oracle, M, st, nsample=256):
    assert out["grf"].dtype == np.float32 and out["tau"].dtype == np.float32
    assert np.isfinite(out["grf"]).all() and np.isfinite(out["tau"]).all()
    so, sr = (out["flags"] >> 24) & 7, (ref["flags"] >> 24) & 7
    assert np.array_equal(so, sr), "status differs from the FP64 oracle"
    assert np.array_equal(out["flags"] & 0xF, ref["flags"] & 0xF)
    e = rel_err(out["grf"].astype(np.float64), ref["grf"])
    p50, p90, p99 = np.percentile(e, [50, 90, 99])
    assert p50 <= F32_MEDIAN and p90 <= F32_P90 and p99 <= F32_P99 and e.max() <= F32_MAX, (p50, p90, p99, e.max())
    et = rel_err(out["tau"].astype(np.float64), ref["tau"])
    assert np.percentile(et, 99) <= 2 * F32_P99 and et.max() <= 2 * F32_MAX
    assert rel_err(out["netwrench"].astype(np.float64), ref["netwrench"]).max() <= F32_NET
    same = ((out["flags"] ^ ref["flags"]) & capi.FLAG_PARITY_MASK) == 0
    assert same.mean() >= F32_SAME_FLAGS
    # feasibility and optimality of the FP32 answer in the FP64 problem, on a sample
    B = st["q"].shape[1]
    worst_feas, worst_obj = 0.0, 0.0
    for i in np.linspace(0, B - 1, nsample).astype(int):
        if sr[i] != 0:
            continue
        qp = oracle.assemble(M, st["q"][:, i], st["quat"][:, i], st["wrench"][:, i], st["mask"][i],
                             mu=None if st.get("mu") is None else st["mu"][:, i],
                             normals=None if st.get("normals") is None else st["normals"][:, i])
        slots = [3 * l + c for l in qp["legs"] for c in range(3)]
        x32 = out["grf"][slots, i].astype(np.float64)
        xs = ref["grf"][slots, i]
        scale = max(1.0, np.abs(xs).max())
        worst_feas = max(worst_feas, float((qp["d"] - qp["D"] @ x32).max() / scale))
        f = lambda x: 0.5 * x @ qp["G"] @ x + qp["g0"] @ x  # noqa: E731
        worst_obj = max(worst_obj, float((f(x32) - f(xs)) / max(1.0, abs(f(xs)))))
    assert worst_feas <= F32_FEAS, worst_feas
    assert worst_obj <= F32_OBJ, worst_obj


@pytest.mark.parametrize("cfg,B", [("C3", 32768), ("C2", 16384)])
def test_f32_twin_fp32_core_stated_tolerance(solver, oracle, models, cfg, B):
    st = synth.make_states(cfg, B)
    ref = _oracle(oracle, models["quadruped_model"], st)
    solver.set_f32_core(False)
    try:
        out = solver.solve_wrench_numpy(st, dtype=np.float32)
    finally:
        solver.set_f32_core(True)
    _f32_checks(out, ref, oracle, models["quadruped_model"], st)


@pytest.mark.parametrize("cfg,B", [("C3", 32768), ("C2", 16384), ("C5", 16384)])
def test_f32_twin_default_core(solver, oracle, models, cfg, B):
    """The default _f32 path: FP32 interface and kinematics, FP64 solver core."""
    st = synth.make_states(cfg, B, start=31)
    ref = _oracle(oracle, models["quadruped_model"], st)
    out = solver.solve_wrench_numpy(st, dtype=np.float32)
    assert out["grf"].dtype == np.float32
    assert rel_err(out["grf"].astype(np.float64), ref["grf"]).max() <= MIXED_TOL
    assert rel_err(out["tau"].astype(np.float64), ref["tau"]).max() <= 2 * MIXED_TOL
    assert np.array_equal((out["flags"] >> 24) & 7, (ref["flags"] >> 24) & 7)
    mism = ((out["flags"] ^ ref["flags"]) & capi.FLAG_PARITY_MASK) != 0
    assert not (mism & (ref["margin"] > 1e-3)).any()


def test_f32_device_pointers_ragged_and_bad_inputs(solver, oracle, models):
    B = 1003  # not a multiple of 8: the last warp has idle quads
    st = synth.make_states("C3", B, start=555)
    st["q"][3, 17] = np.nan
    st["wrench"][2, 400] = np.inf
    st["mask"][5] = 0
    ref = _oracle(oracle, models["quadruped_model"], st)
    dev = torch.device("cuda:0")
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in st.items()}
    d = {k: (v.float() if v.dtype == torch.float64 else v) for k, v in d.items()}
    grf = torch.full((12, B), 7.0, dtype=torch.float32, device=dev); tau = torch.full_like(grf, 7.0)
    flags = torch.zeros(B, dtype=torch.int32, device=dev); net = torch.zeros((6, B), dtype=torch.float32, device=dev)
    before = solver.launches
    solver.solve_wrench(d["q"], d["quat"], d["wrench"], d["mask"], d["mu"], d["normals"], grf, tau, flags, net,
                        stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert solver.launches == before + solver.launches_per_call
    fl = flags.cpu().numpy().view(np.uint32)
    status = (fl >> 24) & 7
    assert status[17] == 4 and status[400] == 4 and status[5] == 1
    g = grf.cpu().numpy()
    assert (g[:, [5, 17, 400]] == 0).all() and np.isfinite(g).all()
    ok = (status == 0)
    assert ok.sum() == B - 3
    e = rel_err(g[:, ok].astype(np.float64), ref["grf"][:, ok])
    assert e.max() <= MIXED_TOL


def test_f32_state_mode_follows_fp64(solver):
    """qlb_solve_state_f32 against qlb_solve_state on the same (FP32-representable) inputs."""
    B = 8192
    st = synth.make_states("C3", B, start=4242)
    rng = np.random.default_rng(5)
    pose = np.concatenate([rng.normal(0, 0.05, (3, B)) + np.array([[0], [0], [0.45]]), st["quat"]])
    twist = rng.normal(0, 0.05, (6, B))
    tpose = pose + np.concatenate([rng.normal(0, 0.004, (3, B)), np.zeros((4, B))])
    ttwist = rng.normal(0, 0.05, (6, B))
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)  # noqa: E731
    ins32 = [f32(a) for a in (st["q"], pose, twist, tpose, ttwist)]
    ins64 = [np.ascontiguousarray(a, dtype=np.float64) for a in ins32]
    mu32, nr32 = f32(st["mu"]), f32(st["normals"])
    o64 = dict(grf=np.zeros((12, B)), tau=np.zeros((12, B)), flags=np.zeros(B, np.uint32), net=np.zeros((6, B)), w=np.zeros((6, B)))
    o32 = dict(grf=np.zeros((12, B), np.float32), tau=np.zeros((12, B), np.float32), flags=np.zeros(B, np.uint32),
               net=np.zeros((6, B), np.float32), w=np.zeros((6, B), np.float32))
    solver.solve_state_host(*ins64, st["mask"], mu32.astype(np.float64), nr32.astype(np.float64), o64["grf"], o64["tau"],
                            o64["flags"], o64["net"], o64["w"])
    solver.solve_state_host(*ins32, st["mask"], mu32, nr32, o32["grf"], o32["tau"], o32["flags"], o32["net"], o32["w"])
    assert rel_err(o32["w"].astype(np.float64), o64["w"]).max() <= 1e-4   # virtual wrench: gains up to 1e4 on FP32 errors
    assert np.array_equal((o32["flags"] >> 24) & 7, (o64["flags"] >> 24) & 7)
    e = rel_err(o32["grf"].astype(np.float64), o64["grf"])
    print("f32 state mode vs f64: median %.2e p99 %.2e max %.2e" % (np.median(e), np.percentile(e, 99), e.max()))
    assert e.max() <= 1e-2    # state mode: the virtual wrench itself is computed in FP32 (gains up to 1e4 on FP32 errors)


def test_concurrent_streams_do_not_share_launch_slots(solver, oracle, models):
    """Several solve calls in flight on different streams (what the *_host pipeline does internally): every call
    owns its work counters and index lists."""
    dev = torch.device("cuda:0")
    streams = [torch.cuda.Stream() for _ in range(10)]
    jobs = []
    for k, s in enumerate(streams):
        B = 20000 + 777 * k
        st = synth.make_states("C3" if k % 2 == 0 else "C5", B, start=1000 * k)
        d = {n: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for n, v in st.items()}
        out = dict(grf=torch.zeros((12, B), dtype=torch.float64, device=dev), tau=torch.zeros((12, B), dtype=torch.float64, device=dev),
                   flags=torch.zeros(B, dtype=torch.int32, device=dev), net=torch.zeros((6, B), dtype=torch.float64, device=dev))
        jobs.append((st, d, out, s))
    torch.cuda.synchronize()
    for _ in range(3):   # three rounds of ten concurrent calls: more in flight than launch slots
        for st, d, out, s in jobs:
            solver.solve_wrench(d["q"], d["quat"], d["wrench"], d["mask"], d["mu"], d["normals"], out["grf"], out["tau"],
                                out["flags"], out["net"], stream=s.cuda_stream)
    torch.cuda.synchronize()
    for st, d, out, s in jobs:
        ref = _oracle(oracle, models["quadruped_model"], st)
        _compare(dict(grf=out["grf"].cpu().numpy(), tau=out["tau"].cpu().numpy(), flags=out["flags"].cpu().numpy().view(np.uint32),
                      netwrench=out["net"].cpu().numpy()), ref)


def test_api_misuse_returns_error_codes(solver):
    """The C ABI never throws and never dereferences a missing required array: int status codes instead
    (SURVEY 8b error convention)."""
    import ctypes as C
    lib, ctx = solver.lib, solver._ctx
    dev = torch.device("cuda:0")
    t = torch.zeros((12, 8), dtype=torch.float64, device=dev)
    m = torch.zeros(8, dtype=torch.uint8, device=dev)
    f = torch.zeros(8, dtype=torch.int32, device=dev)
    null = None
    INVALID, NOT_INIT = -1, lib.qlb_solve_wrench(None, 8, *([null] * 11))
    assert NOT_INIT < 0 and b"" != lib.qlb_strerror(NOT_INIT)
    # missing required arrays
    assert lib.qlb_solve_wrench(ctx, 8, null, t.data_ptr(), t.data_ptr(), m.data_ptr(), null, null, t.data_ptr(), t.data_ptr(),
                                f.data_ptr(), null, null) == INVALID
    assert lib.qlb_solve_wrench(ctx, 8, t.data_ptr(), t.data_ptr(), t.data_ptr(), m.data_ptr(), null, null, t.data_ptr(), t.data_ptr(),
                                null, null, null) == INVALID
    assert lib.qlb_solve_state(ctx, 8, t.data_ptr(), null, t.data_ptr(), t.data_ptr(), t.data_ptr(), m.data_ptr(), null, null,
                               t.data_ptr(), t.data_ptr(), f.data_ptr(), null, null, null) == INVALID
    assert lib.qlb_pack_robot_states(ctx, 8, null, null, null, null, null, null, null) == INVALID
    assert lib.qlb_set_f32_core(ctx, 7) == INVALID
    # an empty batch is a no-op, whatever the pointers
    assert lib.qlb_solve_wrench(ctx, 0, *([null] * 11)) == 0
    # invalid parameters are refused and leave the context usable
    p = solver.get_params()
    bad = solver.get_params()
    bad.ground_force_weight = 0.0
    assert lib.qlb_set_params(ctx, C.byref(bad)) == INVALID
    bad = solver.get_params()
    bad.wrench_weights[2] = -1.0
    assert lib.qlb_set_params(ctx, C.byref(bad)) == INVALID
    assert solver.get_params().ground_force_weight == p.ground_force_weight
    st = synth.make_states("C3", 64)
    out = solver.solve_wrench_numpy(st)
    assert (((out["flags"] >> 24) & 7) == 0).all()
