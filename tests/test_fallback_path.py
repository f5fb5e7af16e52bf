"""The interior-point fallback behind the fused solve kernel (qlb_quad_kernel<..., 2>, launched by launch_single).

The fused kernel hands a state to the interior-point kernel only when its active-set rounds fail: a factorisation
failure, or QLB_DBAS_MAX_ROUNDS (40) rounds.  No known C2 / C3 / C5 state gets there, so with the shipped library the
fallback always finds an empty list, while the fused kernel has already written every hard state provisionally (the
unconstrained minimiser, status OK).  A fallback that missed a state, or wrote the wrong one, would go unnoticed.

These tests build two variants of the library with a smaller round limit (a compile-time macro; the kernel source is
unchanged) and load each in-process next to the shipped library (capi.Solver keeps the library it was created with):
  R1  QLB_DBAS_MAX_ROUNDS=1: every hard state that needs two or more rounds goes to the fallback (a dense list);
  R3  QLB_DBAS_MAX_ROUNDS=3: states parked in the stash after one or two rounds, resumed, then handed off (a sparse list).
The iteration field of the flags tells the two paths apart: a state finished by the rounds reports its round count, one
finished by the interior point its interior-point iterations, of which there are at least QLB_POLISH_MIN_IT = 2 before
the first polish (unless it converges first).  The LDL^T pivot-failure route into the fallback is not covered: no known
input reaches it."""
import contextlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from conftest import rel_err
from quadruped_locomotion_b200 import build, capi, synth
from test_controller import _Outs, _robots, _support, _rel_state, _stance_rows, _state, _tick, _update, _params
from test_gpu_parity import MIXED_TOL, TIGHT, _compare, _oracle

pytestmark = pytest.mark.gpu

B_BIG = 65536
OUT_KEYS = ("grf", "tau", "netwrench")


def _status(flags):
    return (flags >> 24) & 7


def _iters(flags):
    return flags >> 27


def _same(out, ref, sel):
    """Outputs and flags of the states `sel` bit-identical."""
    for k in OUT_KEYS:
        if out.get(k) is not None:
            assert np.array_equal(out[k][:, sel], ref[k][:, sel]), k
    assert np.array_equal(out["flags"][sel], ref["flags"][sel])


def _handed(ref_flags, limit):
    """States a build with round limit `limit` hands to the fallback: those the shipped build verified after more rounds."""
    return (_status(ref_flags) == 0) & (_iters(ref_flags) > limit)


@contextlib.contextmanager
def _with_params(solver, **kw):
    """Solver parameters changed for the duration of a block."""
    saved = solver.get_params()
    p = solver.get_params()
    for k, v in kw.items():
        setattr(p, k, v)
    solver.set_params(p)
    try:
        yield solver
    finally:
        solver.set_params(saved)


def _variant_solver(path):
    """A Solver on the library at `path`; the module-level library of capi is left as it was."""
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(capi, "_lib", None)
        mp.setattr(capi, "LIB_PATH", path)
        s = capi.Solver("quadruped_model")
    s.set_limb_dynamics("quadruped_model")
    return s


@pytest.fixture(scope="module")
def variant_libs(qlb_built, tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device: the product path has no CPU fallback")
    d = tmp_path_factory.mktemp("variants")
    libs = {r: str(d / f"libqlb_r{r}.so") for r in (1, 3)}
    with ThreadPoolExecutor(len(libs)) as ex:   # two independent nvcc runs
        list(ex.map(lambda r: build.build(force=True, extra=[f"-DQLB_DBAS_MAX_ROUNDS={r}"], out=libs[r]), libs))
    return libs


@pytest.fixture(scope="module")
def shipped(qlb_built):
    s = capi.Solver("quadruped_model")
    s.set_limb_dynamics("quadruped_model")
    yield s
    s.close()


@pytest.fixture(scope="module")
def variants(variant_libs):
    ss = {r: _variant_solver(p) for r, p in variant_libs.items()}
    yield ss
    for s in ss.values():
        s.close()


@pytest.fixture(scope="module")
def r1(variants):
    return variants[1]


@pytest.fixture(scope="module")
def batches(shipped, oracle, models):
    """C3 and C5 batches of 65 536 states: inputs, the shipped build's outputs and the oracle's."""
    res = {}
    for cfg in ("C3", "C5"):
        st = synth.make_states(cfg, B_BIG, start=4099)
        res[cfg] = dict(st=st, out=shipped.solve_wrench_numpy(st), ref=_oracle(oracle, models["quadruped_model"], st))
    return res


# ------------------------------------------------------------------------------------------------------------ routing
@pytest.mark.parametrize("cfg", ["C3", "C5"])
def test_fallback_routing_is_the_predicted_set(shipped, r1, batches, cfg):
    """S2 = the states the shipped build verifies with status 0 after two or more rounds.  In R1 the iteration field is
    >= 2 on exactly S2; with ipm_max_iterations = 1 it is 1 on every state of S2 (each went through the interior point),
    while the shipped build gives the same bits with either limit (its fallback list stays empty)."""
    st, out = batches[cfg]["st"], batches[cfg]["out"]
    s2 = _handed(out["flags"], 1)
    print(f"{cfg}: {s2.sum()} of {B_BIG} states handed to the interior-point kernel in R1")
    assert s2.mean() >= 0.01
    o1 = r1.solve_wrench_numpy(st)
    assert np.array_equal(_iters(o1["flags"]) >= 2, s2)
    with _with_params(shipped, ipm_max_iterations=1), _with_params(r1, ipm_max_iterations=1):
        lim = shipped.solve_wrench_numpy(st)
        l1 = r1.solve_wrench_numpy(st)
    _same(lim, out, np.ones(B_BIG, bool))
    assert (_iters(l1["flags"][s2]) == 1).all()
    assert (_iters(l1["flags"]) <= 1).all()


# ------------------------------------------------------------------------------------------------------------ parity
@pytest.mark.parametrize("cfg", ["C3", "C5"])
@pytest.mark.parametrize("rounds", [1, 3])
def test_parity_through_the_fallback(variants, batches, cfg, rounds):
    """The variant against the oracle with the full bar; the states it finishes inside the fused kernel (round count of
    the shipped build <= the limit) bit-identical to the shipped build, iteration field included."""
    st, out, ref = batches[cfg]["st"], batches[cfg]["out"], batches[cfg]["ref"]
    o = variants[rounds].solve_wrench_numpy(st)
    handed = _handed(out["flags"], rounds)
    print(f"{cfg}: {handed.sum()} of {B_BIG} states handed to the interior-point kernel in R{rounds}")
    assert handed.any()
    _compare(o, ref)
    _same(o, out, ~handed)


# ------------------------------------------------------------------------------------------------------------ paths
def test_fp32_arrays_default_core(shipped, r1, oracle, models):
    """The <float, double> instantiation of the fallback: FP32 arrays, FP64 core."""
    st = synth.make_states("C3", 16384, start=31)
    ref = _oracle(oracle, models["quadruped_model"], st)
    base = shipped.solve_wrench_numpy(st, dtype=np.float32)
    out = r1.solve_wrench_numpy(st, dtype=np.float32)
    s2 = _handed(base["flags"], 1)
    assert s2.any() and np.array_equal(_iters(out["flags"]) >= 2, s2)
    _same(out, base, ~s2)
    assert rel_err(out["grf"].astype(np.float64), ref["grf"]).max() <= MIXED_TOL
    assert rel_err(out["tau"].astype(np.float64), ref["tau"]).max() <= 2 * MIXED_TOL
    assert np.array_equal(_status(out["flags"]), _status(ref["flags"]))
    mism = ((out["flags"] ^ ref["flags"]) & capi.FLAG_PARITY_MASK) != 0
    assert not (mism & (ref["margin"] > 1e-3)).any()


def test_state_mode(shipped, r1, oracle, models):
    """qlb_solve_state: the fallback recomputes the virtual-model wrench from the state arrays (its own load path)."""
    B = 20000
    st = synth.make_states("C3", B, start=2024)
    rng = np.random.default_rng(3)
    pose = np.concatenate([rng.normal(0, 0.05, (3, B)) + np.array([[0], [0], [0.45]]), st["quat"]])
    twist = rng.normal(0, 0.05, (6, B))
    tpose = np.concatenate([pose[:3] + rng.normal(0, 0.004, (3, B)), st["quat"]])
    ttwist = rng.normal(0, 0.05, (6, B))

    def run(s):
        o = dict(grf=np.zeros((12, B)), tau=np.zeros((12, B)), flags=np.zeros(B, np.uint32), netwrench=np.zeros((6, B)),
                 wout=np.zeros((6, B)))
        s.solve_state_host(st["q"], pose, twist, tpose, ttwist, st["mask"], st["mu"], st["normals"], o["grf"], o["tau"],
                           o["flags"], o["netwrench"], o["wout"])
        return o

    base, out = run(shipped), run(r1)
    assert np.array_equal(out["wout"], base["wout"])
    s2 = _handed(base["flags"], 1)
    print(f"state mode: {s2.sum()} of {B} states handed to the interior-point kernel in R1")
    assert s2.any() and np.array_equal(_iters(out["flags"]) >= 2, s2)
    _same(out, base, ~s2)
    for k in OUT_KEYS:
        assert rel_err(out[k], base[k]).max() <= TIGHT, k
    assert np.array_equal(_status(out["flags"]), _status(base["flags"]))
    _compare(out, _oracle(oracle, models["quadruped_model"], dict(st, wrench=base["wout"])))


def _mixed_indices(flags, B):
    """B state indices: two fallback states (S2 of R1), then another state, repeated - fallback states at even and odd
    positions of the batch.  Returns the indices and where the fallback states are."""
    s2, other = np.flatnonzero(_handed(flags, 1)), np.flatnonzero(~_handed(flags, 1))
    fb = np.arange(B) % 3 != 2
    idx = np.empty(B, np.int64)
    idx[fb] = s2[:fb.sum()]
    idx[~fb] = other[:(~fb).sum()]
    return idx, fb


@pytest.mark.parametrize("B", [1, 17, 1003])
def test_ragged_batches_cp_async_staging(r1, batches, oracle, models, B):
    """Ragged batches from arrays 8 bytes off a 16-byte boundary (stance masks 1 byte off): the fused kernel stages
    them with cp.async; the fallback reads them directly.  Same bits as from aligned arrays, and the oracle's answer."""
    src = batches["C5"]
    idx, fb = _mixed_indices(src["out"]["flags"], B)
    st = {k: np.ascontiguousarray(v[..., idx]) for k, v in src["st"].items()}
    dev = torch.device("cuda:0")

    def run(shift):
        def put(a):
            flat = torch.empty(a.size + shift, dtype=torch.from_numpy(a).dtype, device=dev)
            view = flat[shift:].view(a.shape)
            view.copy_(torch.from_numpy(a))
            return view
        d = {k: put(v) for k, v in st.items()}
        assert all((t.data_ptr() % 16 == 0) == (shift == 0) for k, t in d.items() if k != "mask")
        grf = torch.zeros((12, B), dtype=torch.float64, device=dev); tau = torch.zeros_like(grf)
        net = torch.zeros((6, B), dtype=torch.float64, device=dev); flags = torch.zeros(B, dtype=torch.int32, device=dev)
        r1.solve_wrench(d["q"], d["quat"], d["wrench"], d["mask"], d["mu"], d["normals"], grf, tau, flags, net)
        torch.cuda.synchronize()
        return dict(grf=grf.cpu().numpy(), tau=tau.cpu().numpy(), netwrench=net.cpu().numpy(),
                    flags=flags.cpu().numpy().view(np.uint32))

    off, aligned = run(1), run(0)
    _same(off, aligned, np.ones(B, bool))
    assert (_iters(off["flags"][fb]) >= 2).all() and (_iters(off["flags"][~fb]) <= 1).all()
    _compare(off, _oracle(oracle, models["quadruped_model"], st))


def test_bad_input_and_no_stance_next_to_fallback_states(r1, batches, oracle, models):
    src = batches["C5"]
    s2 = np.flatnonzero(_handed(src["out"]["flags"], 1))[:64]
    st = {k: np.ascontiguousarray(v[..., s2]) for k, v in src["st"].items()}
    clean = r1.solve_wrench_numpy(st)
    assert (_iters(clean["flags"]) >= 2).all() and (_status(clean["flags"]) == 0).all()
    st["q"][4, 3] = np.nan
    st["mask"][10] = 0
    out = r1.solve_wrench_numpy(st)
    status = _status(out["flags"])
    assert status[3] == 4 and status[10] == 1
    assert not out["grf"][:, [3, 10]].any() and not out["tau"][:, [3, 10]].any()
    ok = np.ones(64, bool); ok[[3, 10]] = False
    _same(out, clean, ok)
    _compare(out, _oracle(oracle, models["quadruped_model"], st))


def test_zero_minimal_force_is_order_independent(shipped, r1, oracle, models):
    """F_min = 0 on C5, the regime of the old wrong result of the interior-point pass (DESIGN.md 8).  The three-pass bars
    of test_nonpositive_minimal_force; a second call gives the same bits: with one state per warp no state's result may
    depend on the order of the list."""
    st = synth.make_states("C5", 8192, start=999)
    op = oracle.default_params()
    op.fmin = 0.0
    ref = _oracle(oracle, models["quadruped_model"], st, params=op)
    with _with_params(shipped, min_normal_force=0.0), _with_params(r1, min_normal_force=0.0):
        base = shipped.solve_wrench_numpy(st)
        out = r1.solve_wrench_numpy(st)
        again = r1.solve_wrench_numpy(st)
    s2 = _handed(base["flags"], 1)
    print(f"F_min = 0: {s2.sum()} of 8192 states handed to the interior-point kernel in R1")
    assert s2.any()
    status = _status(out["flags"])
    assert np.isin(status, (0, 3)).all()
    assert rel_err(out["grf"], ref["grf"]).max() <= 1e-6 and rel_err(out["tau"], ref["tau"]).max() <= 1e-6
    assert rel_err(out["grf"][:, status == 0], ref["grf"][:, status == 0]).max() <= 1e-8
    _same(again, out, np.ones(8192, bool))
    _same(out, base, ~s2)


# ------------------------------------------------------------------------------------------------------------ streams
def test_concurrent_streams_with_non_empty_lists(r1, oracle, models):
    """Ten solve calls in flight on ten streams, three rounds: every call owns its interior-point list (list2) and
    work counter, now that the lists hold entries."""
    dev = torch.device("cuda:0")
    jobs = []
    for k in range(10):
        B = 20000 + 777 * k
        st = synth.make_states("C3" if k % 2 == 0 else "C5", B, start=1000 * k)
        d = {n: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for n, v in st.items()}
        out = dict(grf=torch.zeros((12, B), dtype=torch.float64, device=dev), tau=torch.zeros((12, B), dtype=torch.float64, device=dev),
                   flags=torch.zeros(B, dtype=torch.int32, device=dev), net=torch.zeros((6, B), dtype=torch.float64, device=dev))
        jobs.append((st, d, out, torch.cuda.Stream()))
    torch.cuda.synchronize()
    for _ in range(3):
        for st, d, out, s in jobs:
            r1.solve_wrench(d["q"], d["quat"], d["wrench"], d["mask"], d["mu"], d["normals"], out["grf"], out["tau"],
                            out["flags"], out["net"], stream=s.cuda_stream)
    torch.cuda.synchronize()
    handed = 0
    for st, d, out, s in jobs:
        o = dict(grf=out["grf"].cpu().numpy(), tau=out["tau"].cpu().numpy(), flags=out["flags"].cpu().numpy().view(np.uint32),
                 netwrench=out["net"].cpu().numpy())
        _compare(o, _oracle(oracle, models["quadruped_model"], st))
        handed += int((_iters(o["flags"]) >= 2).sum())
    assert handed > 0


# ------------------------------------------------------------------------------------------------------------ MAX_ITER
@pytest.mark.parametrize("cfg", ["C3", "C5"])
def test_iteration_limit_gives_max_iter_status(r1, batches, cfg):
    """ipm_max_iterations = 1: the fallback states end in OK (the polish verified the pattern of the first iterate),
    MAX_ITER or UNVERIFIED; every other state is the shipped build's.  A state that is not verified still gets finite
    forces on its stance legs only, and the statistics kernel counts what the flags say."""
    st, out, ref = batches[cfg]["st"], batches[cfg]["out"], batches[cfg]["ref"]
    s2 = _handed(out["flags"], 1)
    dev = torch.device("cuda:0")
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in st.items()}
    grf = torch.zeros((12, B_BIG), dtype=torch.float64, device=dev); tau = torch.zeros_like(grf)
    net = torch.zeros((6, B_BIG), dtype=torch.float64, device=dev); flags = torch.zeros(B_BIG, dtype=torch.int32, device=dev)
    with _with_params(r1, ipm_max_iterations=1):
        r1.solve_wrench(d["q"], d["quat"], d["wrench"], d["mask"], d["mu"], d["normals"], grf, tau, flags, net)
        torch.cuda.synchronize()
        stats = r1.batch_stats(flags, d["wrench"], net)
    o = dict(grf=grf.cpu().numpy(), tau=tau.cpu().numpy(), netwrench=net.cpu().numpy(), flags=flags.cpu().numpy().view(np.uint32))
    status, iters = _status(o["flags"]), _iters(o["flags"])
    _same(o, out, ~s2)
    assert np.isin(status[s2], (0, 2, 3)).all()
    ok = s2 & (status == 0)
    for k in OUT_KEYS:
        assert rel_err(o[k][:, ok], ref[k][:, ok]).max() <= TIGHT, k
    bad = s2 & (status != 0)
    print(f"{cfg}: ipm_max_iterations = 1: {(status[s2] == 0).sum()} OK, {(status[s2] == 2).sum()} MAX_ITER, "
          f"{(status[s2] == 3).sum()} UNVERIFIED of {s2.sum()} fallback states")
    assert (status == 2).sum() >= 1
    assert np.isfinite(o["grf"][:, bad]).all() and np.isfinite(o["tau"][:, bad]).all()
    assert (iters[bad] == 1).all()
    for leg in range(4):
        swing = bad & (((st["mask"] >> leg) & 1) == 0)
        assert not o["grf"][3 * leg:3 * leg + 3, swing].any() and not o["tau"][3 * leg:3 * leg + 3, swing].any()
    assert o["grf"][:, bad].any(axis=0).all()
    assert stats[0] == B_BIG
    assert np.array_equal(stats[1:6], [(status == k).sum() for k in range(5)])
    assert stats[6] == iters.sum() and stats[30] == iters.max()


# ------------------------------------------------------------------------------------------------------------ tick
def test_controller_tick_on_the_fallback(shipped, r1, variant_libs):
    """The controller tick (state-mode solve inside) on R1 against the shipped build; then R1 with ipm_max_iterations = 1:
    a robot whose solve ended in MAX_ITER or UNVERIFIED keeps the previous tick's efforts on its stance rows while its
    swing rows are updated - the stale-effort rule on a status the GPU produced itself."""
    B, T = 4096, 20
    rob = _robots(B)
    lim = _variant_solver(variant_libs[1])
    try:
        with _with_params(lim, ipm_max_iterations=1):
            ctrl = {name: capi.Controller(s, B, _params()) for name, s in (("shipped", shipped), ("r1", r1), ("lim", lim))}
            outs = {name: _Outs(B) for name in ctrl}
            handed = stale = 0
            for k in range(T):
                inp = _tick(rob, k)
                d = {key: torch.from_numpy(np.ascontiguousarray(v)).cuda() for key, v in inp.items()}
                prev = _state(ctrl["lim"])[1]
                for name, c in ctrl.items():
                    _update(c, inp, outs[name], d=d)
                torch.cuda.synchronize()
                fl = {name: o.flags.cpu().numpy().view(np.uint32) for name, o in outs.items()}
                cmd = {name: o.command.cpu().numpy() for name, o in outs.items()}
                assert _rel_state(cmd["r1"], cmd["shipped"]) <= 1e-9, k
                assert np.array_equal(_status(fl["r1"]), _status(fl["shipped"])), k
                handed += int(_handed(fl["shipped"], 1).sum())
                limb, eff = _state(ctrl["lim"])
                limb_s, eff_s = _state(ctrl["shipped"])
                assert np.array_equal(limb, limb_s), k
                rows = _stance_rows(_support(limb))
                failed = np.isin(_status(fl["lim"]), (2, 3))
                stale += int(failed.sum())
                keep = rows & failed[None, :]
                assert np.array_equal(eff[keep], prev[keep]), k
                assert np.array_equal(eff[~rows], eff_s[~rows]), k          # swing rows: the swing-leg torques of this tick
                assert np.array_equal(cmd["lim"], np.clip(eff, -300.0, 300.0)), k
            print(f"controller: {handed} solves handed to the interior-point kernel in R1, {stale} left stale at ipm_max_iterations = 1")
            assert handed > 0 and stale > 0
            for c in ctrl.values():
                c.close()
    finally:
        lim.close()
