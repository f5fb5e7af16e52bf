"""A plain high-precision restatement of one wrench-mode solve (mpmath, 50 significant digits).  TEST INFRASTRUCTURE.

The raw double inputs of a state - joint angles, base quaternion, desired wrench, stance mask, friction coefficients,
surface normals - the parameters (S, W, F_min, gravity, default friction) and the leg-model table are taken as exact
values and everything is restated from them, none of it from the oracle's FP64 QP data (its G = A'SA + W I keeps only
three digits of W = 1e-12 next to entries of about 10):
  - quaternion and normals renormalised exactly; rotation R (base -> world); friction frame in base coordinates
    n = R' n_w, t1 = n x (R' e_y) normalised, t2 = n x t1 normalised (ContactForceDistribution.cpp:286-309);
  - leg forward kinematics, Jacobian and gravity torques from the qlb_leg_model table, every joint rpy turned into a
    rotation through the normalised quaternion (as rpy_to_rot and the oracle do);
  - the QP of the reference: minimise (Ax - b)'S(Ax - b)/2 + W|x|^2/2 subject to n.f >= F_min and (mu n +- t_c).f >= 0
    per stance leg, F_min <= 0 acting as 0.  It is written in contact coordinates y = (n.f, t1.f, t2.f) per leg; the
    frame is orthonormal to the working precision, so |x| = |y| and every row of D is one row of the contact form;
  - outputs grf (base frame), tau = G(q) - J'f on stance legs, netwrench = A x, and the status of include/qlb.h:
    BAD_INPUT before NO_STANCE before INFEASIBLE (mu < 0 on a stance leg) before OK.

The solve: candidate active sets (the kernel's flags when given, the oracle's) are solved as equality-constrained QPs
and accepted when their KKT conditions hold (slacks >= -1e-35 scale, multipliers >= -1e-35 scale); if none holds, a
plain dual active-set loop (the method of the fused kernel's rounds, tools/proto/rounds_proto.dbas) runs with 1e-40
tolerances and its result is certified the same way.  The certificate, not the algorithm, is what makes the result
trustworthy.

`sens` is the forward error the problem itself allows: the largest relative change of x* (and of tau*, netwrench*) when
every real input - q, quaternion, wrench, mu, normals, S, W, F_min, gravity, the model table - is perturbed independently
by a random relative +-unit, four times, the active set kept.  The bar of a kernel result is then
    |x_gpu - x*|_inf <= C (sens + u) |x*|_inf,    C = 256, u = unit roundoff of the interface type, no absolute floor.
"""
from __future__ import annotations

import os
import sys

import mpmath
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DPS = 50
MP = mpmath.MPContext()
MP.dps = DPS
_F = MP.mpf
ZERO, ONE = _F(0), _F(1)
CERT_TOL = _F(10) ** -35
LOOP_TOL = _F(10) ** -40
C_BAR = 256
U64, U32 = 2.0 ** -53, 2.0 ** -24
STATUS_OK, STATUS_NO_STANCE, STATUS_BAD_INPUT, STATUS_INFEASIBLE = 0, 1, 4, 5
OUT_KEYS = ("grf", "tau", "netwrench")


class Params:
    """The solve parameters the reference needs (the fields of qlb_params that reach a wrench-mode solve)."""

    def __init__(self, S=(1.0, 5.0, 1.0, 10.0, 10.0, 5.0), W=1e-4, fmin=10.0, gravity=9.8, mu_default=0.6):
        self.S, self.W, self.fmin, self.gravity, self.mu_default = tuple(float(s) for s in S), float(W), float(fmin), \
            float(gravity), float(mu_default)

    def apply(self, p):
        """Copy into a capi.Params (the library's parameter block)."""
        for i in range(6):
            p.wrench_weights[i] = self.S[i]
        p.ground_force_weight, p.min_normal_force, p.gravity, p.friction_default = self.W, self.fmin, self.gravity, self.mu_default
        return p

    def oracle(self, O):
        op = O.default_params()
        for i in range(6):
            op.S[i] = self.S[i]
        op.W, op.fmin, op.gravity = self.W, max(self.fmin, 0.0), self.gravity
        return op


# ------------------------------------------------------------------------------------------------ small exact helpers
def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def _dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def _unit(v):
    n = MP.sqrt(MP.fsum(c * c for c in v))
    return [c / n for c in v]


def _quat_rot(w, x, y, z):
    """Row-major R of a unit Hamilton quaternion (w, x, y, z)."""
    return [w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y),
            2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
            2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z]


def _rpy_rot(rpy):
    hr, hp, hy = rpy[0] / 2, rpy[1] / 2, rpy[2] / 2
    sr, cr, sp, cp, sy, cy = MP.sin(hr), MP.cos(hr), MP.sin(hp), MP.cos(hp), MP.sin(hy), MP.cos(hy)
    x = sr * cp * cy - cr * sp * sy
    y = cr * sp * cy + sr * cp * sy
    z = cr * cp * sy - sr * sp * cy
    w = cr * cp * cy + sr * sp * sy
    n = MP.sqrt(x * x + y * y + z * z + w * w)
    return _quat_rot(w / n, x / n, y / n, z / n)


def _mul(A, B):
    return [A[3 * r] * B[s] + A[3 * r + 1] * B[3 + s] + A[3 * r + 2] * B[6 + s] for r in range(3) for s in range(3)]


def _mv(A, v):
    return [A[3 * r] * v[0] + A[3 * r + 1] * v[1] + A[3 * r + 2] * v[2] for r in range(3)]


def _mtv(A, v):
    return [A[c] * v[0] + A[3 + c] * v[1] + A[6 + c] * v[2] for c in range(3)]


def _solve(H, r):
    """H z = r by Gaussian elimination with partial pivoting (H: list of rows; both are consumed)."""
    n = len(r)
    for j in range(n):
        p = max(range(j, n), key=lambda i: abs(H[i][j]))
        if H[p][j] == 0:
            raise ZeroDivisionError("singular reduced Hessian")
        if p != j:
            H[j], H[p] = H[p], H[j]
            r[j], r[p] = r[p], r[j]
        inv = 1 / H[j][j]
        for i in range(j + 1, n):
            f = H[i][j] * inv
            if f:
                Hi, Hj = H[i], H[j]
                for k in range(j + 1, n):
                    Hi[k] -= f * Hj[k]
                r[i] -= f * r[j]
    z = [ZERO] * n
    for j in range(n - 1, -1, -1):
        s = r[j]
        for k in range(j + 1, n):
            s -= H[j][k] * z[k]
        z[j] = s / H[j][j]
    return z


# ------------------------------------------------------------------------------------------------ kinematics
def leg_kinematics(model_row, q3, gb):
    """Foot position, Jacobian (J[a][j]: component a of column j) and gravity torques of one leg, exact.
    model_row: one row of oracle.model_array (xyz 12, rpy 12, mass 4, com 12) as exact numbers; gb: gravity in base."""
    xyz = [model_row[3 * k:3 * k + 3] for k in range(4)]
    rpy = [model_row[12 + 3 * k:15 + 3 * k] for k in range(4)]
    mass = model_row[24:28]
    com_l = [model_row[28 + 3 * k:31 + 3 * k] for k in range(4)]
    R = [ONE, ZERO, ZERO, ZERO, ONE, ZERO, ZERO, ZERO, ONE]
    p = [ZERO, ZERO, ZERO]
    z, pj, com = [], [], []
    for k in range(4):
        t = _mv(R, xyz[k])
        p = [p[a] + t[a] for a in range(3)]
        R = _mul(R, _rpy_rot(rpy[k]))
        if k < 3:
            z.append([R[2], R[5], R[8]])
            pj.append(list(p))
            c, s = MP.cos(q3[k]), MP.sin(q3[k])
            R = _mul(R, [c, -s, ZERO, s, c, ZERO, ZERO, ZERO, ONE])
        t = _mv(R, com_l[k])
        com.append([p[a] + t[a] for a in range(3)])
    J = [[ZERO] * 3 for _ in range(3)]
    gt = []
    for k in range(3):
        col = _cross(z[k], [p[a] - pj[k][a] for a in range(3)])
        for a in range(3):
            J[a][k] = col[a]
        acc = [ZERO, ZERO, ZERO]
        for l in range(k, 4):
            m = _cross([com[l][a] - pj[k][a] for a in range(3)], [mass[l] * gb[a] for a in range(3)])
            acc = [acc[a] + m[a] for a in range(3)]
        gt.append(-_dot(z[k], acc))
    return p, J, gt


# ------------------------------------------------------------------------------------------------ one state
def _is_bad(raw, mask):
    """BAD_INPUT under include/qlb.h, evaluated on the exact inputs."""
    q, quat, b, mu, nw = raw["q"], raw["quat"], raw["wrench"], raw["mu"], raw["normals"]
    if not all(np.isfinite(v) and abs(v) <= 1e6 for v in q):
        return True
    if not all(np.isfinite(v) for v in list(quat) + list(b)):
        return True
    if abs(sum(_F(v) ** 2 for v in quat) - 1) > _F(1e-5):
        return True
    for leg in range(4):
        if not (mask >> leg) & 1:
            continue
        n = nw[3 * leg:3 * leg + 3]
        if not all(np.isfinite(v) for v in n) or not np.isfinite(mu[leg]) or abs(sum(_F(v) ** 2 for v in n) - 1) > _F(1e-5):
            return True
    return False


def setup(raw, prm, model):
    """Exact QP data of one state.  raw: dict of exact inputs (lists), prm: dict S, W, fmin, gravity; model: 4 x 40.
    Returns dict(status, legs, E, foot, J, gtau, mu, b, S, W, fmin) (the QP part only when status is OK)."""
    mask = raw["mask"]
    legs = [l for l in range(4) if (mask >> l) & 1]
    if raw["bad"]:
        return dict(status=STATUS_BAD_INPUT, legs=legs)
    if not legs:
        return dict(status=STATUS_NO_STANCE, legs=legs)
    if any(raw["mu"][l] < 0 for l in legs):
        return dict(status=STATUS_INFEASIBLE, legs=legs)
    qn = _unit(raw["quat"])
    R = _quat_rot(*qn)
    g = prm["gravity"]
    gb = [-g * R[6 + c] for c in range(3)]
    eyb = [R[3], R[4], R[5]]
    E, foot, J, gtau = [], [], [], []
    for l in legs:
        n = _mtv(R, _unit(raw["normals"][3 * l:3 * l + 3]))
        t1 = _cross(n, eyb)
        if not any(t1):
            return dict(status=STATUS_BAD_INPUT, legs=legs)
        t1 = _unit(t1)
        t2 = _unit(_cross(n, t1))
        E.append([n, t1, t2])
        p, Jl, gl = leg_kinematics(model[l], raw["q"][3 * l:3 * l + 3], gb)
        foot.append(p); J.append(Jl); gtau.append(gl)
    fmin = prm["fmin"] if prm["fmin"] > 0 else ZERO
    # wrench map column of slot c of leg k: [e_c; r_k x e_c]
    cols = [[E[k][c] + _cross(foot[k], E[k][c]) for c in range(3)] for k in range(len(legs))]
    return dict(status=STATUS_OK, legs=legs, E=E, foot=foot, J=J, gtau=gtau, mu=[raw["mu"][l] for l in legs], b=raw["wrench"],
                S=prm["S"], W=prm["W"], fmin=fmin, cols=cols)


def eqp(su, ws):
    """Equality-constrained QP of the working set ws (per stance leg (a0, sg1, sg2): y_n pinned at F_min; y_c = sg_c mu y_n).
    Returns y (per leg), u (multipliers per leg slot), slacks (per leg, five rows), scales (force, gradient)."""
    ns = len(su["legs"])
    S, W, b, fmin = su["S"], su["W"], su["b"], su["fmin"]
    cols, mus = su["cols"], su["mu"]
    # y = P z + c: the free directions of each leg
    P, c = [], []
    for k in range(ns):
        a0, s1, s2 = ws[k]
        mu = mus[k]
        if a0:
            c.append([fmin, s1 * mu * fmin, s2 * mu * fmin])
        else:
            c.append([ZERO, ZERO, ZERO])
            P.append((k, [ONE, s1 * mu, s2 * mu]))
        if s1 == 0:
            P.append((k, [ZERO, ONE, ZERO]))
        if s2 == 0:
            P.append((k, [ZERO, ZERO, ONE]))
    # A P (6 x nz) and A c
    def amap(k, v):
        return [cols[k][0][r] * v[0] + cols[k][1][r] * v[1] + cols[k][2][r] * v[2] for r in range(6)]
    M = [amap(k, v) for k, v in P]
    Ac = [ZERO] * 6
    for k in range(ns):
        a = amap(k, c[k])
        Ac = [Ac[r] + a[r] for r in range(6)]
    res0 = [S[r] * (b[r] - Ac[r]) for r in range(6)]
    nz = len(P)
    H = [[ZERO] * nz for _ in range(nz)]
    rhs = [ZERO] * nz
    for i in range(nz):
        ki, vi = P[i]
        Mi = M[i]
        rhs[i] = sum(Mi[r] * res0[r] for r in range(6)) - W * _dot(vi, c[ki])
        for j in range(i + 1):
            kj, vj = P[j]
            h = sum(Mi[r] * S[r] * M[j][r] for r in range(6))
            if ki == kj:
                h += W * _dot(vi, vj)
            H[i][j] = H[j][i] = h
    z = _solve(H, rhs) if nz else []
    y = [list(ck) for ck in c]
    for (k, v), zi in zip(P, z):
        for a in range(3):
            y[k][a] += v[a] * zi
    # gradient g = A'S(Ay - b) + W y per leg (contact coordinates), its scale, and the multipliers
    Ay = [ZERO] * 6
    for k in range(ns):
        a = amap(k, y[k])
        Ay = [Ay[r] + a[r] for r in range(6)]
    r6 = [S[r] * (Ay[r] - b[r]) for r in range(6)]
    Sb = [S[r] * b[r] for r in range(6)]
    u, sl = [], []
    gs, fs = ZERO, abs(fmin)
    for k in range(ns):
        mu = mus[k]
        g = [sum(cols[k][cc][r] * r6[r] for r in range(6)) + W * y[k][cc] for cc in range(3)]
        gs = max(gs, max(abs(sum(cols[k][cc][r] * Sb[r] for r in range(6))) for cc in range(3)), max(abs(W * v) for v in y[k]))
        a0, s1, s2 = ws[k]
        u1 = -s1 * g[1] if s1 else ZERO
        u2 = -s2 * g[2] if s2 else ZERO
        u0 = g[0] - mu * (u1 + u2) if a0 else ZERO
        u.append([u0, u1, u2])
        yn, y1, y2 = y[k]
        m = mu * yn
        sl.append([yn - fmin, m + y1, m - y1, m + y2, m - y2])
        fs = max(fs, max(abs(v) for v in y[k]))
    return dict(y=y, u=u, slack=sl, fscale=fs, gscale=gs, ws=[tuple(w) for w in ws])


def _rows(ws_k):
    """The active rows (0..4) of one leg's working set."""
    a0, s1, s2 = ws_k
    return ([0] if a0 else []) + ([1] if s1 == -1 else [2] if s1 == 1 else []) + ([3] if s2 == -1 else [4] if s2 == 1 else [])


def certify(sol, tol=CERT_TOL):
    """KKT at the working precision: every slack and every multiplier of an active row >= -tol * its scale.
    Returns the margin: min over rows of max(slack / force scale, multiplier / gradient scale)."""
    fs = sol["fscale"] if sol["fscale"] > 0 else ONE
    gs = sol["gscale"] if sol["gscale"] > 0 else ONE
    margin = None
    ok = True
    for k, ws_k in enumerate(sol["ws"]):
        act = _rows(ws_k)
        for r in range(5):
            s = sol["slack"][k][r] / fs
            if r in act:
                slot = 0 if r == 0 else (1 if r <= 2 else 2)
                v = sol["u"][k][slot] / gs
                ok = ok and v >= -tol
            else:
                v = s
                ok = ok and s >= -tol
            margin = v if margin is None else min(margin, v)
    return ok, margin


def dual_active_set(su, max_rounds=200, tol=LOOP_TOL):
    """Plain dual active-set loop (block additions of every violated row, ratio test on the multipliers)."""
    ns = len(su["legs"])
    ws = [[0, 0, 0] for _ in range(ns)]
    cur = eqp(su, ws)
    y = [list(v) for v in cur["y"]]
    u = [[ZERO] * 3 for _ in range(ns)]
    full = True
    for _ in range(max_rounds):
        if full:
            fs = cur["fscale"] or ONE
            added = False
            for k in range(ns):
                mu = su["mu"][k]
                yn, y1, y2 = y[k]
                e = [yn - su["fmin"], mu * yn + y1, mu * yn - y1, mu * yn + y2, mu * yn - y2]
                if not ws[k][0] and e[0] < -tol * fs:
                    ws[k][0] = 1; added = True
                for slot, (rm, rp) in ((1, (1, 2)), (2, (3, 4))):
                    if ws[k][slot] == 0 and (e[rm] < -tol * fs or e[rp] < -tol * fs):
                        ws[k][slot] = -1 if e[rm] <= e[rp] else 1
                        added = True
            if not added:
                return cur
        nxt = eqp(su, ws)
        gs = nxt["gscale"] or ONE
        t, blk = ONE, []
        for k in range(ns):
            for slot, on in enumerate(ws[k]):
                if on and nxt["u"][k][slot] < -tol * gs:
                    tr = u[k][slot] / (u[k][slot] - nxt["u"][k][slot]) if u[k][slot] > 0 else ZERO
                    if tr < t:
                        t, blk = tr, [(k, slot)]
                    elif tr == t:
                        blk.append((k, slot))
        if not blk:
            y = [list(v) for v in nxt["y"]]
            u = [list(v) for v in nxt["u"]]
            cur = nxt
            full = True
        else:
            y = [[y[k][a] + t * (nxt["y"][k][a] - y[k][a]) for a in range(3)] for k in range(ns)]
            u = [[u[k][s] + t * (nxt["u"][k][s] - u[k][s]) for s in range(3)] for k in range(ns)]
            for k, slot in blk:
                ws[k][slot] = 0
                u[k][slot] = ZERO
            full = False
    return None


def dual_condition(su, ws):
    """Condition number of the kernels' 6x6 dual matrix N = S^-1 + sum over the free slots of v v' / (W |v|^2) for the
    working set ws (v: the slot's wrench-map column; a slot pinned by an active row has no column)."""
    N = [[(1 / su["S"][r] if r == c else ZERO) for c in range(6)] for r in range(6)]
    for k, (a0, s1, s2) in enumerate(ws):
        mu, cols = su["mu"][k], su["cols"][k]
        free = ([[ONE, s1 * mu, s2 * mu]] if not a0 else []) + ([[ZERO, ONE, ZERO]] if s1 == 0 else []) + \
            ([[ZERO, ZERO, ONE]] if s2 == 0 else [])
        for v in free:
            col = [cols[0][r] * v[0] + cols[1][r] * v[1] + cols[2][r] * v[2] for r in range(6)]
            w = 1 / (su["W"] * _dot(v, v))
            for r in range(6):
                for c in range(6):
                    N[r][c] += w * col[r] * col[c]
    ev = MP.eigsy(MP.matrix(N), eigvals_only=True)
    return float(max(ev) / min(ev))


def ws_from_flags(flags, legs):
    """Working set (per stance leg) from the active bits of a flags word; None when a pair has both bits set."""
    ws = []
    for l in legs:
        bits = (int(flags) >> (4 + 5 * l)) & 31
        if (bits & 6) == 6 or (bits & 24) == 24:
            return None
        ws.append((bits & 1, -1 if bits & 2 else (1 if bits & 4 else 0), -1 if bits & 8 else (1 if bits & 16 else 0)))
    return ws


def outputs(su, y):
    """grf [12], tau [12], netwrench [6] (exact) of the contact-coordinate forces y of the stance legs."""
    grf, tau, net = [ZERO] * 12, [ZERO] * 12, [ZERO] * 6
    for k, l in enumerate(su["legs"]):
        E = su["E"][k]
        f = [E[0][a] * y[k][0] + E[1][a] * y[k][1] + E[2][a] * y[k][2] for a in range(3)]
        for a in range(3):
            grf[3 * l + a] = f[a]
        J = su["J"][k]
        for j in range(3):
            tau[3 * l + j] = su["gtau"][k][j] - (J[0][j] * f[0] + J[1][j] * f[1] + J[2][j] * f[2])
        for r in range(6):
            net[r] += su["cols"][k][0][r] * y[k][0] + su["cols"][k][1][r] * y[k][1] + su["cols"][k][2][r] * y[k][2]
    return grf, tau, net


def _exact_inputs(st, i, prm: Params, model_arr, dtype):
    """The inputs of state i as exact numbers (FP32 arrays: the FP32-rounded values)."""
    rnd = (lambda v: float(np.float32(v))) if dtype == np.float32 else float
    mu = st.get("mu")
    nr = st.get("normals")
    raw = dict(q=[rnd(v) for v in st["q"][:, i]], quat=[rnd(v) for v in st["quat"][:, i]], wrench=[rnd(v) for v in st["wrench"][:, i]],
               mask=int(st["mask"][i]) & 0xF,
               mu=[rnd(v) for v in mu[:, i]] if mu is not None else [rnd(prm.mu_default)] * 4,
               normals=[rnd(v) for v in nr[:, i]] if nr is not None else [0.0, 0.0, 1.0] * 4)
    raw["bad"] = _is_bad(raw, raw["mask"])
    return raw


def _to_mp(raw, prm: Params, model_arr, pert=None):
    """Exact mp copies of the real inputs; pert: callable giving the relative perturbation of each value."""
    f = (lambda v: _F(v)) if pert is None else (lambda v: _F(v) * (1 + pert()))
    r = dict(raw)
    for k in ("q", "quat", "wrench", "mu", "normals"):
        r[k] = [f(v) for v in raw[k]]
    p = dict(S=[f(s) for s in prm.S], W=f(prm.W), fmin=f(prm.fmin), gravity=f(prm.gravity))
    model = [[f(v) for v in row] for row in model_arr]
    return r, p, model


def solve_state(st, i, prm: Params, model_arr, candidates=(), dtype=np.float64, units=(U64,), trials=4, seed=0):
    """Reference solve of state i of the SoA batch st.  candidates: flags words whose active bits are tried first.
    Returns dict(status, grf, tau, netwrench (float64 arrays), bits, margin, certified, how, sens {unit: {key: value}})."""
    raw = _exact_inputs(st, i, prm, model_arr, dtype)
    r, p, model = _to_mp(raw, prm, model_arr)
    su = setup(r, p, model)
    out = dict(status=su["status"], bits=0, margin=np.inf, certified=True, how="status", kappa=0.0, ns=len(su["legs"]),
               grf=np.zeros(12), tau=np.zeros(12), netwrench=np.zeros(6), sens={u: dict.fromkeys(OUT_KEYS, 0.0) for u in units})
    if su["status"] != STATUS_OK:
        return out
    sol, how = None, None
    tried = set()
    for name, fl in candidates:
        ws = ws_from_flags(fl, su["legs"])
        if ws is None or tuple(ws) in tried:
            continue
        tried.add(tuple(ws))
        s = eqp(su, ws)
        ok, m = certify(s)
        if ok:
            sol, how, margin = s, name, m
            break
    if sol is None:
        s = dual_active_set(su)
        if s is not None:
            ok, m = certify(s)
            if ok:
                sol, how, margin = s, "loop", m
    if sol is None:
        out.update(certified=False, how="none")
        return out
    grf, tau, net = outputs(su, sol["y"])
    exact = dict(grf=grf, tau=tau, netwrench=net)
    bits = 0
    for k, l in enumerate(su["legs"]):
        for row in _rows(sol["ws"][k]):
            bits |= 1 << (4 + 5 * l + row)
    out.update(bits=bits, margin=float(margin), how=how, **{k: np.array([float(v) for v in exact[k]]) for k in OUT_KEYS})
    out["mult"] = [[float(v) for v in uk] for uk in sol["u"]]
    out["kappa"] = dual_condition(su, sol["ws"])
    rng = np.random.default_rng([seed, i])
    for unit in units:
        sens = dict.fromkeys(OUT_KEYS, 0.0)
        for _ in range(trials):
            signs = iter(rng.choice([-1.0, 1.0], size=512))
            ru, pu, mu_ = _to_mp(raw, prm, model_arr, pert=lambda: _F(unit) * next(signs))
            sp = setup(ru, pu, mu_)
            if sp["status"] != STATUS_OK:
                continue
            g2, t2, n2 = outputs(sp, eqp(sp, sol["ws"])["y"])
            for key, new in zip(OUT_KEYS, (g2, t2, n2)):
                ref = exact[key]
                nrm = max(abs(v) for v in ref)
                if nrm > 0:
                    sens[key] = max(sens[key], float(max(abs(a - b) for a, b in zip(new, ref)) / nrm))
        out["sens"][unit] = sens
    return out


def _solve_chunk(args):
    st, idx, prm, model_arr, cand, dtype, units, trials, seed = args
    return [solve_state(st, i, prm, model_arr, cand[j], dtype, units, trials, seed) for j, i in enumerate(idx)]


def jobs(st, prm: Params, model_arr, kernel_flags=None, dtype=np.float64, units=None, trials=4, seed=0, chunk=64):
    """Work items for run_jobs: the states of the SoA batch st in chunks, with their candidate active sets (the kernel's
    flags when given, then the oracle's on the same - for FP32 arrays FP32-rounded - inputs)."""
    from oracle import oracle as O
    units = units if units is not None else ((U32,) if dtype == np.float32 else (U64,))
    B = st["q"].shape[1]
    ost = {k: (v if v is None or k == "mask" else np.asarray(v, dtype=dtype).astype(np.float64)) for k, v in st.items()}
    orc = O.solve_wrench_batch(model_arr, ost["q"], ost["quat"], ost["wrench"], ost["mask"], mu=ost.get("mu"),
                               normals=ost.get("normals"), params=prm.oracle(O), mu_default=float(np.asarray(prm.mu_default, dtype)))
    cand = [([("kernel", kernel_flags[i])] if kernel_flags is not None else []) + [("oracle", orc["flags"][i])] for i in range(B)]
    return [(st, list(range(a, min(B, a + chunk))), prm, model_arr, cand[a:a + chunk], dtype, units, trials, seed)
            for a in range(0, B, chunk)]


def run_jobs(work, workers=1):
    """Results of work items (jobs(...) lists concatenated), in order; workers > 1: a process pool."""
    if workers <= 1 or len(work) <= 1:
        return [_solve_chunk(w) for w in work]
    import multiprocessing
    from concurrent.futures import ProcessPoolExecutor
    with ProcessPoolExecutor(min(workers, len(work)), mp_context=multiprocessing.get_context("spawn")) as ex:
        return list(ex.map(_solve_chunk, work))


def solve_batch(st, prm: Params, model_arr, kernel_flags=None, dtype=np.float64, units=None, trials=4, seed=0, workers=1):
    """Reference results (solve_state dicts) of every state of the SoA batch st."""
    return [r for part in run_jobs(jobs(st, prm, model_arr, kernel_flags, dtype, units, trials, seed), workers) for r in part]


def default_workers():
    return max(1, min(32, len(os.sched_getaffinity(0))))


def bar_ratios(out, refs, u, sel=None, kappa_u=0.0):
    """Per family (grf, tau, netwrench) and state: |out - ref|_inf / ((sens + u + kappa_u kappa) |ref|_inf), for the states
    whose reference status is OK (sel: further restriction).  0 where both are exactly zero, inf where only the reference
    is.  kappa_u = 2^-53 adds the accuracy limit of the kernels' FP64 dual method (see test_solve_edges.py)."""
    res = {}
    idx = [i for i, r in enumerate(refs) if r["status"] == STATUS_OK and (sel is None or sel[i])]
    for key in OUT_KEYS:
        vals = []
        for i in idx:
            r = refs[i]
            ref = r[key]
            err = float(np.abs(np.asarray(out[key][:, i], dtype=np.float64) - ref).max())
            nrm = float(np.abs(ref).max())
            unit = next(iter(r["sens"]))
            den = (r["sens"][unit][key] + u + kappa_u * r["kappa"]) * nrm
            vals.append(err / den if den > 0 else (0.0 if err == 0 else np.inf))
        res[key] = np.array(vals)
    return idx, res
