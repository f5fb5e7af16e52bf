"""numpy restatement of one controller tick (qlb_controller_update, include/qlb.h): RosBalanceController::update
(ros_balance_controller.cpp:198-716) for B robots, chained from the CPU oracle's pieces (oracle/oracle.py: contact_fsm,
vmc_wrench, solve_wrench_batch, swing_leg_torques) plus what the tick adds around them - the ring of joint-velocity
samples, the stale-effort rule and the command clamp.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

TICK_RING = 11


def controller_init(B: int) -> dict:
    """Per-robot state after create / reset: limb states INIT (0), efforts zero, the joint-velocity ring (ring[0] oldest
    .. ring[10] newest) to be filled by the next sample."""
    return dict(limb_state=np.zeros((4, B), np.uint8), efforts=np.zeros((12, B)), ring=np.zeros((TICK_RING, 12, B)),
                refill=np.ones(B, bool))


def controller_reset(state: dict, mask=None) -> dict:
    """RosBalanceController::starting for the robots with mask[i] != 0 (None = all)."""
    s = {k: v.copy() for k, v in state.items()}
    sel = np.ones(s["refill"].shape[0], bool) if mask is None else np.asarray(mask) != 0
    s["limb_state"][:, sel] = 0
    s["efforts"][:, sel] = 0.0
    s["refill"][sel] = True
    return s


def ring_push(state: dict, qd):
    """The ring after this tick's sample, and the oldest sample the swing legs difference against."""
    qd = np.asarray(qd, dtype=np.float64)
    ring = np.concatenate([state["ring"][1:], qd[None]])
    refill = state["refill"]
    ring[:, :, refill] = qd[None, :, refill]
    return ring, ring[0]


def merge(efforts, stance, flags, tau, swing):
    """Stance rows: the solve's torques when its status is OK (0) or NO_STANCE (1), else kept (RBC.cpp:418,455-458).
    Swing rows: the swing-leg torques unless one of the leg's three is non-finite."""
    eff = np.array(efforts, dtype=np.float64, copy=True)
    status = (np.asarray(flags) >> 24) & 7
    for leg in range(4):
        sl = slice(3 * leg, 3 * leg + 3)
        st = ((np.asarray(stance) >> leg) & 1).astype(bool)
        take = st & ((status == 0) | (status == 1))
        eff[sl, take] = tau[sl, take]
        sw = ~st & np.isfinite(swing[sl]).all(axis=0)
        eff[sl, sw] = swing[sl, sw]
    return eff


def controller_tick(O, model: dict, model_arr, state: dict, q, qd, pose, twist, tpose, ttwist, desired, footstep, contact,
                    phase, mu=None, normals=None, ptarget=None, vtarget=None, period=0.0025, effort_limit=300.0,
                    gravity=(0.0, -9.81, 0.0), acceleration_scale=0.5, kp=(0.0, 0.0, 0.0), kd=(0.0, 0.0, 0.0)):
    """One tick; O = the oracle module.  SoA arrays [C, B].  Returns (new state, dict(command, efforts, grf, tau, flags,
    stance, limb_state, qdd))."""
    q = np.asarray(q, dtype=np.float64); qd = np.asarray(qd, dtype=np.float64)
    pose = np.asarray(pose, dtype=np.float64)
    B = q.shape[1]
    ring, front = ring_push(state, qd)
    qdd = (qd - front) / (10.0 * period)
    limb, stance = O.contact_fsm(desired, footstep, contact, phase, state["limb_state"])
    wrench = np.stack([O.vmc_wrench(pose[:, i], twist[:, i], tpose[:, i], ttwist[:, i]) for i in range(B)], axis=1)
    sol = O.solve_wrench_batch(model_arr, q, pose[3:], wrench, stance, mu=mu, normals=normals)
    swing = O.swing_leg_torques(model, model_arr, q, qd, qdd, ptarget, vtarget, gravity, acceleration_scale, kp, kd)
    eff = merge(state["efforts"], stance, sol["flags"], sol["tau"], swing)
    new = dict(limb_state=limb, efforts=eff, ring=ring, refill=np.zeros(B, bool))
    out = dict(command=np.clip(eff, -effort_limit, effort_limit), efforts=eff, grf=sol["grf"], tau=sol["tau"],
               flags=sol["flags"], stance=stance, limb_state=limb, qdd=qdd)
    return new, out
