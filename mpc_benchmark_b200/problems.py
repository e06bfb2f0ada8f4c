"""Flat problem descriptors of the three reference OCPs (the constants of SURVEY App. C).

These builders produce exactly the `Config` / `Knot` / `Term` blocks that the aligator-compatible shim
(`mpc_benchmark_b200.api`) flattens out of the object graph the reference scripts build
(fulldynamic_talos.py:100-245, kinodynamic_talos.py:72-180, centroidal_talos.py:185-261); bench.py and
the tests use them directly to synthesise the BASELINE.json workloads.
"""
import ctypes as C

import numpy as np

from . import _abi
from .kinematics import center_of_mass, foot_placements
from .talos_like import half_sitting, talos_like_robot

GRAVITY = 9.81


def _set(arr, vals):
    vals = list(np.asarray(vals, float).reshape(-1))
    arr[: len(vals)] = vals


def base_setup(robot=None):
    rb = robot if robot is not None else talos_like_robot()
    q0 = half_sitting()
    x0 = np.concatenate([q0, np.zeros(_abi.NV)])
    lf, rf = foot_placements(rb, q0)
    com0, mass = center_of_mass(rb, q0)
    return rb, q0, x0, lf, rf, com0, mass


# ---------------------------------------------------------------- full dynamics
W_X_FULL = np.array(
    [0, 0, 0, 100, 100, 100] + [0.1] * 6 + [0.1] * 6 + [10, 10] + [1] * 4 + [1] * 4
    + [1] * 6 + [0.1, 0.1, 0.1, 0.1, 0.01, 0.01] * 2 + [10, 10] + [1] * 4 + [1] * 4,
    dtype=float,
)  # fulldynamic_talos.py:121-135


def full_config(rb, x0, lf, rf, T=100, dt=0.01, tol=1e-5, mu_init=1e-8, max_iters=100):
    c = _abi.Config()
    c.kind, c.T, c.dt = _abi.KIND_FULL, T, dt
    _set(c.x_ref, x0)
    _set(c.wx, W_X_FULL)
    _set(c.wu, [1e-4] * 22)  # full:136
    _set(c.w_cent, [0, 0, 10, 0, 0, 10])  # full:141-143
    _set(c.w_force, [1e-4] * 6)  # full:149-151
    _set(c.wx_term, W_X_FULL)  # full:235
    _set(c.w_cent_term, [0, 0, 10, 0, 0, 10])  # full:243
    _set(c.w_foot_term, [2000.0] * 6)  # full:244-245
    c.mu_fric, c.foot_L, c.foot_W = 0.8, 0.1, 0.075  # full:69-71
    _set(c.kp, [0, 0, 10, 0, 0, 0])  # full:93
    _set(c.kd, [50] * 6)  # full:94
    _set(c.contact_place[0], lf)  # full:83
    _set(c.contact_place[1], rf)
    c.mu_contact = 1e-10  # ProximalSettings(1e-9, 1e-10, 1), full:77
    c.tol, c.mu_init, c.max_iters, c.force_initial_condition = tol, mu_init, max_iters, 1
    return c


def full_knot(cs, lf_ref, rf_ref, f_ref_l, f_ref_r, w_lfrf=2000.0):
    """createStage(cs, ...) of fulldynamic_talos.py:153-232."""
    k = _abi.Knot()
    cl, cr = bool(cs[0]), bool(cs[1])
    k.cs[0], k.cs[1] = float(cl), float(cr)
    # force costs (full:187-201): both / left only / right only / none
    k.fcost[0] = 1.0 if cl else 0.0
    k.fcost[1] = 1.0 if cr else 0.0
    # pose-cost switches (full:179-182): w_RF on when the LEFT foot is in contact and vice versa
    _set(k.w_rf, [w_lfrf if cl else 0.0] * 6)
    _set(k.w_lf, [w_lfrf if cr else 0.0] * 6)
    _set(k.lf_ref, lf_ref)
    _set(k.rf_ref, rf_ref)
    _set(k.f_ref, np.concatenate([f_ref_l, f_ref_r]))
    return k


def full_contact_phases(T_ds=30, T_ss=80, total_steps=3, nsteps=100):
    """fulldynamic_talos.py:255-266."""
    ph = [[True, True]] * T_ds
    for _ in range(total_steps):
        ph += [[True, False]] * T_ss + [[True, True]] * T_ds + [[False, True]] * T_ss + [[True, True]] * T_ds
    ph += [[True, False]] * T_ss + [[True, True]] * T_ds
    ph += [[True, True]] * nsteps * 2
    return ph


def make_term(lf_ref, rf_ref, com_ref=None):
    t = _abi.Term()
    _set(t.lf_ref, lf_ref)
    _set(t.rf_ref, rf_ref)
    if com_ref is not None:
        _set(t.com_ref, com_ref)
        t.has_com_cstr = 1.0
    return t


def full_standing_problem(batch=1, T=100, robot=None, **kw):
    """Cold-solve problem of fulldynamic_talos.py:371-397: all-double-support standing horizon."""
    rb, q0, x0, lf, rf, com0, mass = base_setup(robot)
    cfg = full_config(rb, x0, lf, rf, T=T, **kw)
    f_half = mass * GRAVITY / 2.0
    fr = np.array([0, 0, f_half, 0, 0, 0.0])
    knot = full_knot([True, True], lf, rf, fr, fr)
    knots = (_abi.Knot * (batch * T))(*([knot] * (batch * T)))
    terms = (_abi.Term * batch)(*([make_term(lf, rf)] * batch))
    x0s = np.tile(x0, (batch, 1))
    xs = np.tile(x0, (batch, T + 1, 1))
    us = np.zeros((batch, T, 22))
    return dict(robot=rb, cfg=cfg, knots=knots, terms=terms, x0=x0s, xs=xs, us=us, lf=lf, rf=rf, com0=com0, mass=mass)


# ---------------------------------------------------------------- centroidal
def cent_config(rb, com0, mass, T=100, dt=0.01, tol=1e-5, mu_init=1e-8, max_iters=100):
    c = _abi.Config()
    c.kind, c.T, c.dt = _abi.KIND_CENT, T, dt
    _set(c.wu, [0.001] * 3 + [0.1] * 3 + [0.001] * 3 + [0.1] * 3)  # cent:193-200
    _set(c.w_com, [0, 0, 0])  # cent:187
    _set(c.w_linmom, [0.01, 0.01, 100])  # cent:188
    _set(c.w_linacc, [0.01] * 3)  # cent:189
    _set(c.w_angmom, [0.1, 0.1, 1000])  # cent:190
    _set(c.w_angacc, [0.01] * 3)  # cent:191
    _set(c.com_ref, com0)
    c.mass = mass
    c.mu_fric, c.foot_L, c.foot_W = 0.8, 0.1, 0.075  # cent:68-70
    c.tol, c.mu_init, c.max_iters, c.force_initial_condition = tol, mu_init, max_iters, 1
    return c


def cent_knot(cs, lf, rf, u_ref):
    """createStage(contact_state, LF_pose, RF_pose, ur) of centroidal_talos.py:208-247."""
    k = _abi.Knot()
    k.cs[0], k.cs[1] = float(bool(cs[0])), float(bool(cs[1]))
    _set(k.cpos, np.concatenate([np.asarray(lf)[9:12], np.asarray(rf)[9:12]]))
    _set(k.u_ref, u_ref)
    return k


def cent_standing_problem(batch=1, T=100, robot=None, **kw):
    """Cold-solve problem of centroidal_talos.py:252-288."""
    rb, q0, x0mb, lf, rf, com0, mass = base_setup(robot)
    cfg = cent_config(rb, com0, mass, T=T, **kw)
    u0 = np.zeros(12)
    u0[2] = u0[8] = mass * GRAVITY / 2.0  # cent:73-74
    # urefs[0] (cent:132-140 with i = 0, j = 0): un[2] = f_half, un[8] = f_half
    knot = cent_knot([True, True], lf, rf, u0)
    knots = (_abi.Knot * (batch * T))(*([knot] * (batch * T)))
    terms = (_abi.Term * batch)(*([make_term(lf, rf)] * batch))
    x0 = np.zeros(9)
    x0[:3] = com0
    return dict(robot=rb, cfg=cfg, knots=knots, terms=terms, x0=np.tile(x0, (batch, 1)), xs=np.tile(x0, (batch, T + 1, 1)),
                us=np.tile(u0, (batch, T, 1)), lf=lf, rf=rf, com0=com0, mass=mass)


# ---------------------------------------------------------------- synthetic walking batches (BASELINE.json configs 4-5)
def swing_bump(s, apex):
    """Vertical profile of the degree-8 Bezier swing curve of talos_utils.py:281-296 when start == final
    (x_forward = 0, fulldynamic_talos.py:352): control points 4 x start, start + apex, 4 x final."""
    return 70.0 * s ** 4 * (1.0 - s) ** 4 * apex


def perturbed_x0(rb, x0, rng, batch):
    """SURVEY 8d config 4: x0_i = x0 (+) delta_i, sigma = 0.01 (base pos), 0.02 (base ori, joints), 0.05 (velocities);
    samples violating the joint limits are rejected."""
    sig = np.concatenate([[0.01] * 3, [0.02] * 3, [0.02] * 22, [0.05] * 28])
    lo, hi = np.array(rb.q_lo[:]), np.array(rb.q_hi[:])
    out = np.zeros((batch, 57))
    from .kinematics import quat_to_R  # noqa: F401  (host-side helper only)

    for i in range(batch):
        while True:
            d = rng.normal(size=56) * sig
            x = x0.copy()
            # base: p += R * dp (first order is exact enough for the perturbation), quaternion (x) exp(dw)
            R = quat_to_R(x0[3:7])
            x[0:3] = x0[0:3] + R @ d[0:3]
            th = np.linalg.norm(d[3:6])
            dq = np.concatenate([np.sin(th / 2) * d[3:6] / th, [np.cos(th / 2)]]) if th > 0 else np.array([0, 0, 0, 1.0])
            qx, qy, qz, qw = x0[3:7]
            dx_, dy_, dz_, dw_ = dq
            x[3:7] = [qw * dx_ + qx * dw_ + qy * dz_ - qz * dy_, qw * dy_ - qx * dz_ + qy * dw_ + qz * dx_,
                      qw * dz_ + qx * dy_ - qy * dx_ + qz * dw_, qw * dw_ - qx * dx_ - qy * dy_ - qz * dz_]
            x[7:29] = x0[7:29] + d[6:28]
            x[29:57] = x0[29:57] + d[28:56]
            if np.all(x[7:29] > lo) and np.all(x[7:29] < hi):
                out[i] = x
                break
    return out


def random_schedule(rng, T, min_first_ds=30):
    """One random walking contact schedule of T knots.  Like the reference gait (fulldynamic_talos.py:248-266) it
    starts in double support for at least `min_first_ds` knots (the reference's T_ds = 30: the time the robot needs
    to shift its weight), then alternates single / double support with random durations and a random first swing
    foot.  Returns (phases, swing_pos, swing_len): contact pair, index inside the current swing and its length."""
    first = int(rng.integers(min_first_ds, min_first_ds + 31))
    t_ss = int(rng.integers(60, 101))
    t_ds = int(rng.integers(20, 41))
    left_first = bool(rng.integers(0, 2))
    phases, pos, length = [], [], []
    phases += [[True, True]] * first
    pos += [0] * first
    length += [1] * first
    stance_left = left_first
    while len(phases) < T:
        cs = [True, False] if stance_left else [False, True]
        phases += [cs] * t_ss
        pos += list(range(t_ss))
        length += [t_ss] * t_ss
        phases += [[True, True]] * t_ds
        pos += [0] * t_ds
        length += [1] * t_ds
        stance_left = not stance_left
    return phases[:T], pos[:T], length[:T]


def full_walk_batch(batch, seed=5, T=100, robot=None, swing_apex=0.15, perturb=True, stream_ticks=0, **kw):
    """BASELINE.json config 5: batch of full-dynamics MPC problems with RANDOM CONTACT SCHEDULES.
    Instance i gets its own gait (random initial double-support length, single/double-support durations and first
    swing foot; `random_schedule`), swing-foot references following the Bezier bump of talos_utils.py:281-296,
    a perturbed initial state (SURVEY 8d config 4) and the terminal CoM equality of the MPC loop
    (fulldynamic_talos.py:499-507).  Every stage uses force-reference index 0 as the reference does (full:363-366).
    `x0` is the perturbed ("measured") state of each instance, `x0_nominal` the unperturbed one; the cold start `xs`
    repeats the nominal state as the reference's first solve does (full:390-391).  An MPC tick warm-starts from the
    solution of the nominal problem and forces the measured state at knot 0: see `warm_tick_inputs`.
    With `stream_ticks` > 0 every gait is continued that many knots past the horizon and `stream(t)` returns the stage of
    each instance entering its horizon at closed-loop tick t (the `stages_full[t]` of fulldynamic_talos.py:496); the first T
    knots do not depend on `stream_ticks`."""
    rb, q0, x0, lf, rf, com0, mass = base_setup(robot)
    cfg = full_config(rb, x0, lf, rf, T=T, **kw)
    rng = np.random.default_rng(seed)
    f_half = mass * GRAVITY / 2.0
    fr = np.array([0, 0, f_half, 0, 0, 0.0])
    knots = (_abi.Knot * (batch * T))()
    terms = (_abi.Term * batch)()
    n_ds = 0
    tail = (_abi.Knot * (batch * stream_ticks))() if stream_ticks else None
    for i in range(batch):
        phases, pos, length = random_schedule(rng, T + stream_ticks)
        for j in range(T + stream_ticks):
            cs = phases[j]
            lref, rref = np.array(lf, float), np.array(rf, float)
            if cs != [True, True]:
                bump = swing_bump(pos[j] / float(length[j]), swing_apex)
                if cs[0]:
                    rref[11] += bump  # right foot swings
                else:
                    lref[11] += bump
            elif j < T:
                n_ds += 1
            if j < T:
                knots[i * T + j] = full_knot(cs, lref, rref, fr, fr)
            else:
                tail[(j - T) * batch + i] = full_knot(cs, lref, rref, fr, fr)
        com_final = np.array([(lf[9] + rf[9]) / 2, (lf[10] + rf[10]) / 2, com0[2]])
        terms[i] = make_term(lf, rf, com_final)
    x0s = perturbed_x0(rb, x0, rng, batch) if perturb else np.tile(x0, (batch, 1))
    x0n = np.tile(x0, (batch, 1))
    xs = np.repeat(x0n[:, None, :], T + 1, axis=1)
    us = np.zeros((batch, T, 22))
    out = dict(robot=rb, cfg=cfg, knots=knots, terms=terms, x0=x0s, x0_nominal=x0n, xs=xs, us=us, lf=lf, rf=rf, com0=com0, mass=mass,
               ds_fraction=n_ds / float(batch * T))
    if stream_ticks:
        out["stream"] = lambda t: (_abi.Knot * batch).from_buffer(tail, min(t, stream_ticks - 1) * batch * C.sizeof(_abi.Knot))
    return out


def warm_tick_inputs(prob, warm_xs):
    """Inputs of one closed-loop MPC tick (fulldynamic_talos.py:532-540): the previous solution as the warm start, with
    the MEASURED state of each instance (prob["x0"]) at knot 0 — the solver is run with force_initial_condition."""
    xs = np.array(warm_xs, dtype=float, copy=True)
    xs[:, 0, :] = prob["x0"]
    return xs


def sub_problem(prob, lo, hi):
    """Instances [lo, hi) of a batch problem (for bounded CPU-baseline samples and multi-GPU shards)."""
    T = prob["cfg"].T
    n = hi - lo
    knots = (_abi.Knot * (n * T))(*[prob["knots"][i] for i in range(lo * T, hi * T)])
    terms = (_abi.Term * n)(*[prob["terms"][i] for i in range(lo, hi)])
    out = dict(prob)
    out.update(knots=knots, terms=terms, x0=prob["x0"][lo:hi].copy(), xs=prob["xs"][lo:hi].copy(), us=prob["us"][lo:hi].copy())
    if "x0_nominal" in prob:
        out["x0_nominal"] = prob["x0_nominal"][lo:hi].copy()
    return out


def perturbed_robots(robot, batch, seed, mass=0.1, com=0.01, payload=0.0, payload_com=(0.0, 0.0, 0.25), payload_body=None, jplace=0.0):
    """`batch` copies of `robot` with randomised inertial parameters, for BatchSolver.set_instance_models (domain randomisation,
    robustness studies).  Per body, with `default_rng(seed)`:
      - mass and rotational inertia scaled together by one factor uniform in [1 - mass, 1 + mass] (the inertia stays physically valid);
      - CoM shifted by a normal offset of standard deviation `com` metres per axis;
      - a point payload uniform in [0, payload] kg at `payload_com` in `payload_body` (default: the Talos-shaped torso) merged into that
        body's mass, CoM and inertia about the new CoM (parallel-axis theorem).
    The kinematics (joint placements, sole frames) are left alone, so nominal x0 and sole references stay valid, unless `jplace` > 0:
    then every joint translation gets a normal offset of standard deviation `jplace` metres per axis.  Instance 0 is randomised too."""
    from .talos_like import JOINT_NAMES

    rng = np.random.default_rng(seed)
    pb = JOINT_NAMES.index("torso_2_joint") if payload_body is None else int(payload_body)
    out = []
    for _ in range(batch):
        rb = _abi.Robot.from_buffer_copy(robot)
        for b in range(robot.nb):
            s = rng.uniform(1.0 - mass, 1.0 + mass)
            rb.mass[b] = robot.mass[b] * s
            rb.inertia[b][:] = list(np.asarray(robot.inertia[b][:]) * s)
            rb.com[b][:] = list(np.asarray(robot.com[b][:]) + rng.normal(size=3) * com)
            if jplace > 0 and b > 0:
                rb.jplace[b][9:12] = list(np.asarray(robot.jplace[b][9:12]) + rng.normal(size=3) * jplace)
        p = rng.uniform(0.0, payload) if payload > 0 else 0.0
        if p > 0:
            m0, c0, r = rb.mass[pb], np.asarray(rb.com[pb][:]), np.asarray(payload_com, float)
            m1 = m0 + p
            c1 = (m0 * c0 + p * r) / m1
            shift = lambda mm, d: mm * (d @ d * np.eye(3) - np.outer(d, d))  # noqa: E731
            I1 = np.asarray(rb.inertia[pb][:]).reshape(3, 3) + shift(m0, c0 - c1) + shift(p, r - c1)
            rb.mass[pb], rb.com[pb][:], rb.inertia[pb][:] = m1, list(c1), list(I1.reshape(9))
        out.append(rb)
    return out


def lq_flops(n, m, c):
    """ALGORITHMIC dense-LQ FLOPs per knot (SURVEY 8d): backward + forward."""
    s = m + c
    back = (n ** 3 / 3 + 2 * n ** 3 + 4 * n ** 2) + (2 * n ** 3 + 2 * n * n * m) + (2 * n ** 3 + 2 * n * n * m + 2 * n * m * m + 2 * n * n + 2 * n * m) \
        + (s ** 3 / 3 + 2 * s * s * (1 + n)) + (2 * n * n * s + 2 * n * s)
    fwd = 2 * s * n + 2 * n * n + 2 * n * m
    return back + fwd


# ---------------------------------------------------------------- kinodynamics
W_X_KINO = 10.0 * np.array(
    [0, 0, 1000, 1000, 1000, 1000] + [0.1] * 6 + [0.1] * 6 + [1, 1000] + [1, 1, 10, 10] + [1, 1, 10, 10]
    + [0.1, 0.1, 0.1, 1000, 1000, 1000] + [1] * 6 + [1] * 6 + [0.1, 100] + [10] * 4 + [10] * 4,
    dtype=float,
)  # kinodynamic_talos.py:74-88


def kino_config(rb, x0, T=100, dt=0.01, tol=1e-5, mu_init=1e-8, max_iters=100):
    c = _abi.Config()
    c.kind, c.T, c.dt = _abi.KIND_KINO, T, dt
    _set(c.x_ref, x0)
    _set(c.wx, W_X_KINO)
    _set(c.wu, [0.001, 0.001, 0.01, 0.1, 0.1, 0.1] * 2 + [1e-4] * 22)  # kino:89-98
    _set(c.w_cent, [0, 0, 1, 0.1, 0.1, 10])  # kino:100-102
    _set(c.w_centder, [0, 0, 0, 0.1, 0.1, 0.1])  # kino:103-105
    c.mu_fric, c.foot_L, c.foot_W = 0.8, 0.1, 0.075  # kino:45,48-49
    c.tol, c.mu_init, c.max_iters, c.force_initial_condition = tol, mu_init, max_iters, 1
    return c


def kino_knot(cs, lf_ref, rf_ref, u_ref, w_lfrf=1e5):
    """createStage(contact_state, LF_pose, RF_pose, uforce) of kinodynamic_talos.py:117-173."""
    k = _abi.Knot()
    cl, cr = bool(cs[0]), bool(cs[1])
    k.cs[0], k.cs[1] = float(cl), float(cr)
    _set(k.w_rf, [w_lfrf if cl else 0.0] * 6)  # kino:145-148
    _set(k.w_lf, [w_lfrf if cr else 0.0] * 6)
    _set(k.lf_ref, lf_ref)
    _set(k.rf_ref, rf_ref)
    _set(k.u_ref, u_ref)
    return k


def kino_standing_problem(batch=1, T=100, robot=None, **kw):
    """Cold-solve problem of kinodynamic_talos.py:269-304: all-double-support, terminal CoM equality on com0."""
    rb, q0, x0, lf, rf, com0, mass = base_setup(robot)
    cfg = kino_config(rb, x0, T=T, **kw)
    f_half = mass * GRAVITY / 2.0
    uref0 = np.zeros(34)
    uref0[2] = uref0[8] = f_half  # urefs[0] (kino:205-212 with i = 0, j = 0)
    knot = kino_knot([True, True], lf, rf, uref0)
    knots = (_abi.Knot * (batch * T))(*([knot] * (batch * T)))
    ident = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0.0])
    terms = (_abi.Term * batch)(*([make_term(ident, ident, com0)] * batch))
    u_init = np.zeros(34)
    u_init[2] = u_init[8] = f_half  # u_ref = [f_ref, f_ref, 0] (kino:296-298)
    return dict(robot=rb, cfg=cfg, knots=knots, terms=terms, x0=np.tile(x0, (batch, 1)), xs=np.tile(x0, (batch, T + 1, 1)),
                us=np.tile(u_init, (batch, T, 1)), lf=lf, rf=rf, com0=com0, mass=mass)


# ---------------------------------------------------------------- reference-gait walking batches (all three models)
def _swap_feet_u(u, kind):
    u = np.array(u, float)
    if kind in (_abi.KIND_KINO, _abi.KIND_CENT):
        u[:6], u[6:12] = u[6:12].copy(), u[:6].copy()
    return u


def reference_horizon(kind, tick, mirror, lf, rf, com0, mass, T=100, stairs=False):
    """What the solver of ONE robot sees at MPC tick `tick` of the reference loop when the feet stand at (lf, rf): per-slot contact
    phase, index into `contact_phases` / `urefs`, swing-foot references (write-then-rotate order, SURVEY App. D.2) and the terminal
    CoM target (gait.GaitPlan; fulldynamic_talos.py:444-510, kinodynamic_talos.py:362-409, centroidal_talos.py:354-384,459).
    `stairs`: BASELINE configs[3] — every step goes x_forward = 0.3 m ahead and z_height = +0.10 m up (talos_utils.py:187-192 with the
    stair tread of bullet_robot.py:298-300), and the forward step is kept to the end of the gait."""
    from . import gait

    kw = dict(x_forward=0.3, z_height=0.10, keep_forward=True) if stairs else {}
    plan = gait.GaitPlan(kind, lf, rf, com0, nsteps=T, mirror=mirror, **kw)
    for _ in range(tick):
        plan.tick(sample=False)
    LF, RF, _, com_final = plan.tick(sample=True)
    return dict(phase=plan.h_phase, index=plan.h_index, lf=plan.h_lf, rf=plan.h_rf, com_final=com_final, lf_last=LF[-1], rf_last=RF[-1],
                lf_refs=LF, rf_refs=RF)


def walk_batch(kind, batch, seed=5, T=100, ticks=None, mirror=None, stairs=False, perturb=True, robot=None, **kw):
    """Batch of MPC problems along the REFERENCE gait of the given model (BASELINE.json configs[0]-[4] as concretised in SURVEY 8d):
    instance i sits at MPC tick `ticks[i]` (default: uniform over the whole contact-phase list, `default_rng(seed)`) of the
    schedule of fulldynamic_talos.py:256-266 / kinodynamic_talos.py:191-198 / centroidal_talos.py:108-116, mirrored (first swing
    with the other foot) with probability 1/2, with the swing references of talos_utils.footTrajectory from the nominal foot
    placements and a perturbed measured state (config 4 recipe).  Horizons hold single-support knots, moving references /
    contact positions and ramping force references; `x0_nominal`, `xs`, `us` are the reference's cold start."""
    from . import gait

    rb, q0, x0mb, lf, rf, com0, mass = base_setup(robot)
    rng = np.random.default_rng(seed)
    nph = len(gait.contact_phases(kind, T))
    ticks = rng.integers(0, nph, size=batch) if ticks is None else np.asarray(ticks, int)
    mirror = rng.integers(0, 2, size=batch).astype(bool) if mirror is None else np.asarray(mirror, bool)
    nx, n, m, nc = _abi.DIMS[kind]
    f_half = mass * GRAVITY / 2.0
    fr = np.array([0, 0, f_half, 0, 0, 0.0])
    if kind == _abi.KIND_FULL:
        cfg = full_config(rb, x0mb, lf, rf, T=T, **kw)
        x0n, u_init = x0mb, np.zeros(22)
    elif kind == _abi.KIND_KINO:
        cfg = kino_config(rb, x0mb, T=T, **kw)
        x0n = x0mb
        u_init = np.zeros(34)
        u_init[2] = u_init[8] = f_half
        urefs = gait.force_ramp_refs(kind, mass, 34, T)
    else:
        cfg = cent_config(rb, com0, mass, T=T, **kw)
        x0n = np.zeros(9)
        x0n[:3] = com0
        u_init = np.zeros(12)
        u_init[2] = u_init[8] = f_half
        urefs = gait.force_ramp_refs(kind, mass, 12, T)
    knots = (_abi.Knot * (batch * T))()
    terms = (_abi.Term * batch)()
    ident = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0.0])
    cache, n_ds = {}, 0
    for i in range(batch):
        key = (int(ticks[i]), bool(mirror[i]))
        if key not in cache:
            h = reference_horizon(kind, key[0], key[1], lf, rf, com0, mass, T=T, stairs=stairs)
            ks = []
            for j in range(T):
                cs = h["phase"][j]
                if kind == _abi.KIND_FULL:
                    ks.append(full_knot(cs, h["lf"][j], h["rf"][j], fr, fr))
                elif kind == _abi.KIND_KINO:
                    u = urefs[h["index"][j]]
                    ks.append(kino_knot(cs, h["lf"][j], h["rf"][j], _swap_feet_u(u, kind) if key[1] else u))
                else:
                    u = urefs[h["index"][j]]
                    # contact positions follow the references for ACTIVE contacts only (cent:374-384); others keep the construction value
                    lpos = h["lf"][j] if cs[0] else lf
                    rpos = h["rf"][j] if cs[1] else rf
                    ks.append(cent_knot(cs, lpos, rpos, _swap_feet_u(u, kind) if key[1] else u))
            if kind == _abi.KIND_FULL:
                term = make_term(h["lf_last"], h["rf_last"], h["com_final"])
            elif kind == _abi.KIND_KINO:
                term = make_term(ident, ident, h["com_final"])
            else:
                term = make_term(lf, rf)
            cache[key] = (ks, term, sum(1 for p in h["phase"] if p == [True, True]))
        ks, term, nds = cache[key]
        knots[i * T:(i + 1) * T] = ks
        terms[i] = term
        n_ds += nds
    x0n_b = np.tile(x0n, (batch, 1))
    if not perturb:
        x0s = x0n_b.copy()
    elif kind == _abi.KIND_CENT:
        x0s = x0n_b + rng.normal(size=(batch, 9)) * np.array([0.01] * 3 + [0.05 * mass] * 3 + [0.05] * 3)
    else:
        x0s = perturbed_x0(rb, x0mb, rng, batch)
    xs = np.repeat(x0n_b[:, None, :], T + 1, axis=1)
    us = np.tile(u_init, (batch, T, 1))
    return dict(robot=rb, cfg=cfg, knots=knots, terms=terms, x0=x0s, x0_nominal=x0n_b, xs=xs, us=us, lf=lf, rf=rf, com0=com0, mass=mass,
                ticks=ticks, mirror=mirror, ds_fraction=n_ds / float(batch * T))


def kino_walk_batch(batch, **kw):
    """BASELINE configs[1]: kinodynamic_talos.py flat-ground walk (x_forward 0.3, T_ds 20, T_ss 80)."""
    return walk_batch(_abi.KIND_KINO, batch, **kw)


def cent_walk_batch(batch, **kw):
    """BASELINE configs[0]: centroidal_talos.py flat-ground walk (x_forward 0.2, moving contact positions)."""
    return walk_batch(_abi.KIND_CENT, batch, **kw)


def full_reference_walk_batch(batch, **kw):
    """BASELINE configs[4]: full-dynamics batch with per-instance offsets into the schedule of fulldynamic_talos.py:256-266."""
    return walk_batch(_abi.KIND_FULL, batch, **kw)


def full_stairs_batch(batch=512, seed=4, **kw):
    """BASELINE configs[3]: stair climbing (x_forward 0.3, z_height +0.10 per step), perturbed initial states, default_rng(4)."""
    return walk_batch(_abi.KIND_FULL, batch, seed=seed, stairs=True, **kw)
