"""Descriptor compiler: aligator-style object graph -> flat C-ABI blocks (SURVEY 8b "Binding layer").

Only the stage structures the reference scripts build are recognised (fulldynamic_talos.py:153-232, 234-245;
centroidal_talos.py:208-247; kinodynamic_talos.py:117-173); anything else raises with the offending component named.
Called on every setup()/run(), so every mutation made through `problem.stages[j]` is picked up (<= 100 knots x ~90 doubles: cheap).
"""
import numpy as np

from . import _abi, api
from . import pin as _pin


class FlatProblem:
    def __init__(self, robot, cfg, knots, terms, x0):
        self.robot, self.cfg, self.knots, self.terms, self.x0 = robot, cfg, knots, terms, x0


def _set(arr, vals):
    vals = list(np.asarray(vals, float).reshape(-1))
    arr[: len(vals)] = vals


def _diag(W, n, what):
    W = np.asarray(W, float)
    if W.ndim == 0:
        return np.full(n, float(W))
    if W.ndim == 1:
        d = W
    else:
        d = np.diag(W)
        if np.abs(W - np.diag(d)).max() > 0:
            raise NotImplementedError(f"{what}: only diagonal weight matrices are supported (every reference weight is diagonal)")
    if d.shape[0] != n:
        raise ValueError(f"{what}: weight has dimension {d.shape[0]}, expected {n}")
    return d


def _same(a, b, what):
    if not np.allclose(np.asarray(a, float), np.asarray(b, float), rtol=0, atol=0):
        raise NotImplementedError(f"{what} differs between stages; the flat descriptor keeps it global (SURVEY App. C)")


def _foot_index(model, frame_id=None, name=None):
    names = ["left_sole_link", "right_sole_link"]
    if name is None:
        name = model.frames[frame_id].name
    if name not in names:
        raise NotImplementedError(f"only the sole frames {names} are supported, got {name!r}")
    return names.index(name)


def _robot_from_model(model):
    return model.robot


# ---------------------------------------------------------------- full dynamics
def _flatten_full_stage(stage, G, first):
    """-> Knot; fills/validates the global dict G."""
    dyn = stage.dynamics
    if not isinstance(dyn, api.IntegratorSemiImplEuler) or not isinstance(dyn.differential_dynamics, api.MultibodyConstraintFwdDynamics):
        raise NotImplementedError("full-dynamics stage must use IntegratorSemiImplEuler(MultibodyConstraintFwdDynamics)")
    ode = dyn.differential_dynamics
    model = ode.space.model
    k = _abi.Knot()
    names = [cm.name for cm in ode.constraint_models]
    cs = ["left_sole_link" in names, "right_sole_link" in names]
    if len(names) != sum(cs):
        raise NotImplementedError(f"unsupported contact models {names}")
    k.cs[0], k.cs[1] = float(cs[0]), float(cs[1])
    nv, nu = model.nv, ode.nu
    B = np.eye(nv, nu, -6)
    if ode.actuation_matrix.shape != B.shape or np.abs(ode.actuation_matrix - B).max() > 0:
        raise NotImplementedError("actuation matrix must be eye(nv, nu, -6) (fulldynamic_talos.py:65)")
    glob = dict(dt=dyn.timestep, mu_contact=ode.prox_settings.mu)
    for cm in ode.constraint_models:
        f = _foot_index(model, name=cm.name)
        if cm.type != _pin.ContactType.CONTACT_6D or cm.reference_frame != _pin.LOCAL:
            raise NotImplementedError("contacts must be CONTACT_6D in the LOCAL frame (fulldynamic_talos.py:84-92)")
        glob[f"kp{f}"], glob[f"kd{f}"] = np.array(cm.corrector.Kp, float), np.array(cm.corrector.Kd, float)
        glob[f"place{f}"] = cm.joint2_placement.to12()
    seen_pose = [False, False]
    for key, c, wgt in stage.cost.items():
        if wgt != 1.0:
            raise NotImplementedError("CostStack component weights other than 1 are not supported")
        if isinstance(c, api.QuadraticStateCost):
            glob["x_ref"], glob["wx"] = c.target, _diag(c.weights, 2 * nv, "QuadraticStateCost")
        elif isinstance(c, api.QuadraticControlCost):
            _set(k.u_ref, c.target)
            glob["wu"] = _diag(c.weights, nu, "QuadraticControlCost")
        elif isinstance(c, api.QuadraticResidualCost):
            r = c.residual
            if isinstance(r, api.CentroidalMomentumResidual):
                if np.abs(r.ref).max() > 0:
                    raise NotImplementedError("CentroidalMomentumResidual reference must be zero")
                glob["w_cent"] = _diag(c.weights, 6, "centroidal momentum cost")
            elif isinstance(r, api.FramePlacementResidual):
                f = _foot_index(model, frame_id=r.frame_id)
                seen_pose[f] = True
                _set(k.w_lf if f == 0 else k.w_rf, _diag(c.weights, 6, "frame placement cost"))
                _set(k.lf_ref if f == 0 else k.rf_ref, r.ref.to12())
            elif isinstance(r, api.ContactForceResidual):
                f = _foot_index(model, name=r.contact_name)
                if not cs[f] and any(cs):
                    raise ValueError(f"ContactForceResidual on {r.contact_name} but the contact is not in the dynamics")
                k.fcost[f] = 1.0
                fr = list(k.f_ref)
                fr[6 * f: 6 * f + 6] = list(np.asarray(r.ref, float))
                k.f_ref[:] = fr
                glob["w_force"] = _diag(c.weights, 6, "contact force cost")
            else:
                raise NotImplementedError(f"unsupported residual in a full-dynamics cost: {type(r).__name__}")
        else:
            raise NotImplementedError(f"unsupported cost component {type(c).__name__}")
    # constraints
    for func, cset in zip(stage.constraints.funcs, stage.constraints.sets):
        if isinstance(func, api.ControlErrorResidual) and isinstance(cset, api.BoxConstraint):
            if np.abs(func.target).max() > 0:
                raise NotImplementedError("torque box must be centred on a zero ControlErrorResidual target")
            _same(cset.lower_limit, -cset.upper_limit, "torque limits (must be symmetric)")
            glob["tau_max"] = cset.upper_limit
        elif isinstance(func, api.SlicedResidual) and isinstance(func.base, api.StateErrorResidual) and isinstance(cset, api.BoxConstraint):
            if func.indices != list(range(6, nv)):
                raise NotImplementedError("joint-limit constraint must be StateErrorResidual[6:nv] (fulldynamic_talos.py:208)")
            # r = target (-) x with target = neutral: bounds are (-upper, -lower) (fulldynamic_talos.py:209)
            glob["q_hi"], glob["q_lo"] = -cset.lower_limit, -cset.upper_limit
        elif isinstance(func, api.MultibodyWrenchConeResidual) and isinstance(cset, api.NegativeOrthant):
            f = _foot_index(model, name=func.contact_name)
            if not cs[f] and any(cs):
                raise ValueError("wrench cone on a contact that is not in the dynamics")
            glob["cone"] = np.array([func.mu, func.half_length, func.half_width])
        else:
            raise NotImplementedError(f"unsupported stage constraint {type(func).__name__} / {type(cset).__name__}")
    for key, val in glob.items():
        if key in G:
            _same(G[key], val, key)
        else:
            G[key] = val
    G.setdefault("model", model)
    return k


def _flatten_full_term(problem, G):
    t = _abi.Term()
    model = G["model"]
    nv = model.nv
    wx_t, wc_t, wf_t = np.zeros(2 * nv), np.zeros(6), np.zeros(6)
    lf = rf = None
    for key, c, wgt in problem.term_cost.items():
        if isinstance(c, api.QuadraticStateCost):
            _same(c.target, G["x_ref"], "terminal state-cost target")
            wx_t = _diag(c.weights, 2 * nv, "terminal state cost")
        elif isinstance(c, api.QuadraticResidualCost) and isinstance(c.residual, api.CentroidalMomentumResidual):
            wc_t = _diag(c.weights, 6, "terminal centroidal cost")
        elif isinstance(c, api.QuadraticResidualCost) and isinstance(c.residual, api.FramePlacementResidual):
            f = _foot_index(model, frame_id=c.residual.frame_id)
            w = _diag(c.weights, 6, "terminal frame cost")
            if wf_t.any():
                _same(wf_t, w, "terminal foot-pose weights (left/right)")
            wf_t = w
            if f == 0:
                lf = c.residual.ref.to12()
            else:
                rf = c.residual.ref.to12()
        else:
            raise NotImplementedError(f"unsupported terminal cost component {type(c).__name__}")
    ident = _pin.SE3().to12()
    _set(t.lf_ref, lf if lf is not None else ident)
    _set(t.rf_ref, rf if rf is not None else ident)
    G["wx_term"], G["w_cent_term"], G["w_foot_term"] = wx_t, wc_t, wf_t
    if len(problem.term_constraints) > 1:
        raise NotImplementedError("at most one terminal constraint (CoM equality) is supported")
    for func, cset in zip(problem.term_constraints.funcs, problem.term_constraints.sets):
        if isinstance(func, api.CenterOfMassTranslationResidual) and isinstance(cset, api.EqualityConstraintSet):
            _set(t.com_ref, func.ref)
            t.has_com_cstr = 1.0
        else:
            raise NotImplementedError(f"unsupported terminal constraint {type(func).__name__}")
    return t


def _flatten_full(problem, tol, mu_init, max_iters):
    T = len(problem.stages)
    G = {}
    knots = (_abi.Knot * T)()
    for j, st in enumerate(problem.stages):
        knots[j] = _flatten_full_stage(st, G, j == 0)
    term = _flatten_full_term(problem, G)
    model = G["model"]
    rb = _abi.Robot.from_buffer_copy(_robot_from_model(model))
    if "tau_max" in G:
        _set(rb.tau_max, G["tau_max"])
    if "q_lo" in G:
        _set(rb.q_lo, G["q_lo"])
        _set(rb.q_hi, G["q_hi"])
    c = _abi.Config()
    c.kind, c.T, c.dt = _abi.KIND_FULL, T, G["dt"]
    _set(c.x_ref, G.get("x_ref", np.concatenate([_pin.neutral(model), np.zeros(model.nv)])))
    _set(c.wx, G.get("wx", np.zeros(2 * model.nv)))
    _set(c.wu, G.get("wu", np.zeros(22)))
    _set(c.w_cent, G.get("w_cent", np.zeros(6)))
    _set(c.w_force, G.get("w_force", np.zeros(6)))
    _set(c.wx_term, G["wx_term"])
    _set(c.w_cent_term, G["w_cent_term"])
    _set(c.w_foot_term, G["w_foot_term"])
    cone = G.get("cone", np.array([0.8, 0.1, 0.075]))
    c.mu_fric, c.foot_L, c.foot_W = cone
    for f in range(2):
        if f"kp{f}" in G:
            if "kp" in G:
                _same(G["kp"], G[f"kp{f}"], "Baumgarte Kp (left/right)")
            G["kp"], G["kd"] = G[f"kp{f}"], G[f"kd{f}"]
            _set(c.contact_place[f], G[f"place{f}"])
        else:
            _set(c.contact_place[f], _pin.SE3().to12())
    _set(c.kp, G["kp"])
    _set(c.kd, G["kd"])
    c.mu_contact = G["mu_contact"]
    c.tol, c.mu_init, c.max_iters, c.force_initial_condition = tol, mu_init, max_iters, 1
    terms = (_abi.Term * 1)(term)
    return FlatProblem(rb, c, knots, terms, np.array(problem.x0_init, float).reshape(1, -1))


# ---------------------------------------------------------------- centroidal
def _flatten_cent_stage(stage, G):
    dyn = stage.dynamics
    ode = dyn.differential_dynamics
    cmap = ode.contact_map
    if cmap.size != 2 or ode.force_size != 6:
        raise NotImplementedError("centroidal model: two 6-D contacts expected (centroidal_talos.py:40-44)")
    k = _abi.Knot()
    k.cs[0], k.cs[1] = float(bool(cmap.contact_states[0])), float(bool(cmap.contact_states[1]))
    _set(k.cpos, np.concatenate([np.asarray(cmap.contact_poses[0], float)[:3], np.asarray(cmap.contact_poses[1], float)[:3]]))
    glob = dict(dt=dyn.timestep, mass=ode.mass, gravity=ode.gravity)
    for key, c, wgt in stage.cost.items():
        if isinstance(c, api.QuadraticControlCost):
            _set(k.u_ref, c.target)
            glob["wu"] = _diag(c.weights, 12, "control cost")
        elif isinstance(c, api.QuadraticResidualCost):
            r, w = c.residual, _diag(c.weights, 3, f"cost {key!r}")
            if isinstance(r, api.CentroidalCoMResidual):
                glob["w_com"], glob["com_ref"] = w, r.ref
            elif isinstance(r, api.AngularMomentumResidual):
                glob["w_angmom"] = w
                if np.abs(r.ref).max() > 0:
                    raise NotImplementedError("momentum references must be zero")
            elif isinstance(r, api.LinearMomentumResidual):
                glob["w_linmom"] = w
                if np.abs(r.ref).max() > 0:
                    raise NotImplementedError("momentum references must be zero")
            elif isinstance(r, api.AngularAccelerationResidual):
                glob["w_angacc"] = w
                _check_cmap(r.contact_map, cmap)
            elif isinstance(r, api.CentroidalAccelerationResidual):
                glob["w_linacc"] = w
                _check_cmap(r.contact_map, cmap)
            else:
                raise NotImplementedError(f"unsupported residual in a centroidal cost: {type(r).__name__}")
        else:
            raise NotImplementedError(f"unsupported cost component {type(c).__name__}")
    cones = [False, False]
    for func, cset in zip(stage.constraints.funcs, stage.constraints.sets):
        if isinstance(func, api.CentroidalWrenchConeResidual) and isinstance(cset, api.NegativeOrthant):
            cones[func.k] = True
            glob["cone"] = np.array([func.mu, func.half_length, func.half_width])
        else:
            raise NotImplementedError(f"unsupported stage constraint {type(func).__name__}")
    if cones != [bool(s) for s in cmap.contact_states]:
        raise NotImplementedError("wrench cones must be present exactly on the active contacts (centroidal_talos.py:242-245)")
    for key, val in glob.items():
        if key in G:
            _same(G[key], val, key)
        else:
            G[key] = val
    return k


def _check_cmap(a, b):
    if list(a.contact_states) != list(b.contact_states) or any(np.abs(np.asarray(p) - np.asarray(q)).max() > 0 for p, q in zip(a.contact_poses, b.contact_poses)):
        raise NotImplementedError("residual contact_map differs from the dynamics contact_map (the reference updates all three together, "
                                  "centroidal_talos.py:377-384)")


def _flatten_cent(problem, tol, mu_init, max_iters):
    from .talos_like import talos_like_robot

    T = len(problem.stages)
    G = {}
    knots = (_abi.Knot * T)()
    for j, st in enumerate(problem.stages):
        knots[j] = _flatten_cent_stage(st, G)
    if problem.term_cost.size() != 0 or len(problem.term_constraints) != 0:
        raise NotImplementedError("centroidal problem: empty terminal cost and no terminal constraint expected (centroidal_talos.py:249,261)")
    rb = talos_like_robot()
    _set(rb.gravity, G["gravity"])
    c = _abi.Config()
    c.kind, c.T, c.dt, c.mass = _abi.KIND_CENT, T, G["dt"], G["mass"]
    _set(c.wu, G.get("wu", np.zeros(12)))
    for name in ["w_com", "w_linmom", "w_angmom", "w_linacc", "w_angacc", "com_ref"]:
        _set(getattr(c, name), G.get(name, np.zeros(3)))
    cone = G.get("cone", np.array([0.8, 0.1, 0.075]))
    c.mu_fric, c.foot_L, c.foot_W = cone
    c.tol, c.mu_init, c.max_iters, c.force_initial_condition = tol, mu_init, max_iters, 1
    terms = (_abi.Term * 1)()
    return FlatProblem(rb, c, knots, terms, np.array(problem.x0_init, float).reshape(1, -1))


# ---------------------------------------------------------------- kinodynamics
def _flatten_kino_stage(stage, G):
    dyn = stage.dynamics
    if not isinstance(dyn, api.IntegratorSemiImplEuler):
        raise NotImplementedError("kinodynamic stage must use IntegratorSemiImplEuler (kinodynamic_talos.py:111)")
    ode = dyn.differential_dynamics
    model = ode.model
    if len(ode.contact_states) != 2 or ode.force_size != 6:
        raise NotImplementedError("kinodynamic model: two 6-D contacts expected (kinodynamic_talos.py:41-43)")
    if [_foot_index(model, frame_id=i) for i in ode.contact_ids] != [0, 1]:
        raise NotImplementedError("contact_ids must be [left_sole_link, right_sole_link] (kinodynamic_talos.py:69)")
    k = _abi.Knot()
    cs = [bool(ode.contact_states[0]), bool(ode.contact_states[1])]
    k.cs[0], k.cs[1] = float(cs[0]), float(cs[1])
    nv, nu = model.nv, ode.nu
    glob = dict(dt=dyn.timestep, gravity=ode.gravity)
    for key, c, wgt in stage.cost.items():
        if wgt != 1.0:
            raise NotImplementedError("CostStack component weights other than 1 are not supported")
        if isinstance(c, api.QuadraticStateCost):
            glob["x_ref"], glob["wx"] = c.target, _diag(c.weights, 2 * nv, "QuadraticStateCost")
        elif isinstance(c, api.QuadraticControlCost):
            _set(k.u_ref, c.target)
            glob["wu"] = _diag(c.weights, nu, "QuadraticControlCost")
        elif isinstance(c, api.QuadraticResidualCost):
            r = c.residual
            if isinstance(r, api.CentroidalMomentumResidual):
                if np.abs(r.ref).max() > 0:
                    raise NotImplementedError("CentroidalMomentumResidual reference must be zero")
                glob["w_cent"] = _diag(c.weights, 6, "centroidal momentum cost")
            elif isinstance(r, api.CentroidalMomentumDerivativeResidual):
                if [bool(x) for x in r.contact_states] != cs:
                    raise NotImplementedError("CentroidalMomentumDerivativeResidual contact states differ from the dynamics")
                glob["w_centder"] = _diag(c.weights, 6, "centroidal momentum derivative cost")
            elif isinstance(r, api.FramePlacementResidual):
                f = _foot_index(model, frame_id=r.frame_id)
                _set(k.w_lf if f == 0 else k.w_rf, _diag(c.weights, 6, "frame placement cost"))
                _set(k.lf_ref if f == 0 else k.rf_ref, r.ref.to12())
            else:
                raise NotImplementedError(f"unsupported residual in a kinodynamic cost: {type(r).__name__}")
        else:
            raise NotImplementedError(f"unsupported cost component {type(c).__name__}")
    cones, vels = [False, False], [False, False]
    for func, cset in zip(stage.constraints.funcs, stage.constraints.sets):
        if isinstance(func, api.SlicedResidual) and isinstance(func.base, api.StateErrorResidual) and isinstance(cset, api.BoxConstraint):
            if func.indices != list(range(6, nv)):
                raise NotImplementedError("joint-limit constraint must be StateErrorResidual[6:nv] (kinodynamic_talos.py:161)")
            glob["q_hi"], glob["q_lo"] = -cset.lower_limit, -cset.upper_limit
        elif isinstance(func, api.CentroidalWrenchConeResidual) and isinstance(cset, api.NegativeOrthant):
            cones[func.k] = True
            glob["cone"] = np.array([func.mu, func.half_length, func.half_width])
        elif isinstance(func, api.FrameVelocityResidual) and isinstance(cset, api.EqualityConstraintSet):
            if func.ref_frame != _pin.LOCAL or np.abs(np.asarray(func.ref.np, float)).max() > 0:
                raise NotImplementedError("frame-velocity constraint must be zero velocity in the LOCAL frame (kinodynamic_talos.py:129-130)")
            vels[_foot_index(model, frame_id=func.frame_id)] = True
        else:
            raise NotImplementedError(f"unsupported stage constraint {type(func).__name__} / {type(cset).__name__}")
    if cones != cs or vels != cs:
        raise NotImplementedError("cone + zero-velocity constraints must be present exactly on the active contacts (kinodynamic_talos.py:164-171)")
    for key, val in glob.items():
        if key in G:
            _same(G[key], val, key)
        else:
            G[key] = val
    G.setdefault("model", model)
    return k


def _flatten_kino(problem, tol, mu_init, max_iters):
    T = len(problem.stages)
    G = {}
    knots = (_abi.Knot * T)()
    for j, st in enumerate(problem.stages):
        knots[j] = _flatten_kino_stage(st, G)
    if problem.term_cost.size() != 0:
        raise NotImplementedError("kinodynamic problem: empty terminal cost expected (kinodynamic_talos.py:175)")
    model = G["model"]
    t = _abi.Term()
    ident = _pin.SE3().to12()
    _set(t.lf_ref, ident)
    _set(t.rf_ref, ident)
    if len(problem.term_constraints) > 1:
        raise NotImplementedError("at most one terminal constraint (CoM equality) is supported")
    for func, cset in zip(problem.term_constraints.funcs, problem.term_constraints.sets):
        if isinstance(func, api.CenterOfMassTranslationResidual) and isinstance(cset, api.EqualityConstraintSet):
            _set(t.com_ref, func.ref)
            t.has_com_cstr = 1.0
        else:
            raise NotImplementedError(f"unsupported terminal constraint {type(func).__name__}")
    rb = _abi.Robot.from_buffer_copy(_robot_from_model(model))
    _set(rb.gravity, G["gravity"])
    if "q_lo" in G:
        _set(rb.q_lo, G["q_lo"])
        _set(rb.q_hi, G["q_hi"])
    c = _abi.Config()
    c.kind, c.T, c.dt = _abi.KIND_KINO, T, G["dt"]
    _set(c.x_ref, G.get("x_ref", np.concatenate([_pin.neutral(model), np.zeros(model.nv)])))
    _set(c.wx, G.get("wx", np.zeros(2 * model.nv)))
    _set(c.wu, G.get("wu", np.zeros(34)))
    _set(c.w_cent, G.get("w_cent", np.zeros(6)))
    _set(c.w_centder, G.get("w_centder", np.zeros(6)))
    cone = G.get("cone", np.array([0.8, 0.1, 0.075]))
    c.mu_fric, c.foot_L, c.foot_W = cone
    c.tol, c.mu_init, c.max_iters, c.force_initial_condition = tol, mu_init, max_iters, 1
    terms = (_abi.Term * 1)(t)
    return FlatProblem(rb, c, knots, terms, np.array(problem.x0_init, float).reshape(1, -1))


def flatten_problem(problem, tol, mu_init, max_iters, rollout=0, lq_legs=0):
    """rollout: solver.rollout_type (0 = ROLLOUT_LINEAR, fulldynamic_talos.py:381; 1 = ROLLOUT_NONLINEAR).
    lq_legs: 0 or 1 = serial LQ solve, 2..min(16, T) = time-parallel LQ solve over that many horizon legs (mpc_config_t.lq_legs)."""
    if not problem.stages:
        raise ValueError("TrajOptProblem has no stages")
    ode = problem.stages[0].dynamics.differential_dynamics
    if isinstance(ode, api.CentroidalFwdDynamics):
        flat = _flatten_cent(problem, tol, mu_init, max_iters)
    elif isinstance(ode, api.MultibodyConstraintFwdDynamics):
        flat = _flatten_full(problem, tol, mu_init, max_iters)
    elif isinstance(ode, api.KinodynamicsFwdDynamics):
        flat = _flatten_kino(problem, tol, mu_init, max_iters)
    else:
        raise NotImplementedError(f"unsupported dynamics {type(ode).__name__}")
    flat.cfg.rollout = int(rollout)
    flat.cfg.lq_legs = int(lq_legs)
    return flat
