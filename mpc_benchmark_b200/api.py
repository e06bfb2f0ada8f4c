"""Aligator-compatible modelling surface (SURVEY 8a/8b): the names, positional signatures and mutation semantics
the three reference scripts use, implemented as plain Python parameter carriers.

`import mpc_benchmark_b200 as aligator` + `from mpc_benchmark_b200 import manifolds, dynamics, constraints`
replaces `import aligator` (fulldynamic_talos.py:8,23-25; kinodynamic_talos.py:10,30-32; centroidal_talos.py:8,30-32).
Objects only HOLD parameters; `SolverProxDDP.setup/run` flattens the object graph (flatten.py) into the C-ABI
descriptor on every call, so mutation through the problem (`problem.stages[j].cost.getComponent(k).residual.setReference`,
`...contact_map.contact_poses[i] = p`) is always visible.  `TrajOptProblem` stores stages and the terminal cost BY VALUE
(Aligator >= 0.10 keeps them as `xyz::polymorphic` values and copies the list on construction): the `[stage] * 100` of
fulldynamic_talos.py:371 becomes 100 independent stages, so the per-knot `setReference` loop of :461-463 gives every
knot its own swing-foot reference.
All arithmetic of the solve runs in the CUDA library; nothing here evaluates a cost or a derivative.
"""
import copy

import numpy as np

from . import _abi
from . import pin as _pin

ROLLOUT_LINEAR, ROLLOUT_NONLINEAR = 0, 1
LQ_SOLVER_SERIAL, LQ_SOLVER_PARALLEL, LQ_SOLVER_STAGEDENSE = 0, 1, 2


class VerboseLevel:
    QUIET, VERBOSE, VERYVERBOSE = 0, 1, 2


class StdVec(list):
    """list with the `.tolist()` of eigenpy's StdVec_VectorXs (fulldynamic_talos.py:403-404)."""

    def tolist(self):
        return list(self)


# ------------------------------------------------------------------ Lie-group helpers (host side, numpy)
def _skew(w):
    return np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])


def _log3(R):
    s = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    ct = 0.5 * (np.trace(R) - 1.0)
    sn = np.linalg.norm(s)
    if sn < 1e-9 and ct > 0:
        return s
    return s * (np.arctan2(sn, ct) / sn)


def _log6(R, p):
    w = _log3(R)
    t2 = w @ w
    if t2 < 1e-6:
        c = 1.0 / 12 + t2 / 720
    else:
        t = np.sqrt(t2)
        c = (1.0 - t * np.sin(t) / (2.0 * (1.0 - np.cos(t)))) / t2
    W = _skew(w)
    Vi = np.eye(3) - 0.5 * W + c * W @ W
    return np.concatenate([Vi @ p, w])


def _quat_to_R(q):
    from .kinematics import quat_to_R

    return quat_to_R(q)


# ------------------------------------------------------------------ manifolds
class VectorSpace:
    def __init__(self, nx):
        self.nx = self.ndx = int(nx)

    def neutral(self):
        return np.zeros(self.nx)

    def difference(self, x0, x1):
        return np.asarray(x1, float) - np.asarray(x0, float)

    def integrate(self, x, dx):
        return np.asarray(x, float) + np.asarray(dx, float)


class MultibodyPhaseSpace:
    def __init__(self, model):
        self.model = model
        self.nx, self.ndx = model.nq + model.nv, 2 * model.nv

    def neutral(self):
        return np.concatenate([_pin.neutral(self.model), np.zeros(self.model.nv)])

    def difference(self, x0, x1):
        """x1 (-) x0 (SURVEY App. A1): [log6(M0^-1 M1); theta1 - theta0; v1 - v0]."""
        x0, x1 = np.asarray(x0, float), np.asarray(x1, float)
        R0, R1 = _quat_to_R(x0[3:7]), _quat_to_R(x1[3:7])
        nq = self.model.nq
        return np.concatenate([_log6(R0.T @ R1, R0.T @ (x1[:3] - x0[:3])), x1[7:nq] - x0[7:nq], x1[nq:] - x0[nq:]])


# ------------------------------------------------------------------ constraint sets
class BoxConstraint:
    def __init__(self, lower, upper):
        self.lower_limit, self.upper_limit = np.array(lower, float), np.array(upper, float)


class NegativeOrthant:
    pass


class EqualityConstraintSet:
    pass


# ------------------------------------------------------------------ residuals
class _Residual:
    nr = 0

    def __getitem__(self, idx):
        return SlicedResidual(self, idx)


class SlicedResidual(_Residual):
    def __init__(self, base, idx):
        self.base, self.idx = base, idx
        rng = range(base.nr)[idx] if isinstance(idx, slice) else [range(base.nr)[idx]]
        self.indices = list(rng)
        self.nr = len(self.indices)

    def setReference(self, ref):
        self.base.setReference(ref)

    def getReference(self):
        return self.base.getReference()


class StateErrorResidual(_Residual):
    def __init__(self, space, nu, target):
        self.space, self.nu, self.target, self.nr = space, nu, np.array(target, float), space.ndx


class ControlErrorResidual(_Residual):
    def __init__(self, ndx, target):
        if np.isscalar(target):
            raise TypeError("ControlErrorResidual(ndx, target): target must be a vector")
        self.ndx, self.target, self.nr = ndx, np.array(target, float), len(target)


class _RefResidual(_Residual):
    def setReference(self, ref):
        self.ref = ref.copy() if hasattr(ref, "copy") else np.array(ref, float)

    def getReference(self):
        return self.ref


class CentroidalMomentumResidual(_RefResidual):
    def __init__(self, ndx, nu, model, h_ref):
        self.ndx, self.nu, self.model, self.ref, self.nr = ndx, nu, model, np.array(h_ref, float), 6


class FramePlacementResidual(_RefResidual):
    def __init__(self, ndx, nu, model, M_ref, frame_id):
        self.ndx, self.nu, self.model, self.ref, self.frame_id, self.nr = ndx, nu, model, M_ref.copy(), frame_id, 6


class FrameVelocityResidual(_RefResidual):
    def __init__(self, ndx, nu, model, v_ref, frame_id, ref_frame=_pin.LOCAL):
        self.ndx, self.nu, self.model, self.ref, self.frame_id, self.ref_frame, self.nr = ndx, nu, model, v_ref, frame_id, ref_frame, 6


class FrameTranslationResidual(_RefResidual):
    def __init__(self, ndx, nu, model, p_ref, frame_id):
        self.ndx, self.nu, self.model, self.ref, self.frame_id, self.nr = ndx, nu, model, np.array(p_ref, float), frame_id, 3


class CenterOfMassTranslationResidual(_RefResidual):
    def __init__(self, ndx, nu, model, c_ref):
        self.ndx, self.nu, self.model, self.ref, self.nr = ndx, nu, model, np.array(c_ref, float), 3


class DCMPositionResidual(_RefResidual):
    def __init__(self, ndx, nu, model, dcm_ref, alpha):
        self.ndx, self.nu, self.model, self.ref, self.alpha, self.nr = ndx, nu, model, np.array(dcm_ref, float), alpha, 3


class ContactForceResidual(_RefResidual):
    def __init__(self, ndx, model, actuation_matrix, constraint_models, prox_settings, f_ref, contact_name):
        self.ndx, self.model, self.actuation_matrix = ndx, model, np.array(actuation_matrix, float)
        self.constraint_models, self.prox_settings = list(constraint_models), prox_settings
        self.ref, self.contact_name, self.nr = np.array(f_ref, float), contact_name, 6


class MultibodyWrenchConeResidual(_Residual):
    def __init__(self, ndx, model, actuation_matrix, constraint_models, prox_settings, contact_name, mu, half_length, half_width):
        self.ndx, self.model, self.actuation_matrix = ndx, model, np.array(actuation_matrix, float)
        self.constraint_models, self.prox_settings, self.contact_name = list(constraint_models), prox_settings, contact_name
        self.mu, self.half_length, self.half_width, self.nr = mu, half_length, half_width, 17


class CentroidalWrenchConeResidual(_Residual):
    def __init__(self, ndx, nu, k, mu, half_length, half_width):
        self.ndx, self.nu, self.k, self.mu, self.half_length, self.half_width, self.nr = ndx, nu, k, mu, half_length, half_width, 17


class CentroidalMomentumDerivativeResidual(_Residual):
    def __init__(self, ndx, model, gravity, contact_states, contact_ids, force_size):
        self.ndx, self.model, self.gravity, self.contact_states = ndx, model, np.array(gravity, float), list(contact_states)
        self.contact_ids, self.force_size, self.nr = list(contact_ids), force_size, 6


class LinearMomentumResidual(_RefResidual):
    def __init__(self, nx, nu, ref):
        self.nx, self.nu, self.ref, self.nr = nx, nu, np.array(ref, float), 3


class AngularMomentumResidual(LinearMomentumResidual):
    pass


class CentroidalCoMResidual(LinearMomentumResidual):
    pass


class ContactMap:
    def __init__(self, contact_names, contact_states, contact_poses):
        self.contact_names = list(contact_names)
        self.contact_states = list(contact_states)
        self.contact_poses = [np.array(p, float) for p in contact_poses]

    @property
    def size(self):
        return len(self.contact_states)


class CentroidalAccelerationResidual(_Residual):
    def __init__(self, nx, nu, mass, gravity, contact_map, force_size):
        self.nx, self.nu, self.mass, self.gravity, self.contact_map, self.force_size, self.nr = nx, nu, mass, np.array(gravity, float), contact_map, force_size, 3


class AngularAccelerationResidual(CentroidalAccelerationResidual):
    pass


# ------------------------------------------------------------------ costs
class QuadraticStateCost:
    def __init__(self, space, nu, target, weights):
        self.space, self.nu, self.target, self.weights = space, nu, np.array(target, float), np.array(weights, float)


class QuadraticControlCost:
    def __init__(self, space, target, weights):
        self.space, self.target, self.weights = space, np.array(target, float), np.array(weights, float)


class QuadraticResidualCost:
    def __init__(self, space, residual, weights):
        self.space, self.residual, self.weights = space, residual, np.array(weights, float)


class _ComponentView:
    """`cost.components[k]` -> (cost, weight) as in aligator's std::pair binding (fulldynamic_talos.py:509-510)."""

    def __init__(self, stack):
        self._stack = stack

    def __getitem__(self, key):
        c = self._stack.getComponent(key)
        return (c, self._stack._weights[self._stack._key(key)])

    def __len__(self):
        return len(self._stack._order)


class CostStack:
    def __init__(self, space, nu, components=None, weights=None):
        self.space, self.nu = space, nu
        self._order, self._comps, self._weights = [], {}, {}
        for i, c in enumerate(components or []):
            self.addCost(c, (weights or [1.0] * len(components))[i])

    def addCost(self, *args):
        """addCost(cost[, weight]) or addCost(name, cost[, weight]) (fulldynamic_talos.py:175; kinodynamic_talos.py:139)."""
        if isinstance(args[0], str):
            key, cost, weight = args[0], args[1], (args[2] if len(args) > 2 else 1.0)
        else:
            key, cost, weight = len(self._order), args[0], (args[1] if len(args) > 1 else 1.0)
        self._order.append(key)
        self._comps[key], self._weights[key] = cost, float(weight)
        return cost

    def _key(self, key):
        if key in self._comps:
            return key
        if isinstance(key, int) and 0 <= key < len(self._order):
            return self._order[key]
        raise KeyError(key)

    def getComponent(self, key):
        return self._comps[self._key(key)]

    @property
    def components(self):
        return _ComponentView(self)

    def size(self):
        return len(self._order)

    def items(self):
        return [(k, self._comps[k], self._weights[k]) for k in self._order]


# ------------------------------------------------------------------ dynamics
class MultibodyConstraintFwdDynamics:
    def __init__(self, space, actuation_matrix, constraint_models, prox_settings):
        self.space, self.actuation_matrix = space, np.array(actuation_matrix, float)
        self.constraint_models, self.prox_settings = list(constraint_models), prox_settings
        self.ndx, self.nu = space.ndx, self.actuation_matrix.shape[1]


class KinodynamicsFwdDynamics:
    def __init__(self, space, model, gravity, contact_states, contact_ids, force_size):
        self.space, self.model, self.gravity = space, model, np.array(gravity, float)
        self.contact_states, self.contact_ids, self.force_size = list(contact_states), list(contact_ids), force_size
        self.ndx, self.nu = space.ndx, model.nv - 6 + force_size * len(contact_states)


class CentroidalFwdDynamics:
    def __init__(self, space, mass, gravity, contact_map, force_size):
        self.space, self.mass, self.gravity, self.contact_map, self.force_size = space, float(mass), np.array(gravity, float), contact_map, force_size
        self.ndx, self.nu = space.ndx, force_size * contact_map.size


class _Integrator:
    def __init__(self, ode, timestep):
        self.differential_dynamics, self.ode, self.timestep = ode, ode, float(timestep)
        self.space, self.ndx, self.nu = ode.space, ode.ndx, ode.nu


class IntegratorSemiImplEuler(_Integrator):
    pass


class IntegratorEuler(_Integrator):
    pass


# ------------------------------------------------------------------ stages / problem
class StageConstraint:
    def __init__(self, func, cstr_set):
        self.func, self.set = func, cstr_set


class _ConstraintStack:
    def __init__(self):
        self.funcs, self.sets = [], []

    def append(self, c):
        self.funcs.append(c.func)
        self.sets.append(c.set)

    def clear(self):
        self.funcs.clear()
        self.sets.clear()

    def __len__(self):
        return len(self.funcs)


class StageData:
    """Opaque token: the device workspace is owned by the solver (createData exists for API compatibility)."""

    def __init__(self, stage):
        self.stage = stage


class StageModel:
    def __init__(self, cost, dynamics):
        self.cost, self.dynamics, self.dyn_model = cost, dynamics, dynamics
        self.constraints = _ConstraintStack()

    def addConstraint(self, *args):
        c = args[0] if len(args) == 1 else StageConstraint(args[0], args[1])
        self.constraints.append(c)

    def createData(self):
        return StageData(self)

    @property
    def ndx1(self):
        return self.dynamics.ndx

    @property
    def nu(self):
        return self.dynamics.nu


def _clone(obj):
    """Value copy of a stage / cost stack (robot models are immutable carriers and stay shared, see pin.Model.__deepcopy__)."""
    return copy.deepcopy(obj)


class TrajOptProblem:
    """Stages and terminal cost are held by value, as aligator >= 0.10 does: `problem.stages[j]` is the problem's own copy
    and the object passed in is not aliased (fulldynamic_talos.py:371-372,461-463; kinodynamic_talos.py:274-276,384-385)."""

    def __init__(self, x0, stages, term_cost):
        self.x0_init = np.array(x0, float)
        self.stages = [_clone(s) for s in stages]
        self.term_cost = _clone(term_cost)
        self.term_constraints = _ConstraintStack()

    @property
    def num_steps(self):
        return len(self.stages)

    def addTerminalConstraint(self, c):
        self.term_constraints.append(c)

    def removeTerminalConstraint(self):
        self.term_constraints.clear()

    def replaceStageCircular(self, stage):
        """Drop stage 0, append `stage` at the end (fulldynamic_talos.py:496)."""
        self.stages.pop(0)
        self.stages.append(_clone(stage))

    def addStage(self, stage):
        self.stages.append(_clone(stage))


# ------------------------------------------------------------------ solver
class _ContactForceView:
    def __init__(self, w):
        self.linear, self.angular = w[:3].copy(), w[3:].copy()


class _ConstraintDataView:
    def __init__(self, w):
        self.contact_force = _ContactForceView(w)


class _ContinuousData:
    def __init__(self, xdot, forces):
        self.xdot = xdot
        self.constraint_datas = [_ConstraintDataView(f) for f in forces]


class _DynData:
    def __init__(self, cd):
        self.continuous_data = cd


class _StageDataView:
    def __init__(self, cd):
        self.dynamics_data = _DynData(cd)


class _StageDataList:
    def __init__(self, solver):
        self._solver = solver

    def __len__(self):
        return self._solver._T

    def __getitem__(self, k):
        return self._solver._stage_data(k)


class _ProblemData:
    def __init__(self, solver):
        self.stage_data = _StageDataList(solver)


class Workspace:
    def __init__(self, solver):
        self._solver = solver
        self.problem_data = _ProblemData(solver)

    def cycleAppend(self, stage_data):
        """The reference rotates the per-stage data (fulldynamic_talos.py:497); the device workspace is re-indexed from the
        problem at the next run, so only the shift of the warm multipliers is recorded here."""
        self._solver._pending_cycles += 1


class Results:
    def __init__(self):
        self.xs, self.us, self.vs, self.lams = StdVec(), StdVec(), StdVec(), StdVec()
        self._K = []
        self.num_iters, self.conv, self.prim_infeas, self.dual_infeas = 0, False, 0.0, 0.0
        self.traj_cost, self.merit_value, self.al_iter, self.mu = 0.0, 0.0, 0, 0.0

    def controlFeedbacks(self):
        return self._K

    def __str__(self):
        return (f"Results {{\n  num_iters:    {self.num_iters},\n  converged:    {self.conv},\n  traj. cost:   {self.traj_cost:.6g},\n"
                f"  merit.value:  {self.merit_value:.6g},\n  prim_infeas:  {self.prim_infeas:.4g},\n  dual_infeas:  {self.dual_infeas:.4g},\n}}")


class SolverProxDDP:
    """aligator.SolverProxDDP(tol, mu_init, ...) — setup/run/results/workspace as used at fulldynamic_talos.py:379-405."""

    def __init__(self, tol, mu_init=1e-2, rho_init=0.0, max_iters=1000, verbose=VerboseLevel.QUIET, device=0):
        self.target_tol, self.mu_init, self.max_iters, self.verbose = float(tol), float(mu_init), int(max_iters), verbose
        self.rollout_type, self.linear_solver_choice = ROLLOUT_NONLINEAR, LQ_SOLVER_SERIAL
        self.force_initial_condition = True
        self.ldlt_algo_choice = 0
        self.num_threads = 1
        # horizon legs of the time-parallel LQ solve (0 = serial).  Independent of linear_solver_choice, which stays recorded only.
        self.lq_legs = 0
        self.device = device
        self.results, self.workspace = Results(), Workspace(self)
        self._bs, self._sig, self._T, self._flat = None, None, 0, None
        self._pending_cycles = 0

    def setNumThreads(self, n):
        self.num_threads = int(n)  # recorded only: the GPU path has no host threads (SURVEY 8b)

    def getNumThreads(self):
        return self.num_threads

    def _check_options(self):
        if self.rollout_type not in (ROLLOUT_LINEAR, ROLLOUT_NONLINEAR):
            raise ValueError("rollout_type must be ROLLOUT_LINEAR or ROLLOUT_NONLINEAR")
        if not self.force_initial_condition:
            raise NotImplementedError("force_initial_condition = False is not implemented")

    def setup(self, problem):
        from . import flatten
        from .batch import BatchSolver

        self._check_options()
        flat = flatten.flatten_problem(problem, tol=self.target_tol, mu_init=self.mu_init, max_iters=self.max_iters,
                                       rollout=int(self.rollout_type == ROLLOUT_NONLINEAR), lq_legs=self.lq_legs)
        sig = (flat.cfg.kind, flat.cfg.T)
        if self._bs is None or sig != self._sig:
            if self._bs is not None:
                self._bs.close()
            self._bs = BatchSolver(flat.robot, flat.cfg, 1, device=self.device, model_blob=flat)
            self._sig = sig
        else:
            self._bs.reconfigure(flat.robot, flat.cfg)
        self._bs.setup(flat.knots, flat.terms, flat.x0)
        self._flat, self._T, self._pending_cycles = flat, flat.cfg.T, 0

    def cycleProblem(self, problem, stage_data):
        """kinodynamic_talos.py:488 / centroidal_talos.py:460: rotate the workspace in place (multipliers shift by one)."""
        self._pending_cycles += 1

    def run(self, problem, xs_init=(), us_init=(), vs_init=(), lams_init=()):
        from . import flatten

        if self._bs is None:
            raise RuntimeError("SolverProxDDP.run: call setup(problem) first")
        self._check_options()
        flat = flatten.flatten_problem(problem, tol=self.target_tol, mu_init=self.mu_init, max_iters=self.max_iters,
                                       rollout=int(self.rollout_type == ROLLOUT_NONLINEAR), lq_legs=self.lq_legs)
        if (flat.cfg.kind, flat.cfg.T) != self._sig:
            raise RuntimeError("problem structure changed since setup(); call setup(problem) again")
        bs = self._bs
        bs.reconfigure(flat.robot, flat.cfg)
        bs.update_knots(flat.knots, 0, flat.cfg.T)
        bs.update_terms(flat.terms)
        bs.set_x0(flat.x0)
        if self._pending_cycles:
            bs.shift_multipliers(self._pending_cycles)
            self._pending_cycles = 0
        nx, n, m, nc = _abi.DIMS[flat.cfg.kind]
        T = flat.cfg.T
        xs = np.array(xs_init, float).reshape(1, T + 1, nx) if len(xs_init) else np.tile(flat.x0, (1, T + 1, 1))
        us = np.array(us_init, float).reshape(1, T, m) if len(us_init) else np.zeros((1, T, m))
        res = bs.run(xs, us, max_iters=self.max_iters)
        r = self.results
        r.xs = StdVec(res.xs[0, k].copy() for k in range(T + 1))
        r.us = StdVec(res.us[0, k].copy() for k in range(T))
        r.vs = StdVec(res.vs[0, k].copy() for k in range(T + 1))
        r.lams = StdVec(res.lams[0, k].copy() for k in range(T + 1))
        r._K = [res.K[0, k].copy() for k in range(T)]
        i = res.info[0]
        r.num_iters, r.conv, r.prim_infeas, r.dual_infeas = i.num_iters, bool(i.conv), i.prim_infeas, i.dual_infeas
        r.traj_cost, r.merit_value, r.al_iter, r.mu = i.traj_cost, i.merit, i.al_iters, i.mu
        self._flat = flat
        return r.conv

    def _stage_data(self, k):
        xdot, force = self._bs.stage_data(k)
        kn = self._flat.knots[k]
        forces = []
        left, right = kn.cs[0] != 0.0, kn.cs[1] != 0.0
        if self._flat.cfg.kind == _abi.KIND_FULL and not left and not right:
            left = right = True
        if left:
            forces.append(force[0, :6])
        if right:
            forces.append(force[0, 6:])
        return _StageDataView(_ContinuousData(xdot[0].copy(), forces))


class SolverFDDP:
    """Referenced only in comments of the reference (fulldynamic_talos.py:380); constructor exists, no kernel."""

    def __init__(self, tol, verbose=VerboseLevel.QUIET, **kw):
        self.target_tol = tol

    def setup(self, problem):
        raise NotImplementedError("SolverFDDP is not part of the ProxDDP hot path (SURVEY 8a row C15)")

    run = setup
