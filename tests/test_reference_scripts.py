"""'Switch backends with one import' (BASELINE north_star): the TOP HALF of the unmodified reference scripts runs on this
package's aligator/pinocchio shim, and the flattened descriptor equals the hand-written one of mpc_benchmark_b200.problems.
The reference scripts are not part of this repository: the descriptors they flatten to are committed as
tests/golden/ref_flat_*.npz (tests/golden/make_golden.py regenerates them from a checkout of the scripts)."""
import numpy as np
import pytest

import golden_util
from mpc_benchmark_b200 import _abi, problems


def _doubles(x):
    return np.frombuffer(bytes(x), dtype=np.float64)


@pytest.mark.parametrize("script,maker,golden", [("fulldynamic_talos.py", problems.full_standing_problem, "ref_flat_full.npz"),
                                                 ("kinodynamic_talos.py", problems.kino_standing_problem, "ref_flat_kino.npz"),
                                                 ("centroidal_talos.py", problems.cent_standing_problem, "ref_flat_cent.npz")])
def test_script_top_half_flattens_to_expected_descriptor(script, maker, golden):
    """`golden` holds what the top half of `script` flattened to (cfg, robot, knots, x0 and the xs / us handed to the cold solve)."""
    flat, z = golden_util.load(golden)
    ref = maker()
    assert bytes(flat["cfg"]) == bytes(ref["cfg"]) and bytes(flat["robot"]) == bytes(ref["robot"])
    assert np.allclose(_doubles(flat["knots"]), _doubles(ref["knots"]), rtol=1e-13, atol=0)
    assert np.array_equal(flat["x0"], ref["x0"]) and np.array_equal(flat["xs"], ref["xs"]) and np.array_equal(flat["us"], ref["us"])


def test_mutation_through_problem_stages_is_seen_by_flatten():
    """centroidal_talos.py:374-384 mutates contact poses through problem.stages[n]; the problem holds its stages BY VALUE
    (aligator >= 0.10), so the objects passed to the constructor are not aliased."""
    import mpc_benchmark_b200 as aligator
    from mpc_benchmark_b200 import flatten, pin

    ns = _build_cent(aligator, pin)
    problem, stages = ns["problem"], ns["stages"]
    f0 = flatten.flatten_problem(problem, 1e-5, 1e-8, 10)
    new = np.array([0.5, 0.1, 0.0])
    st = problem.stages[3]
    st.dynamics.differential_dynamics.contact_map.contact_poses[0] = new
    for name in ("angular_acc_cost", "linear_acc_cost"):
        st.cost.getComponent(name).residual.contact_map.contact_poses[0] = new
    f1 = flatten.flatten_problem(problem, 1e-5, 1e-8, 10)
    assert list(f1.knots[3].cpos)[:3] == [0.5, 0.1, 0.0] and list(f0.knots[3].cpos)[:3] != [0.5, 0.1, 0.0]
    assert list(stages[3].dynamics.differential_dynamics.contact_map.contact_poses[0]) != [0.5, 0.1, 0.0]  # caller's object untouched
    problem.replaceStageCircular(stages[0])
    f2 = flatten.flatten_problem(problem, 1e-5, 1e-8, 10)
    assert list(f2.knots[2].cpos)[:3] == [0.5, 0.1, 0.0]  # horizon rotated by one
    assert problem.term_cost.size() == 0


def test_aliased_stage_list_gets_one_reference_per_knot():
    """fulldynamic_talos.py:371 builds the problem from `[stage] * nsteps` and :461-463 then writes a different swing-foot
    reference into every problem.stages[j]: each knot must keep its own (value semantics), not the last write."""
    import mpc_benchmark_b200 as aligator
    from mpc_benchmark_b200 import constraints, dynamics, flatten, manifolds, pin

    rmodel = pin.Model()
    rdata = rmodel.createData()
    q0 = rmodel.referenceConfigurations["half_sitting"]
    pin.framesForwardKinematics(rmodel, rdata, q0)
    nv, nu = rmodel.nv, rmodel.nv - 6
    space = manifolds.MultibodyPhaseSpace(rmodel)
    x0 = np.concatenate([q0, np.zeros(nv)])
    act = np.eye(nv, nu, -6)
    prox = pin.ProximalSettings(1e-9, 1e-10, 1)
    ids = [rmodel.getFrameId("left_sole_link"), rmodel.getFrameId("right_sole_link")]
    cms = []
    for fid, name in zip(ids, ["left_sole_link", "right_sole_link"]):
        fr = rmodel.frames[fid]
        cm = pin.RigidConstraintModel(pin.ContactType.CONTACT_6D, rmodel, fr.parentJoint, fr.placement, 0, rdata.oMf[fid], pin.LOCAL)
        cm.corrector.Kp[:] = (0, 0, 10, 0, 0, 0)
        cm.corrector.Kd[:] = 50
        cm.name = name
        cms.append(cm)
    rcost = aligator.CostStack(space, nu)
    rcost.addCost(aligator.QuadraticStateCost(space, nu, x0, np.eye(2 * nv)))
    rcost.addCost(aligator.QuadraticControlCost(space, np.zeros(nu), 1e-4 * np.eye(nu)))
    rcost.addCost(aligator.QuadraticResidualCost(space, aligator.CentroidalMomentumResidual(space.ndx, nu, rmodel, np.zeros(6)), np.eye(6)))
    for fid in ids:
        rcost.addCost(aligator.QuadraticResidualCost(space, aligator.FramePlacementResidual(space.ndx, nu, rmodel, rdata.oMf[fid].copy(), fid), 2000 * np.eye(6)))
    stage = aligator.StageModel(rcost, dynamics.IntegratorSemiImplEuler(dynamics.MultibodyConstraintFwdDynamics(space, act, cms, prox), 0.01))
    T = 5
    problem = aligator.TrajOptProblem(x0, [stage] * T, aligator.CostStack(space, nu))
    for j in range(T):
        ref = rdata.oMf[ids[0]].copy()
        ref.translation[2] += 0.01 * (j + 1)
        problem.stages[j].cost.getComponent(3).residual.setReference(ref)
    flat = flatten.flatten_problem(problem, 1e-5, 1e-8, 10)
    z0 = rdata.oMf[ids[0]].translation[2]
    assert np.allclose([flat.knots[j].lf_ref[11] - z0 for j in range(T)], [0.01 * (j + 1) for j in range(T)], atol=1e-15)
    assert stage.cost.getComponent(3).residual.getReference().translation[2] == z0  # the caller's stage is not aliased


def _build_cent(aligator, pin, T=6):
    """Centroidal problem built through the public API exactly as centroidal_talos.py:208-261 does."""
    from mpc_benchmark_b200 import constraints, dynamics, manifolds

    rmodel = pin.Model()
    rdata = rmodel.createData()
    q0 = rmodel.referenceConfigurations["half_sitting"]
    pin.forwardKinematics(rmodel, rdata, q0)
    pin.updateFramePlacements(rmodel, rdata)
    com0 = pin.centerOfMass(rmodel, rdata, q0)
    mass = pin.computeTotalMass(rmodel)
    nx, nu = 9, 12
    space = manifolds.VectorSpace(nx)
    gravity = np.array([0, 0, -9.81])
    LF, RF = rmodel.getFrameId("left_sole_link"), rmodel.getFrameId("right_sole_link")
    u0 = np.zeros(nu)
    u0[2] = u0[8] = mass * 9.81 / 2
    w_control = np.diag([0.001] * 3 + [0.1] * 3 + [0.001] * 3 + [0.1] * 3)

    def createStage(cs):
        cmap = aligator.ContactMap(["left_sole_link", "right_sole_link"], cs, [rdata.oMf[LF].translation, rdata.oMf[RF].translation])
        rcost = aligator.CostStack(space, nu)
        rcost.addCost("state_cost", aligator.QuadraticControlCost(space, u0, w_control))
        rcost.addCost("com_cost", aligator.QuadraticResidualCost(space, aligator.CentroidalCoMResidual(nx, nu, com0), np.diag([0, 0, 0.0])))
        rcost.addCost("linear_mom_cost", aligator.QuadraticResidualCost(space, aligator.LinearMomentumResidual(nx, nu, np.zeros(3)), np.diag([0.01, 0.01, 100])))
        rcost.addCost("angular_mom_cost", aligator.QuadraticResidualCost(space, aligator.AngularMomentumResidual(nx, nu, np.zeros(3)), np.diag([0.1, 0.1, 1000])))
        rcost.addCost("angular_acc_cost", aligator.QuadraticResidualCost(space, aligator.AngularAccelerationResidual(nx, nu, mass, gravity, cmap, 6), 0.01 * np.eye(3)))
        rcost.addCost("linear_acc_cost", aligator.QuadraticResidualCost(space, aligator.CentroidalAccelerationResidual(nx, nu, mass, gravity, cmap, 6), 0.01 * np.eye(3)))
        stm = aligator.StageModel(rcost, dynamics.IntegratorEuler(dynamics.CentroidalFwdDynamics(space, mass, gravity, cmap, 6), 0.01))
        for i in range(2):
            if cs[i]:
                stm.addConstraint(aligator.CentroidalWrenchConeResidual(space.ndx, nu, i, 0.8, 0.1, 0.075), constraints.NegativeOrthant())
        return stm

    stages = [createStage([True, True]) for _ in range(T)]
    x0 = space.neutral()
    x0[:3] = com0
    problem = aligator.TrajOptProblem(x0, stages, aligator.CostStack(space, nu))
    return dict(problem=problem, stages=stages, x0=x0, u0=u0, T=T)


def test_unsupported_structures_raise_with_a_name():
    import mpc_benchmark_b200 as aligator
    from mpc_benchmark_b200 import flatten, pin

    ns = _build_cent(aligator, pin)
    ns["problem"].stages[0].cost.addCost("bad", aligator.QuadraticStateCost(aligator.manifolds.VectorSpace(9), 12, np.zeros(9), np.eye(9)))
    with pytest.raises(NotImplementedError, match="QuadraticStateCost"):
        flatten.flatten_problem(ns["problem"], 1e-5, 1e-8, 10)
    # the default rollout is NONLINEAR, as in aligator (the scripts set LINEAR): it flattens to cfg.rollout = 1
    assert aligator.SolverProxDDP(1e-5, 1e-8).rollout_type == aligator.ROLLOUT_NONLINEAR
    ns2 = _build_cent(aligator, pin)
    assert flatten.flatten_problem(ns2["problem"], 1e-5, 1e-8, 10, rollout=1).cfg.rollout == 1
    assert flatten.flatten_problem(ns2["problem"], 1e-5, 1e-8, 10).cfg.rollout == 0
