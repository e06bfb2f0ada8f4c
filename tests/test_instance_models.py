"""Per-instance robot parameters and cost constants (mpc_set_instance_models / BatchSolver.set_instance_models).

CPU: the kernel sources under the host emulation (emu_solve_models) with a heterogeneous batch against the oracle run per instance on
its own (robot_i, cfg_i), and the validation of what must stay uniform.  GPU (`-m gpu`): the device path against the oracle per instance,
bitwise equality with the shared path when every instance carries the shared model, bitwise equality of instance i of a heterogeneous
batch with instance i of a homogeneous batch of (robot_i, cfg_i), the device gait's sole placements from each robot's own kinematics,
the rigid-body terms per robot and the error paths."""
import numpy as np
import pytest

import emu_lib
import emu_models_lib
from mpc_benchmark_b200 import _abi, problems

RTOL = 1e-6
ARM_BODIES = range(15, 23)  # arm joints of the Talos-shaped tree: their placements move no sole


def rel(a, b):
    return np.abs(a - b).max() / max(1e-12, np.abs(b).max())


def _copy(st):
    return type(st).from_buffer_copy(st)


def hetero_models(prob, seed):
    """Per-instance robots (masses, inertias, CoMs, a torso payload, arm joint placements) and configs (state / control / contact-force /
    centroidal weights, friction, Baumgarte gains, centroidal mass and CoM target) around prob's shared ones."""
    B, cfg = prob["x0"].shape[0], prob["cfg"]
    rng = np.random.default_rng(seed + 100)
    robots = problems.perturbed_robots(prob["robot"], B, seed, mass=0.15, com=0.01, payload=4.0)
    for r in robots:
        for b in ARM_BODIES:
            r.jplace[b][9:12] = list(np.asarray(r.jplace[b][9:12]) + rng.normal(size=3) * 0.01)
    cfgs = []
    for _ in range(B):
        c = _copy(cfg)
        for name in ("wx", "wu", "w_cent", "w_force", "wx_term", "w_linmom", "w_angmom"):
            a = getattr(c, name)
            a[:] = list(np.asarray(a[:]) * rng.uniform(0.5, 2.0, size=len(a)))
        c.mu_fric *= rng.uniform(0.8, 1.1)
        c.kp[:] = list(np.asarray(c.kp[:]) * rng.uniform(0.5, 1.5))
        c.kd[:] = list(np.asarray(c.kd[:]) * rng.uniform(0.5, 1.5))
        if cfg.kind == _abi.KIND_CENT:
            c.mass *= rng.uniform(0.9, 1.1)
            c.com_ref[:] = list(np.asarray(c.com_ref[:]) + rng.normal(size=3) * 0.01)
        cfgs.append(c)
    return robots, cfgs


def oracle_per_instance(oracle, prob, robots, cfgs, max_iters, xs=None, us=None):
    """The oracle run on each instance alone with its own (robot_i, cfg_i), stacked like a batch result."""
    B = prob["x0"].shape[0]
    outs = []
    for i in range(B):
        p = problems.sub_problem(prob, i, i + 1)
        p["robot"], p["cfg"] = robots[i], cfgs[i]
        outs.append(oracle.solve(p, max_iters=max_iters, xs=None if xs is None else xs[i:i + 1], us=None if us is None else us[i:i + 1]))
    r = {k: np.concatenate([o[k] for o in outs]) for k in ("xs", "us", "K", "vs", "lams")}
    r["info"] = [o["info"][0] for o in outs]
    return r


def _with_solver_consts(prob, rollout=0, lq_legs=0):
    prob["cfg"].rollout, prob["cfg"].lq_legs = rollout, lq_legs
    return prob


def _check(got_xs, got_us, got_K, got_iters, ref, vs=None):
    assert list(got_iters) == [i.num_iters for i in ref["info"]]
    assert rel(got_xs, ref["xs"]) < RTOL and rel(got_us, ref["us"]) < RTOL
    assert rel(got_K, ref["K"]) < 1e-5
    if vs is not None:
        assert rel(vs, ref["vs"]) < 1e-5


# ---------------------------------------------------------------- CPU: host emulation of the kernel sources
COLD = [(problems.cent_standing_problem, 30, 0), (problems.full_standing_problem, 8, 0), (problems.kino_standing_problem, 8, 0),
        (problems.full_standing_problem, 8, 1)]


@pytest.mark.parametrize("maker,T,rollout", COLD)
def test_emulated_cold_solve_matches_oracle_per_instance(oracle, maker, T, rollout):
    prob = _with_solver_consts(maker(batch=3, T=T), rollout)
    robots, cfgs = hetero_models(prob, 1)
    e = emu_models_lib.solve_models(prob, robots, cfgs, 100)
    ref = oracle_per_instance(oracle, prob, robots, cfgs, 100)
    _check(e["xs"], e["us"], e["K"], [i.num_iters for i in e["info"]], ref)
    assert [i.conv for i in e["info"]] == [i.conv for i in ref["info"]]
    # the instances really differ: a shared-model solve is far from them
    shared = emu_lib.solve(prob, 100)
    assert rel(shared["us"], ref["us"]) > 1e3 * RTOL


@pytest.mark.parametrize("kind,rollout", [(_abi.KIND_FULL, 0), (_abi.KIND_KINO, 0), (_abi.KIND_CENT, 0), (_abi.KIND_KINO, 1)])
def test_emulated_walking_batch_matches_oracle_per_instance(oracle, kind, rollout):
    """Horizons of the reference gait (single support, moving references, active cone / box rows) with per-instance models."""
    prob = _with_solver_consts(problems.walk_batch(kind, 2, seed=2, T=40, ticks=[15, 90], mirror=[False, True]), rollout)
    assert 0.1 < prob["ds_fraction"] < 0.9
    robots, cfgs = hetero_models(prob, 2)
    e = emu_models_lib.solve_models(prob, robots, cfgs, 4)
    ref = oracle_per_instance(oracle, prob, robots, cfgs, 4)
    _check(e["xs"], e["us"], e["K"], [i.num_iters for i in e["info"]], ref, e["vs"])
    assert [i.ls_evals for i in e["info"]] == [i.ls_evals for i in ref["info"]]
    if kind != _abi.KIND_CENT:  # (the centroidal horizons keep every cone row inactive in these iterations)
        assert np.abs(ref["vs"]).max() > 0  # constraints are active


def test_emulated_identical_copies_equal_the_shared_model():
    prob = problems.walk_batch(_abi.KIND_FULL, 2, seed=3, T=20, ticks=[60, 99], mirror=[False, True])
    B = 2
    a = emu_lib.solve(prob, 3)
    b = emu_models_lib.solve_models(prob, [prob["robot"]] * B, [prob["cfg"]] * B, 3)
    c = emu_models_lib.solve_models(prob, None, [prob["cfg"]] * B, 3)
    for k in ("xs", "us", "K", "vs", "lams"):
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], c[k]), k


def _rejected(prob, robots, cfgs):
    with pytest.raises(emu_models_lib.EmuError) as ei:
        emu_models_lib.solve_models(prob, robots, cfgs, 1)
    return str(ei.value)


@pytest.mark.parametrize("field,value", [("kind", _abi.KIND_KINO), ("T", 5), ("dt", 0.02), ("tol", 1e-4), ("mu_init", 1e-6), ("max_iters", 7),
                                         ("force_initial_condition", 0), ("rollout", 1), ("lq_legs", 2)])
def test_validation_rejects_a_differing_config_constant(field, value):
    prob = problems.full_standing_problem(batch=3, T=4)
    cfgs = [_copy(prob["cfg"]) for _ in range(3)]
    setattr(cfgs[1], field, value)
    msg = _rejected(prob, None, cfgs)
    assert "instance 1" in msg and f"cfg.{field}" in msg, msg


@pytest.mark.parametrize("field", ["parent", "foot_body"])
def test_validation_rejects_a_differing_topology(field):
    prob = problems.full_standing_problem(batch=3, T=4)
    robots = [_copy(prob["robot"]) for _ in range(3)]
    if field == "parent":
        robots[2].parent[22] = 15  # still parents-first: only the comparison with the shared tree catches it
    else:
        robots[2].foot_body[1] = 11
    msg = _rejected(prob, robots, None)
    assert "instance 2" in msg and f"robot.{field}" in msg, msg


def test_perturbed_robots_keep_kinematics_and_valid_inertia():
    rb = problems.base_setup()[0]
    rs = problems.perturbed_robots(rb, 16, seed=0, mass=0.2, com=0.01, payload=5.0)
    assert len(rs) == 16 and len({round(sum(r.mass), 9) for r in rs}) == 16
    for r in rs:
        assert np.array_equal(np.asarray(r.jplace), np.asarray(rb.jplace)) and np.array_equal(np.asarray(r.foot_place), np.asarray(rb.foot_place))
        for b in range(rb.nb):
            ev = np.linalg.eigvalsh(np.asarray(r.inertia[b][:]).reshape(3, 3))
            assert r.mass[b] > 0 and ev.min() > 0 and ev.sum() - 2 * ev.max() >= -1e-12  # positive, triangle inequality
    assert [r.mass[5] for r in problems.perturbed_robots(rb, 4, seed=0)] == [r.mass[5] for r in problems.perturbed_robots(rb, 4, seed=0)]  # seeded


# ---------------------------------------------------------------- GPU
def _solver(prob, robots=None, cfgs=None):
    from mpc_benchmark_b200.batch import BatchSolver

    B = prob["x0"].shape[0]
    s = BatchSolver(prob["robot"], prob["cfg"], B)
    if robots is not None or cfgs is not None:
        s.set_instance_models(robots, cfgs)
    s.setup(prob["knots"], prob["terms"], prob["x0"])
    return s


def _perturbed(prob, oracle, seed, sx=0.005, su=0.5):
    rng = np.random.default_rng(seed)
    xs, us = prob["xs"].copy(), prob["us"].copy()
    for b in range(xs.shape[0]):
        for k in range(xs.shape[1]):
            xs[b, k] = xs[b, k] + rng.normal(size=9) * sx if prob["cfg"].kind == _abi.KIND_CENT else oracle.integrate(xs[b, k], rng.normal(size=56) * sx)
    us += rng.normal(size=us.shape) * su
    return xs, us


@pytest.mark.gpu
@pytest.mark.parametrize("maker", [problems.cent_standing_problem, problems.full_standing_problem, problems.kino_standing_problem])
def test_gpu_lq_blocks_match_oracle_per_instance(oracle, maker):
    prob = maker(batch=2, T=8)
    cfg = prob["cfg"]
    nx, n, m, nc = _abi.DIMS[cfg.kind]
    xs, us = _perturbed(prob, oracle, 3, sx=0.02, su=1.0)
    robots, cfgs = hetero_models(prob, 3)
    s = _solver(prob, robots, cfgs)
    for inst in range(2):
        d = s.debug_lq(xs, us, inst)
        x = xs[inst].copy()
        x[0] = prob["x0"][inst]
        for k in range(cfg.T):
            o = oracle.eval_knot(robots[inst], cfgs[inst], prob["knots"][inst * cfg.T + k], x[k], us[inst, k], x[k + 1])
            assert np.abs(np.hstack([o["A"], o["B"]]) - d["AB"][k]).max() < 1e-9
            H = o["H"] + 1e-9 * np.eye(n + m)
            assert np.abs(H - d["H"][k]).max() <= 1e-9 * max(1.0, np.abs(H).max())
            assert np.abs(o["gap"] - d["gap"][k]).max() < 1e-10
            assert np.abs(o["h"] - d["h"][k]).max() < 1e-8
            assert abs(o["cost"] - d["scal"][k, 0]) <= 1e-10 * max(1.0, abs(o["cost"]))
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("maker,T,rollout,lq_legs", [(problems.cent_standing_problem, 100, 0, 0), (problems.full_standing_problem, 30, 0, 0),
                                                     (problems.kino_standing_problem, 30, 0, 0), (problems.full_standing_problem, 30, 1, 0),
                                                     (problems.kino_standing_problem, 30, 1, 0), (problems.full_standing_problem, 30, 0, 4)])
def test_gpu_cold_solve_and_tick_match_oracle_per_instance(oracle, maker, T, rollout, lq_legs):
    prob = _with_solver_consts(maker(batch=3, T=T), rollout, lq_legs)
    robots, cfgs = hetero_models(prob, 4)
    s = _solver(prob, robots, cfgs)
    res = s.run(prob["xs"], prob["us"], max_iters=100)
    ref = oracle_per_instance(oracle, prob, robots, cfgs, 100)
    _check(res.xs, res.us, res.K, res.num_iters, ref)
    # one-iteration tick from a perturbed warm start
    xs, us = _perturbed(prob, oracle, 5)
    prob["x0"] = xs[:, 0].copy()
    s.set_x0(prob["x0"])
    s.reset_multipliers()
    res = s.run(xs, us, max_iters=1)
    ref = oracle_per_instance(oracle, prob, robots, cfgs, 1, xs=xs, us=us)
    _check(res.xs, res.us, res.K, res.num_iters, ref)
    s.close()


@pytest.mark.gpu
def test_gpu_identical_copies_are_bitwise_the_shared_path():
    prob = problems.walk_batch(_abi.KIND_FULL, 12, seed=6, T=40)
    B = 12
    out = []
    for models in (None, ([prob["robot"]] * B, [prob["cfg"]] * B)):
        s = _solver(prob, *(models or (None, None)))
        r = s.run(prob["xs"], prob["us"], max_iters=4)
        xs_o, us_o = np.zeros_like(r.xs), np.zeros_like(r.us)
        K0 = np.zeros((B, s.m, s.n))
        s.reset_multipliers()
        inf = s.run_pipelined(prob["xs"], prob["us"], xs_o, us_o, K0, max_iters=4, parts=2, info=True)
        out.append((r, xs_o, us_o, K0, [bytes(i) for i in inf]))
        s.close()
    (a, *pa), (b, *pb) = out
    for k in ("xs", "us", "K", "vs", "lams"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert [bytes(i) for i in a.info] == [bytes(i) for i in b.info]
    for x, y in zip(pa, pb):
        assert np.array_equal(np.asarray(x), np.asarray(y))


@pytest.mark.gpu
def test_gpu_heterogeneous_instance_equals_homogeneous_batch_of_its_model():
    """Every launch of a batch of 8 has the same Riccati shape (<= 148 instances), so instance i of the heterogeneous batch and instance i
    of a homogeneous batch built on (robot_i, cfg_i) run the same arithmetic: bit for bit equal."""
    from mpc_benchmark_b200.batch import BatchSolver

    B = 8
    prob = problems.walk_batch(_abi.KIND_FULL, B, seed=7, T=40)
    robots, cfgs = hetero_models(prob, 7)
    s = _solver(prob, robots, cfgs)
    het = s.run(prob["xs"], prob["us"], max_iters=3)
    s.close()
    for i in range(B):
        h = BatchSolver(robots[i], cfgs[i], B)
        h.setup(prob["knots"], prob["terms"], prob["x0"])
        hom = h.run(prob["xs"], prob["us"], max_iters=3)
        for k in ("xs", "us", "K", "vs", "lams"):
            assert np.array_equal(getattr(het, k)[i], getattr(hom, k)[i]), (i, k)
        assert bytes(het.info[i]) == bytes(hom.info[i])
        h.close()


@pytest.mark.gpu
def test_gpu_gait_tick_places_soles_from_each_robots_kinematics(oracle):
    from mpc_benchmark_b200 import gait

    B, T = 4, 100
    prob = problems.full_standing_problem(batch=B, T=T)
    robots = problems.perturbed_robots(prob["robot"], B, seed=8, jplace=0.01)
    lf0, rf0 = prob["lf"], prob["rf"]
    g = gait.device_gait(_abi.KIND_FULL, lf0, rf0, prob["com0"], prob["mass"])
    mirror = [False, True, False, True]
    solvers = []
    for _ in range(2):
        s = _solver(prob, robots)
        s.run(prob["xs"], prob["us"], max_iters=2)
        s.gait_setup(g, mirror)
        solvers.append(s)
    xs1 = solvers[0].results().xs[:, 1]
    assert np.array_equal(xs1, solvers[1].results().xs[:, 1])
    kin = [oracle.kinematics(robots[i], xs1[i]) for i in range(B)]
    lf, rf = np.array([k["lf"] for k in kin]), np.array([k["rf"] for k in kin])
    assert np.ptp(lf[:, 9:12], axis=0).max() > 1e-3  # the robots' soles really differ
    for t in range(45):
        solvers[0].gait_tick()
        solvers[1].gait_tick(lf, rf)
        if t % 4 == 0 or t in (29, 30, 31):
            (ka, ta), (kb, tb) = solvers[0].knots(), solvers[1].knots()
            da = np.frombuffer(bytes(ka), float) - np.frombuffer(bytes(kb), float)
            dt = np.frombuffer(bytes(ta), float) - np.frombuffer(bytes(tb), float)
            assert np.abs(da).max() < 1e-12 and np.abs(dt).max() < 1e-12, t
    for s in solvers:
        s.close()


@pytest.mark.gpu
def test_gpu_rbd_and_ikid_terms_per_robot(oracle):
    from test_ikid_from_state import _states

    from mpc_benchmark_b200 import pin

    x = _states(n_random=4)  # 12 states
    B = x.shape[0]
    prob = problems.full_standing_problem(batch=B, T=4)
    robots = problems.perturbed_robots(prob["robot"], B, seed=9, payload=3.0, jplace=0.01)
    s = _solver(prob, robots)
    r = s.rbd_terms(x)
    model = pin.load_talos_like()[0]
    ids = [model.getFrameId("base_link"), model.getFrameId("torso_2_link")]
    fb, fp = [model.frames[i].parentJoint - 1 for i in ids], np.array([model.frames[i].placement.to12() for i in ids])
    M, rbd = s.ikid_terms(x, list(zip(fb, fp)))
    for i in range(B):
        kin = oracle.kinematics(robots[i], x[i])
        assert np.abs(r["M"][i] - kin["M"]).max() < 1e-10 * np.abs(kin["M"]).max()
        assert np.abs(r["nle"][i] - kin["b"]).max() < 1e-10 * np.abs(kin["b"]).max()
        e = emu_lib.rbd_terms(robots[i], prob["cfg"], x[i:i + 1])
        for k in ("M", "nle", "Jc", "dJv", "vf"):
            assert np.abs(r[k][i] - e[k][0]).max() <= 1e-12 * max(1.0, np.abs(e[k]).max()), (i, k)
        o = oracle.ikid_terms(robots[i], x[i:i + 1], fb, fp)
        assert np.abs(rbd.Ag[i] - o["Ag"][0]).max() < 1e-9 * np.abs(o["Ag"]).max()
        assert np.abs(np.stack([rbd.J_base[i], rbd.J_torso[i]]) - o["Jang"][0]).max() < 1e-9
        assert np.array_equal(M[i], r["M"][i])
    # the shared robot would give other terms
    assert np.abs(r["M"] - s.__class__(prob["robot"], prob["cfg"], B).rbd_terms(x)["M"]).max() > 1e-3
    for bad in (x[:B - 1], np.concatenate([x, x[:1]])):
        with pytest.raises(RuntimeError, match="count must equal the solver batch"):
            s.rbd_terms(bad)
        with pytest.raises(RuntimeError, match="count must equal the solver batch"):
            s.ikid_terms(bad, list(zip(fb, fp)))
    s.close()


@pytest.mark.gpu
def test_gpu_id_qp_solve_from_state_uses_each_robots_terms():
    """IDSolver_ulim.solve_from_state with a per-instance-model solver of the QP's batch: row i equals the solve with a homogeneous solver of
    robot_i; a QP batch other than the solver batch is rejected."""
    from test_qp import FIXTURE, FOOT_L, FOOT_W, MU

    from mpc_benchmark_b200 import pin, qp_utils
    from mpc_benchmark_b200.batch import BatchSolver

    d = np.load(FIXTURE)
    B = 6
    prob = problems.full_standing_problem(batch=B, T=4)
    robots = problems.perturbed_robots(prob["robot"], B, seed=10, payload=3.0)
    s = _solver(prob, robots)
    model = pin.load_talos_like()[0]
    q = qp_utils.IDSolver_ulim(model, [1, 1], 2, MU, FOOT_L, FOOT_W, [0, 1], 6, False, batch=B)
    args = (d["x"][:B], d["cs"][:B], d["a"][:B], d["forces"][:B])
    got = np.concatenate(q.solve_from_state(s, *args), axis=1)
    for i in range(B):
        h = BatchSolver(robots[i], prob["cfg"], B)
        ref = np.concatenate(q.solve_from_state(h, *args), axis=1)
        assert np.array_equal(got[i], ref[i]), i
        h.close()
    q.qp.close()
    q5 = qp_utils.IDSolver_ulim(model, [1, 1], 2, MU, FOOT_L, FOOT_W, [0, 1], 6, False, batch=B - 1)
    with pytest.raises(RuntimeError, match="count must equal the solver batch"):
        q5.solve_from_state(s, *(a[:B - 1] for a in args))
    q5.qp.close()
    s.close()


@pytest.mark.gpu
def test_gpu_instance_model_error_paths():
    prob = problems.full_standing_problem(batch=3, T=8)
    robots, cfgs = hetero_models(prob, 11)
    s = _solver(prob)
    base = s.workspace_bytes
    for bad in ((robots[:2], None), (None, cfgs + cfgs[:1])):
        with pytest.raises(ValueError, match="expected 3"):
            s.set_instance_models(*bad)
    wrong = [_copy(c) for c in cfgs]
    wrong[2].T = 9
    with pytest.raises(RuntimeError, match="instance 2: cfg.T"):
        s.set_instance_models(None, wrong)
    s.set_instance_models(robots, cfgs)
    assert s.workspace_bytes > base
    with pytest.raises(RuntimeError, match="clear them first"):
        s.reconfigure(prob["robot"], prob["cfg"])
    het = s.run(prob["xs"], prob["us"], max_iters=5)
    s.set_instance_models(None, None)  # back to the shared model
    s.reconfigure(prob["robot"], prob["cfg"])
    s.reset_multipliers()  # every run below starts from zero multipliers, as the first one did
    shared = s.run(prob["xs"], prob["us"], max_iters=5)
    ref = _solver(prob).run(prob["xs"], prob["us"], max_iters=5)
    assert np.array_equal(shared.xs, ref.xs) and np.array_equal(shared.us, ref.us)
    assert not np.array_equal(het.us, ref.us)
    s.set_instance_models(robots, cfgs)  # set again: the same models as before
    s.reset_multipliers()
    again = s.run(prob["xs"], prob["us"], max_iters=5)
    assert np.array_equal(again.xs, het.xs)
    s.close()
