"""IKID QP (IKIDSolver_f6, QP_utils.py:584-768) assembled and solved from measured states on the device: the task terms of
csrc/rbd_terms.cuh (ikid_terms_group: Ag, dAg v, LOCAL angular Jacobians of the base / torso frames and their dJ v), the cost and
constraint assembly of csrc/qp.cuh (qp_assemble_ikid_group) and `IKIDSolver_f6.solve_from_state`.

CPU (`-m "not gpu"`): the oracle's task terms (orc_ikid_terms in oracle/capi.cpp, on oracle/rbd.hpp) against central differences, the base-frame known answer, and the kernel sources run
serially under the host emulation (tests/emu/emu.cpp) against the oracle and the literal cost formulas.  GPU (`-m gpu`): the device path against the
emulation, the oracle and the host-assembled `solve`."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import emu_lib
import oracle_lib

from test_qp import FIXTURE, FOOT_L, FOOT_W, MU, _ikid_reference_cost

NV = 28


def _frames(model):
    """(body, placement 12) of the base_link and torso_2_link frames, as IKIDSolver_f6 derives them from frame ids."""
    ids = [model.getFrameId("base_link"), model.getFrameId("torso_2_link")]
    return ids, [model.frames[i].parentJoint - 1 for i in ids], np.array([model.frames[i].placement.to12() for i in ids])


@pytest.fixture(scope="module")
def setup():
    from mpc_benchmark_b200 import pin, problems

    model = pin.load_talos_like()[0]
    prob = problems.full_standing_problem(batch=1, T=4)
    ids, fb, fp = _frames(model)
    return dict(model=model, robot=prob["robot"], cfg=prob["cfg"], ids=ids, fb=fb, fp=fp)


def _states(n_random=4, seed=3):
    """Eight fixture states, then seeded random ones: any base orientation, joints around the fixture posture, velocities of order 1."""
    fx = np.load(FIXTURE)["x"][:8]
    rng = np.random.default_rng(seed)
    x = np.zeros((n_random, 57))
    x[:, :3] = rng.normal(0, 0.3, (n_random, 3))
    quat = rng.normal(size=(n_random, 4))
    x[:, 3:7] = quat / np.linalg.norm(quat, axis=1, keepdims=True)
    x[:, 7:29] = fx[0, 7:29] + rng.normal(0, 0.4, (n_random, 22))
    x[:, 29:] = rng.normal(0, 1.0, (n_random, 28))
    return np.concatenate([fx, x])


# ------------------------------------------------------------------------------------------------ oracle against differences (CPU)
def test_oracle_ikid_terms_match_central_differences(oracle, setup):
    rb, fb, fp = setup["robot"], setup["fb"], setup["fp"]
    for x in _states():
        o = oracle_lib.ikid_terms(rb, x, fb, fp)
        Ag, dAgv, Jang, dJang = o["Ag"][0], o["dAgv"][0], o["Jang"][0], o["dJang"][0]
        hg = lambda xx: oracle.kinematics(rb, xx)["hg"]  # noqa: E731
        # Ag = d h_g / d v: h_g is linear in v, so the difference is exact up to rounding
        h = 1e-3
        fd = np.zeros((6, NV))
        for j in range(NV):
            xp, xm = x.copy(), x.copy()
            xp[29 + j] += h
            xm[29 + j] -= h
            fd[:, j] = (hg(xp) - hg(xm)) / (2 * h)
        assert np.abs(fd - Ag).max() < 1e-10 * np.abs(Ag).max()
        # dA_g v = d/dt h_g along (q + t v, v)
        v = x[29:]
        along = lambda t: oracle.integrate(x, np.concatenate([t * v, np.zeros(NV)]))  # noqa: E731
        t = 1e-5
        fd = (hg(along(t)) - hg(along(-t))) / (2 * t)
        assert np.abs(fd - dAgv).max() < 1e-6 * max(1.0, np.abs(dAgv).max())
        # angular Jacobian columns: log3(R(q)' R(q + h e_j)) / h, central
        R = lambda xx: oracle_lib.ikid_terms(rb, xx, fb, fp)["oMf"][0, :, :9].reshape(2, 3, 3)  # noqa: E731
        R0, h = R(x), 1e-6
        for j in range(NV):
            e = np.zeros(2 * NV)
            e[j] = h
            Rp, Rm = R(oracle.integrate(x, e)), R(oracle.integrate(x, -e))
            for f in range(2):
                col = (Rotation.from_matrix(R0[f].T @ Rp[f]).as_rotvec() - Rotation.from_matrix(R0[f].T @ Rm[f]).as_rotvec()) / (2 * h)
                assert np.abs(col - Jang[f, :, j]).max() < 1e-7
        # dJ v = d/dt (Jang(q + t v) v)
        Jv = lambda t: oracle_lib.ikid_terms(rb, along(t), fb, fp)["Jang"][0] @ v  # noqa: E731
        fd = (Jv(t) - Jv(-t)) / (2 * t)
        assert np.abs(fd - dJang).max() < 1e-6 * max(1.0, np.abs(dJang).max())


def test_base_frame_known_answer(setup):
    """base_link is body 0 with the identity placement: its LOCAL angular Jacobian is [0 | I | 0] and its dJ v is zero."""
    x = _states()
    expect = np.zeros((3, NV))
    expect[:, 3:6] = np.eye(3)
    for o in (oracle_lib.ikid_terms(setup["robot"], x, setup["fb"], setup["fp"]),
              emu_lib.ikid_terms(setup["robot"], setup["cfg"], x, setup["fb"], setup["fp"])):
        Jb = o["Jang"][:, 0]
        assert not Jb[:, :, :3].any() and not Jb[:, :, 6:].any()  # exact zeros off the angular base columns
        assert np.abs(Jb - expect).max() < 1e-15  # R' R e_j: identity to rounding
        assert not o["dJang"][:, 0].any()


# ------------------------------------------------------------------------------------------------ kernel sources, emulated (CPU)
def _check_against_oracle(o, ref):
    for k in ("Ag", "dAgv", "Jang", "dJang"):
        assert np.abs(o[k] - ref[k]).max() <= 1e-12 * max(1.0, np.abs(ref[k]).max()), k


def test_emulated_ikid_terms_match_oracle_and_rbd_terms(setup):
    x = _states()
    e = emu_lib.ikid_terms(setup["robot"], setup["cfg"], x, setup["fb"], setup["fp"])
    _check_against_oracle(e, oracle_lib.ikid_terms(setup["robot"], x, setup["fb"], setup["fp"]))
    r = emu_lib.rbd_terms(setup["robot"], setup["cfg"], x)
    for k in ("M", "nle", "Jc", "dJv"):
        assert np.array_equal(e[k], r[k]), k


def test_emulated_sole_frame_rows_equal_contact_jacobian(setup):
    """Named as frames, the soles give the angular rows of the contact Jacobians and of dJ v, bit for bit."""
    rb = setup["robot"]
    x = _states()
    fp = np.array([rb.foot_place[0][:], rb.foot_place[1][:]])
    e = emu_lib.ikid_terms(rb, setup["cfg"], x, [rb.foot_body[0], rb.foot_body[1]], fp)
    Jc = e["Jc"].reshape(-1, 2, 6, NV)
    assert np.array_equal(e["Jang"], Jc[:, :, 3:])
    assert np.abs(e["dJang"] - e["dJv"].reshape(-1, 2, 6)[:, :, 3:]).max() < 1e-15


def _gains(rng, offdiag=True):
    """K_gains with general (non-diagonal) matrices, as [[Kp_q, Kd_q], [Kp_f, Kd_f], None, [Kp_b, Kd_b]]."""
    def K(k, m):
        return np.eye(m) * k + (rng.normal(0, 0.1 * k, (m, m)) if offdiag else 0.0)
    return [[K(100, NV), K(20, NV)], [K(400, 6), K(40, 6)], None, [K(100, 3), K(20, 3)]]


def _pack(K):
    return np.concatenate([np.asarray(k, float).ravel() for k in (K[0][0], K[0][1], K[1][0], K[1][1], K[3][0], K[3][1])])


def _task(t, B):
    return np.concatenate([t[k].reshape(B, -1) for k in ("q_diff", "dq_diff", "LF_diff", "dLF_diff", "RF_diff", "dRF_diff", "base_diff", "dbase_diff",
                                                          "torso_diff", "dtorso_diff", "dH")], axis=1)


def _task_inputs(B, seed=9):
    """PD errors and dH seeded like test_qp._ikid_inputs, on the fixture states tiled to B."""
    d = np.load(FIXTURE)
    rng = np.random.default_rng(seed)
    reps = -(-B // d["x"].shape[0])
    tile = lambda a: np.ascontiguousarray(np.tile(a, (reps,) + (1,) * (a.ndim - 1))[:B])  # noqa: E731
    t = dict(x=tile(d["x"]), cs=tile(d["cs"]), forces=tile(d["forces"]), dH=rng.normal(0, 1.0, (B, 6)),
             q_diff=rng.normal(0, 0.02, (B, 28)), dq_diff=rng.normal(0, 0.05, (B, 28)), LF_diff=rng.normal(0, 0.01, (B, 6)), dLF_diff=rng.normal(0, 0.02, (B, 6)),
             RF_diff=rng.normal(0, 0.01, (B, 6)), dRF_diff=rng.normal(0, 0.02, (B, 6)), base_diff=rng.normal(0, 0.02, (B, 3)), dbase_diff=rng.normal(0, 0.05, (B, 3)),
             torso_diff=rng.normal(0, 0.02, (B, 3)), dtorso_diff=rng.normal(0, 0.05, (B, 3)))
    t["K_gains"] = _gains(rng)
    t["weights"] = [1.0, 100.0, 0.1, 10.0, 1e-3]
    return t


def _with_terms(t, o):
    """t plus the rigid-body / task terms o (arrays of ikid_terms) under the names _ikid_reference_cost reads."""
    t = dict(t)
    t.update(M=o["M"], nle=o["nle"], Jc=o["Jc"], dJv=o["dJv"], Ag=o["Ag"], dAgv=o["dAgv"], J_base=o["Jang"][:, 0], J_torso=o["Jang"][:, 1],
             dJv_base=o["dJang"][:, 0], dJv_torso=o["dJang"][:, 1])
    return t


def test_emulated_ikid_assembly_matches_reference_formulas(setup):
    B = 24
    t = _task_inputs(B)
    o = emu_lib.ikid_terms(setup["robot"], setup["cfg"], t["x"], setup["fb"], setup["fp"])
    t = _with_terms(t, o)
    H, g, A, b, Cm, l = emu_lib.qp_assemble_ikid(o["M"], o["nle"], o["Jc"], o["dJv"], o["Ag"], o["dAgv"], o["Jang"], o["dJang"], _task(t, B), t["forces"],
                                             t["cs"], t["weights"], _pack(t["K_gains"]), MU, FOOT_L, FOOT_W)
    for i in range(B):
        Hr, gr = _ikid_reference_cost(t, i)
        assert np.abs(H[i, :28, :28] - Hr).max() <= 1e-12 * np.abs(Hr).max()
        assert np.abs(g[i, :28] - gr).max() <= 1e-12 * np.abs(gr).max()
        assert np.array_equal(H[i, :28, :28], H[i, :28, :28].T)
        assert np.array_equal(np.diag(H[i])[28:40], np.full(12, t["weights"][4]))
        Hz = H[i].copy()
        Hz[:28, :28] = 0
        Hz[np.arange(28, 40), np.arange(28, 40)] = 0
        assert not Hz.any() and not g[i, 28:].any()
    gamma = o["dJv"] * np.repeat(t["cs"], 6, axis=1)
    ref = emu_lib.qp_assemble_id(o["M"], o["nle"], o["Jc"], gamma, np.zeros((B, 28)), t["forces"], t["cs"], MU, FOOT_L, FOOT_W)
    for got, want in zip((A, b, Cm, l), ref):
        assert np.array_equal(got, want)


# ------------------------------------------------------------------------------------------------ the device (GPU)
@pytest.fixture(scope="module")
def device_solver(setup):
    from mpc_benchmark_b200.batch import BatchSolver

    s = BatchSolver(setup["robot"], setup["cfg"], 1)
    yield s
    s.close()


def _ikid_solver(setup, t, B):
    from mpc_benchmark_b200 import qp_utils

    ids = setup["ids"]
    return qp_utils.IKIDSolver_f6(setup["model"], t["weights"], t["K_gains"], 2, MU, FOOT_L, FOOT_W, [0, 1], ids[0], ids[1], 6, False, batch=B)


def _solve_from_state(s, dev, t):
    return s.solve_from_state(dev, t["x"], t["cs"], t["q_diff"], t["dq_diff"], t["LF_diff"], t["dLF_diff"], t["RF_diff"], t["dRF_diff"], t["base_diff"],
                              t["dbase_diff"], t["torso_diff"], t["dtorso_diff"], t["forces"], t["dH"])


@pytest.mark.gpu
def test_gpu_ikid_terms_match_emulation_and_oracle(setup, device_solver):
    x = _states()
    M, rbd = device_solver.ikid_terms(x, list(zip(setup["fb"], setup["fp"])))
    d = dict(M=M, nle=rbd.nle, Jc=rbd.Jc, dJv=rbd.dJv, Ag=rbd.Ag, dAgv=rbd.dAgv, Jang=np.stack([rbd.J_base, rbd.J_torso], 1),
             dJang=np.stack([rbd.dJv_base, rbd.dJv_torso], 1))
    e = emu_lib.ikid_terms(setup["robot"], setup["cfg"], x, setup["fb"], setup["fp"])
    _check_against_oracle(d, oracle_lib.ikid_terms(setup["robot"], x, setup["fb"], setup["fp"]))
    _check_against_oracle(d, e)
    r = device_solver.rbd_terms(x)
    for k in ("M", "nle", "Jc", "dJv"):
        assert np.abs(d[k] - e[k]).max() <= 1e-12 * max(1.0, np.abs(e[k]).max()), k
        assert np.array_equal(d[k], r[k]), k  # the same kernel phases as k_rbd_terms


@pytest.mark.gpu
def test_gpu_solve_from_state_matches_host_assembled_solve_and_oracle(oracle, setup, device_solver):
    B = 64
    t = _task_inputs(B)
    s = _ikid_solver(setup, t, B)
    anew, fnew, tau = _solve_from_state(s, device_solver, t)
    r = s.qp.results
    it_ext, it_in, status = r.info.iter_ext.copy(), r.info.iter.copy(), r.info.status.copy()
    assert (status == 0).all()
    x = np.concatenate([anew, fnew - t["forces"], tau], axis=1)
    # the same QPs with the cost assembled on the host from the device's own terms
    M, rbd = device_solver.ikid_terms(t["x"], s._frames())
    v = t["x"][:, 29:]
    a2, f2, tau2 = s.solve(rbd, t["cs"], v, t["q_diff"], t["dq_diff"], t["LF_diff"], t["dLF_diff"], t["RF_diff"], t["dRF_diff"], t["base_diff"], t["dbase_diff"],
                           t["torso_diff"], t["dtorso_diff"], t["forces"], t["dH"], M)
    x2 = np.concatenate([a2, f2 - t["forces"], tau2], axis=1)
    same = (it_ext == s.qp.results.info.iter_ext) & (it_in == s.qp.results.info.iter)
    assert same.mean() >= 0.9
    assert np.abs(x - x2)[same].max() <= 1e-8 * np.abs(x2).max()
    # and the oracle's QP solver on the same assembled QPs
    tt = _with_terms(t, dict(M=M, nle=rbd.nle, Jc=rbd.Jc, dJv=rbd.dJv, Ag=rbd.Ag, dAgv=rbd.dAgv, Jang=np.stack([rbd.J_base, rbd.J_torso], 1),
                             dJang=np.stack([rbd.dJv_base, rbd.dJv_torso], 1)))
    H, g = np.zeros((B, 62, 62)), np.zeros((B, 62))
    for i in range(B):
        H[i, :28, :28], g[i, :28] = _ikid_reference_cost(tt, i)
        H[i, np.arange(28, 40), np.arange(28, 40)] = t["weights"][4]
    gamma = rbd.dJv * np.repeat(t["cs"], 6, axis=1)
    A, b, Cm, l = oracle.qp_assemble_id(M, rbd.nle, rbd.Jc, gamma, np.zeros((B, 28)), t["forces"], t["cs"], MU, FOOT_L, FOOT_W)
    st = oracle.qp_default_settings(eps_abs=1e-3, eps_rel=0.0, max_iter=100, max_iter_in=100, check_duality_gap=1)
    X, _, _, info = oracle.qp_solve(H, g, A, b, Cm, l, np.full(18, 1e5), s.l_box, s.u_box, settings=st)
    same = (it_ext == [i.iter for i in info]) & (it_in == [i.iter_in for i in info])
    assert same.mean() >= 0.9
    assert np.abs(x - X)[same].max() <= 1e-8 * np.abs(X).max()
    s.qp.close()


@pytest.mark.gpu
def test_gpu_solve_from_state_at_batch_4096(setup, device_solver):
    B = 4096
    t = _task_inputs(B)
    s = _ikid_solver(setup, t, B)
    anew, fnew, tau = _solve_from_state(s, device_solver, t)
    r = s.qp.results
    assert (r.info.status == 0).all() and r.info.pri_res.max() <= 1e-3 and r.info.dua_res.max() <= 1e-3
    again = _solve_from_state(s, device_solver, t)
    for u, w in zip((anew, fnew, tau), again):
        assert np.array_equal(u, w)  # identical inputs, identical outputs
    eff = np.asarray(setup["model"].effortLimit, float)[6:]
    assert (np.abs(tau) <= eff + 1e-6).all()  # the torque box holds
    M, rbd = device_solver.ikid_terms(t["x"], s._frames())
    cs = np.repeat(t["cs"], 6, axis=1)
    lhs = np.einsum("bij,bj->bi", M, anew) + rbd.nle - np.einsum("bji,bj->bi", rbd.Jc, fnew * cs)
    lhs[:, 6:] -= tau
    assert np.abs(lhs).max() < 2e-3
    s.qp.close()


@pytest.mark.gpu
def test_gpu_ikid_argument_errors(setup, device_solver):
    from mpc_benchmark_b200 import _native, problems, proxqp, qp_utils
    from mpc_benchmark_b200.batch import BatchSolver

    B = 4
    t = _task_inputs(B)
    s = _ikid_solver(setup, t, B)
    frames = s._frames()
    with pytest.raises(_native.NativeError):  # a frame body out of range
        device_solver.ikid_terms(t["x"], [(23, frames[0][1]), frames[1]])
    with pytest.raises(_native.NativeError):
        device_solver.ikid_terms(t["x"], [(-1, frames[0][1]), frames[1]])
    args = (t["x"], _task(t, B), t["forces"], t["cs"], t["weights"], _pack(t["K_gains"]))
    with pytest.raises(_native.NativeError):
        s.qp.assemble_ikid_from_state(device_solver, *args, [(99, frames[0][1]), frames[1]], MU, FOOT_L, FOOT_W)
    with pytest.raises(_native.NativeError):  # the QP shape without box constraints
        qp_utils.IDSolver_ulim(setup["model"], [1, 1], 2, MU, FOOT_L, FOOT_W, [0, 1], 6, False, batch=B).qp.assemble_ikid_from_state(
            device_solver, *args, frames, MU, FOOT_L, FOOT_W)
    with pytest.raises(_native.NativeError):  # a wrong QP shape
        q = proxqp.dense.BatchQP(20, 4, 6, B, True)
        q.assemble_ikid_from_state(device_solver, *args, frames, MU, FOOT_L, FOOT_W)
    with pytest.raises(_native.NativeError):  # a batch above the handle's capacity
        q = proxqp.dense.BatchQP(62, 40, 18, 2, True)
        q._handle()  # capacity 2
        q.batch = B
        q.assemble_ikid_from_state(device_solver, *args, frames, MU, FOOT_L, FOOT_W)
    cent = problems.cent_standing_problem(batch=1, T=4)
    c = BatchSolver(cent["robot"], cent["cfg"], 1)
    with pytest.raises(_native.NativeError):  # a centroidal solver has no rigid-body tree
        s.qp.assemble_ikid_from_state(c, *args, frames, MU, FOOT_L, FOOT_W)
    with pytest.raises(_native.NativeError):
        c.ikid_terms(t["x"], frames)
    c.close()
    s.qp.close()
