"""Time-parallel LQ solve (cfg.lq_legs >= 2, csrc/riccati_par.cuh): the horizon cut into legs must give the serial Riccati
solve's step and gains up to rounding (SURVEY 7.3 'serial = parallel-legs')."""
import ctypes as C

import numpy as np
import pytest

import emu_lib
from mpc_benchmark_b200 import _abi, _native, problems
from test_lq import dense_kkt_solution, random_lq


def rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(1e-300, np.abs(np.asarray(b)).max()))


def _lq_case(n, m, nc, T, mu, legs):
    rng = np.random.default_rng(n + T)
    H, g, AB, f, CD, d, E6, HT, gT = random_lq(rng, n, m, nc, T, 5)
    # active rows on both knots around every boundary: random_lq already activates rows on every knot; a terminal constraint
    CT, dT = rng.normal(size=(3, n)), rng.normal(size=3) * 0.01
    return (n, m, nc, T, mu, mu, H, g, AB, f, CD, d, E6, HT, gT, CT, dT)


@pytest.mark.parametrize("n,m,nc,T", [(9, 12, 34, 7), (14, 5, 8, 9), (56, 22, 78, 7)])
@pytest.mark.parametrize("mu", [1e-2, 1e-8])
@pytest.mark.parametrize("legs", [2, 3, 7, "T"])
def test_oracle_legs_match_serial_and_dense_kkt(oracle, n, m, nc, T, mu, legs):
    L = T if legs == "T" else legs
    args = _lq_case(n, m, nc, T, mu, L)
    E6 = args[12] if n >= 6 else None
    a = list(args)
    a[12] = E6
    o = oracle.riccati(*a)
    p = oracle.riccati_par(*a, legs=L)
    dxs, dus, dvs, dls, dvT = dense_kkt_solution(*a)
    assert not np.allclose(args[12].reshape(-1, 6, 6)[0], -np.eye(6))  # E6 != -I
    sc = max(1.0, np.abs(dxs).max(), np.abs(dus).max())
    # against the dense KKT solution: test_lq's tolerances, or the serial recursion's own distance to it where the system is worse
    # conditioned than test_lq's cases (longer horizons at mu = 1e-8)
    for key, ref, sl, tol in (("dxs", dxs, np.s_[:], 1e-7 * sc), ("dus", dus, np.s_[:], 1e-7 * sc), ("dlams", dls, np.s_[1:], 1e-6 * max(1.0, np.abs(dls).max())),
                              ("dvs", dvs, np.s_[:T], 1e-6 * max(1.0, np.abs(dvs).max())), ("dvs", dvT, np.s_[T, :3], 1e-6 * max(1.0, np.abs(dvT).max()))):
        e_o, e_p = np.abs(o[key][sl] - ref).max(), np.abs(p[key][sl] - ref).max()
        assert e_p < max(tol, 4 * e_o), (key, e_p, e_o, tol)
        # legs against serial: within the serial solve's own rounding error
        assert np.abs(p[key][sl] - o[key][sl]).max() < max(tol, 4 * e_o), key
    assert np.abs(p["K"] - o["K"]).max() < 1e-8 * max(1.0, np.abs(o["K"]).max())


# emulated solver: every kind, both rollouts; the walking horizons of the reference gaits
EMU_TOL, EMU_TOL_K = 1e-8, 1e-8


def _emu_case(kind, batch):
    T = 100 if kind == _abi.KIND_CENT else 20
    return problems.walk_batch(kind, batch, seed=3, T=T)


@pytest.mark.parametrize("kind", [_abi.KIND_CENT, _abi.KIND_FULL, _abi.KIND_KINO])
@pytest.mark.parametrize("rollout", [0, 1])
def test_emulated_solver_legs_match_serial(kind, rollout):
    prob = _emu_case(kind, 2)

    def solve(legs):
        cfg = _abi.Config.from_buffer_copy(prob["cfg"])
        cfg.lq_legs, cfg.rollout = legs, rollout
        return emu_lib.solve(dict(prob, cfg=cfg), max_iters=3)

    ref = solve(0)
    for L in (2, 4, 8):
        r = solve(L)
        assert [(i.num_iters, i.status, i.ls_evals) for i in r["info"]] == [(i.num_iters, i.status, i.ls_evals) for i in ref["info"]], L
        for k in ("xs", "us", "vs", "lams"):
            assert rel(r[k], ref[k]) < EMU_TOL, (L, k, rel(r[k], ref[k]))
        assert rel(r["K"], ref["K"]) < EMU_TOL_K, (L, rel(r["K"], ref["K"]))
        for a, b in zip(r["info"], ref["info"]):
            assert abs(a.merit - b.merit) <= EMU_TOL * max(1.0, abs(b.merit))
            assert abs(a.prim_infeas - b.prim_infeas) <= EMU_TOL * max(1.0, abs(b.prim_infeas)) + 1e-12


def test_abi_keeps_config_size():
    assert C.sizeof(_abi.Config) % 8 == 0
    assert _abi.Config.lq_legs.offset == _abi.Config.rollout.offset + 4


# ---- on the device
RTOL = 1e-6


def _solver(prob, legs, batch):
    from mpc_benchmark_b200.batch import BatchSolver

    cfg = _abi.Config.from_buffer_copy(prob["cfg"])
    cfg.lq_legs = legs
    s = BatchSolver(prob["robot"], cfg, batch)
    s.setup(prob["knots"], prob["terms"], prob["x0"])
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("bad", [-1, 17, 31])
def test_argument_errors(bad):
    from mpc_benchmark_b200.batch import BatchSolver

    prob = problems.cent_standing_problem(batch=1, T=30)
    cfg = _abi.Config.from_buffer_copy(prob["cfg"])
    cfg.lq_legs = bad
    with pytest.raises(_native.NativeError, match="lq_legs"):
        BatchSolver(prob["robot"], cfg, 1)
    s = BatchSolver(prob["robot"], prob["cfg"], 1)
    with pytest.raises(_native.NativeError, match="lq_legs"):
        s.reconfigure(prob["robot"], cfg)
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [_abi.KIND_CENT, _abi.KIND_FULL, _abi.KIND_KINO])
def test_device_legs_match_serial_cold_and_ticks(oracle, kind):
    B = 3
    prob = problems.walk_batch(kind, B, seed=4, T=100 if kind == _abi.KIND_CENT else 40)
    iters = 8
    outs = {}
    for L in (0, 2, 4, 8, 16):
        s = _solver(prob, L, B)
        cold = s.run(prob["xs"], prob["us"], max_iters=iters)
        ticks = []
        for _ in range(5):
            s.tick(max_iters=1)
            ticks.append(s.results())
        outs[L] = (cold, ticks)
        s.close()
    ref = oracle.solve(prob, max_iters=iters)
    assert rel(outs[0][0].xs, ref["xs"]) < RTOL and rel(outs[0][0].us, ref["us"]) < RTOL
    c0, t0 = outs[0]
    for L in (2, 4, 8, 16):
        c, t = outs[L]
        for a, b in [(c, c0)] + list(zip(t, t0)):
            assert list(a.num_iters) == list(b.num_iters), L
            assert [i.status for i in a.info] == [i.status for i in b.info], L
            assert rel(a.xs, b.xs) < RTOL and rel(a.us, b.us) < RTOL, (L, rel(a.xs, b.xs), rel(a.us, b.us))
            assert rel(a.K[:, 0], b.K[:, 0]) < RTOL, (L, rel(a.K[:, 0], b.K[:, 0]))
        assert rel(c.xs, ref["xs"]) < RTOL and rel(c.us, ref["us"]) < RTOL


@pytest.mark.gpu
def test_device_legs_mixed_batch():
    """Instances that converge at different iterations, so later passes run the legs over compacted instance lists (the list
    handling is the same for every model kind; the centroidal walking batch is one whose instances finish at 14 to 30 iterations)."""
    B = 6
    prob = problems.walk_batch(_abi.KIND_CENT, B, seed=7, T=100)
    s0 = _solver(prob, 0, B)
    r0 = s0.run(prob["xs"], prob["us"], max_iters=40)
    s0.close()
    assert len(set(r0.num_iters)) > 1  # really a mixed batch
    for L in (4, 16):
        s = _solver(prob, L, B)
        r = s.run(prob["xs"], prob["us"], max_iters=40)
        s.close()
        assert list(r.num_iters) == list(r0.num_iters), L
        assert [i.status for i in r.info] == [i.status for i in r0.info], L
        assert rel(r.xs, r0.xs) < RTOL and rel(r.us, r0.us) < RTOL and rel(r.K[:, 0], r0.K[:, 0]) < RTOL, L


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [_abi.KIND_CENT, _abi.KIND_FULL])
def test_device_legs_deterministic(kind):
    """Two runs from the same starting point are bitwise equal (every boundary entry has one writer)."""
    B = 4
    prob = problems.walk_batch(kind, B, seed=7, T=100 if kind == _abi.KIND_CENT else 30)
    rs = []
    for _ in range(2):  # two handles: a second run on one handle would start from the first run's multipliers
        s = _solver(prob, 4, B)
        rs.append(s.run(prob["xs"], prob["us"], max_iters=10))
        s.close()
    r1, r2 = rs
    for k in ("xs", "us", "K", "vs", "lams"):
        assert np.array_equal(getattr(r1, k), getattr(r2, k)), k
