"""ctypes bindings of the time-parallel LQ test libraries built from tests/lqpar/ (tests/_emu/liblq_par_{oracle,emu}.so): the CPU
restatement of the leg-parallel Riccati solve, and the solver's kernel SOURCES with lq_legs run serially on the host.
TEST-ONLY: never loaded by the product."""
import ctypes as C
import os
import subprocess

import numpy as np

from mpc_benchmark_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
dp = C.POINTER(C.c_double)
_libs = {}


def _lib(name):
    if name not in _libs:
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "lqpar")], stdout=subprocess.DEVNULL)
        _libs[name] = C.CDLL(os.path.join(ROOT, "tests", "_emu", f"lib{name}.so"))
    return _libs[name]


def _p(a):
    return a.ctypes.data_as(dp) if a is not None else None


def riccati_par(n, m, nc, T, mu_d, mu, H, g, AB, f, CD, d, E6, HT, gT, CT=None, dT=None, legs=2):
    """The oracle's leg-parallel LQ solve; the same outputs as oracle_lib.riccati."""
    nct = 0 if CT is None else CT.shape[0]
    s = m + nc
    o = dict(dxs=np.zeros((T + 1, n)), dus=np.zeros((T, m)), dvs=np.zeros((T + 1, nc)), dlams=np.zeros((T + 1, n)), K=np.zeros((T, s, 1 + n)))
    args = [np.ascontiguousarray(a, float) if a is not None else None for a in (H, g, AB, f, CD, d, E6, HT, gT, CT, dT)]
    _lib("lq_par_oracle").orc_riccati_par(n, m, nc, T, C.c_double(mu_d), C.c_double(mu), *[_p(a) for a in args], nct, int(legs),
                                          _p(o["dxs"]), _p(o["dus"]), _p(o["dvs"]), _p(o["dlams"]), _p(o["K"]))
    return o


def emu_solve(prob, lq_legs, max_iters=None, rollout=None):
    """The host emulation of the solver's kernel sources on a problem dict of mpc_benchmark_b200.problems, with cfg.lq_legs = lq_legs
    (and cfg.rollout = rollout when given).  Returns dict(xs, us, K, vs, lams, info)."""
    cfg = _abi.Config.from_buffer_copy(prob["cfg"])
    cfg.lq_legs = int(lq_legs)
    if rollout is not None:
        cfg.rollout = int(rollout)
    nx, n, m, nc = _abi.DIMS[cfg.kind]
    T = cfg.T
    B = prob["x0"].shape[0]
    xs = np.ascontiguousarray(prob["xs"], float).copy()
    us = np.ascontiguousarray(prob["us"], float).copy()
    K = np.zeros((B, T, m, n))
    vs = np.zeros((B, T + 1, nc))
    lams = np.zeros((B, T + 1, n))
    info = (_abi.Info * B)()
    rc = _lib("lq_par_emu").emu_solve_legs(C.byref(prob["robot"]), C.byref(cfg), B, prob["knots"], prob["terms"],
                                           _p(np.ascontiguousarray(prob["x0"], float)), _p(xs), _p(us), _p(K), _p(vs), _p(lams), info,
                                           int(cfg.max_iters if max_iters is None else max_iters))
    assert rc == 0
    return dict(xs=xs, us=us, K=K, vs=vs, lams=lams, info=info)
