"""ctypes bindings of the CPU oracle (oracle/_build/liboracle.so).  TEST INFRASTRUCTURE ONLY:
nothing under mpc_benchmark_b200/ imports this module."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from mpc_benchmark_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = os.path.join(ROOT, "oracle", "_build", "liboracle.so")

dp = C.POINTER(C.c_double)


def _p(a):
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(dp)


def build():
    srcs = [os.path.join(ROOT, "oracle", f) for f in os.listdir(os.path.join(ROOT, "oracle")) if f.endswith((".cpp", ".hpp"))]
    srcs.append(os.path.join(ROOT, "include", "mpcb200.h"))
    if os.path.exists(_LIB) and all(os.path.getmtime(_LIB) >= os.path.getmtime(s) for s in srcs):
        return
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)


_lib = None


def use_native():
    """CPU-baseline legs of bench.py only: build the oracle with -march=native ON THIS MACHINE (BASELINE.md section 3) and bind that
    library instead of the portable one.  The library is built in a temporary directory, removed once it is loaded, so that the
    source tree stays untouched (it may be read-only).  Must be called before the first lib() call.  Falls back to the portable
    build if the compiler is unavailable."""
    global _lib
    assert _lib is None, "use_native() must come before the first oracle call"
    with tempfile.TemporaryDirectory(prefix="liboracle-") as tmp:
        so = os.path.join(tmp, "liboracle_native.so")
        try:
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "native", f"NATIVE_LIB={so}"], stdout=subprocess.DEVNULL,
                                  stderr=subprocess.DEVNULL)
            _bind(so)  # the loaded mapping outlives the file
            return True
        except (subprocess.CalledProcessError, OSError):
            return False


def _bind(path):
    global _lib
    _lib = C.CDLL(path)
    _lib.orc_check_jlog6.restype = C.c_double
    _lib.orc_check_jexp6.restype = C.c_double
    _lib.orc_check_centroidal.restype = C.c_double
    return _lib


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB)
        _lib.orc_check_jlog6.restype = C.c_double
        _lib.orc_check_jexp6.restype = C.c_double
        _lib.orc_check_centroidal.restype = C.c_double
    return _lib


def check_jlog6(M12):
    return lib().orc_check_jlog6(_p(np.ascontiguousarray(M12, float)))


def check_jexp6(xi):
    return lib().orc_check_jexp6(_p(np.ascontiguousarray(xi, float)))


def exp6(xi):
    out = np.zeros(12)
    lib().orc_exp6(_p(np.ascontiguousarray(xi, float)), _p(out))
    return out


def log6(M12):
    out = np.zeros(6)
    lib().orc_log6(_p(np.ascontiguousarray(M12, float)), _p(out))
    return out


def integrate(x, dx):
    out = np.zeros(57)
    lib().orc_integrate(_p(np.ascontiguousarray(x, float)), _p(np.ascontiguousarray(dx, float)), _p(out))
    return out


def difference(x0, x1):
    out = np.zeros(56)
    lib().orc_difference(_p(np.ascontiguousarray(x0, float)), _p(np.ascontiguousarray(x1, float)), _p(out))
    return out


def cone_matrix(mu, L, W):
    A = np.zeros((17, 6))
    lib().orc_cone_matrix(C.c_double(mu), C.c_double(L), C.c_double(W), _p(A))
    return A


def kinematics(rb, x):
    com, mass, hg = np.zeros(3), C.c_double(0), np.zeros(6)
    lf, rf, M, b = np.zeros(12), np.zeros(12), np.zeros((28, 28)), np.zeros(28)
    lib().orc_kinematics(C.byref(rb), _p(np.ascontiguousarray(x, float)), _p(com), C.byref(mass), _p(hg), _p(lf), _p(rf), _p(M), _p(b))
    return dict(com=com, mass=mass.value, hg=hg, lf=lf, rf=rf, M=M, b=b)


def rnea(rb, x, a):
    tau = np.zeros(28)
    lib().orc_rnea(C.byref(rb), _p(np.ascontiguousarray(x, float)), _p(np.ascontiguousarray(a, float)), _p(tau))
    return tau


def cdyn(rb, cfg, x, tau, active, check=True):
    o = dict(a=np.zeros(28), lam=np.zeros(12), da_dq=np.zeros((28, 28)), da_dv=np.zeros((28, 28)), da_dtau=np.zeros((28, 28)),
             dl_dq=np.zeros((12, 28)), dl_dv=np.zeros((12, 28)), dl_dtau=np.zeros((12, 28)), errs=np.zeros(6))
    act = (C.c_int * 2)(int(active[0]), int(active[1]))
    lib().orc_cdyn(C.byref(rb), C.byref(cfg), _p(np.ascontiguousarray(x, float)), _p(np.ascontiguousarray(tau, float)), act,
                   _p(o["a"]), _p(o["lam"]), _p(o["da_dq"]), _p(o["da_dv"]), _p(o["da_dtau"]), _p(o["dl_dq"]), _p(o["dl_dv"]),
                   _p(o["dl_dtau"]), _p(o["errs"]) if check else None)
    return o


def check_centroidal(rb, x):
    return lib().orc_check_centroidal(C.byref(rb), _p(np.ascontiguousarray(x, float)))


def eval_knot(rb, cfg, knot, x, u, xn, derivs=True, term=None):
    nx, n, m, nc = _abi.DIMS[cfg.kind]
    nz = n + m
    o = dict(xnext=np.zeros(nx), gap=np.zeros(n), A=np.zeros((n, n)), B=np.zeros((n, m)), E6=np.zeros((6, 6)), cost=C.c_double(0),
             lx=np.zeros(n), lu=np.zeros(m), H=np.zeros((nz, nz)), h=np.zeros(nc), Cx=np.zeros((nc, n)), Cu=np.zeros((nc, m)),
             ctype=np.zeros(nc, dtype=np.int32), lo=np.zeros(nc), hi=np.zeros(nc), xdot=np.zeros(56), lam=np.zeros(12))
    x = np.ascontiguousarray(x, float)
    u = np.ascontiguousarray(u, float) if u is not None else np.zeros(m)
    xn = np.ascontiguousarray(xn, float) if xn is not None else x
    lib().orc_eval_knot(C.byref(rb), C.byref(cfg), C.byref(knot) if knot is not None else None, C.byref(term) if term is not None else None,
                        _p(x), _p(u), _p(xn), int(derivs), _p(o["xnext"]), _p(o["gap"]), _p(o["A"]), _p(o["B"]), _p(o["E6"]),
                        C.byref(o["cost"]), _p(o["lx"]), _p(o["lu"]), _p(o["H"]), _p(o["h"]), _p(o["Cx"]), _p(o["Cu"]),
                        o["ctype"].ctypes.data_as(C.POINTER(C.c_int)), _p(o["lo"]), _p(o["hi"]), _p(o["xdot"]), _p(o["lam"]))
    o["cost"] = o["cost"].value
    return o


def riccati(n, m, nc, T, mu_d, mu, H, g, AB, f, CD, d, E6, HT, gT, CT=None, dT=None):
    nct = 0 if CT is None else CT.shape[0]
    s = m + nc
    o = dict(dxs=np.zeros((T + 1, n)), dus=np.zeros((T, m)), dvs=np.zeros((T + 1, nc)), dlams=np.zeros((T + 1, n)), K=np.zeros((T, s, 1 + n)))
    lib().orc_riccati(n, m, nc, T, C.c_double(mu_d), C.c_double(mu), _p(H), _p(g), _p(AB), _p(f), _p(CD), _p(d), _p(E6), _p(HT), _p(gT),
                      _p(CT), _p(dT), nct, _p(o["dxs"]), _p(o["dus"]), _p(o["dvs"]), _p(o["dlams"]), _p(o["K"]))
    return o


def riccati_par(n, m, nc, T, mu_d, mu, H, g, AB, f, CD, d, E6, HT, gT, CT=None, dT=None, legs=2):
    """The leg-parallel LQ solve (oracle/riccati_par.hpp) over `legs` legs; the same outputs as riccati."""
    nct = 0 if CT is None else CT.shape[0]
    s = m + nc
    o = dict(dxs=np.zeros((T + 1, n)), dus=np.zeros((T, m)), dvs=np.zeros((T + 1, nc)), dlams=np.zeros((T + 1, n)), K=np.zeros((T, s, 1 + n)))
    lib().orc_riccati_par(n, m, nc, T, C.c_double(mu_d), C.c_double(mu), _p(H), _p(g), _p(AB), _p(f), _p(CD), _p(d), _p(E6), _p(HT), _p(gT),
                          _p(CT), _p(dT), nct, int(legs), _p(o["dxs"]), _p(o["dus"]), _p(o["dvs"]), _p(o["dlams"]), _p(o["K"]))
    return o


def solve(prob, max_iters=None, inst_threads=1, knot_threads=1, vs=None, lams=None, xs=None, us=None):
    """Run the oracle ProxDDP on a problem dict from mpc_benchmark_b200.problems."""
    cfg = prob["cfg"]
    nx, n, m, nc = _abi.DIMS[cfg.kind]
    T = cfg.T
    batch = prob["x0"].shape[0]
    xs = np.ascontiguousarray(prob["xs"] if xs is None else xs, float).copy()
    us = np.ascontiguousarray(prob["us"] if us is None else us, float).copy()
    K = np.zeros((batch, T, m, n))
    vs = np.zeros((batch, T + 1, nc)) if vs is None else vs.copy()
    lams = np.zeros((batch, T + 1, n)) if lams is None else lams.copy()
    info = (_abi.Info * batch)()
    stage0 = np.zeros((batch, 68))
    lib().orc_solve(C.byref(prob["robot"]), C.byref(cfg), batch, prob["knots"], prob["terms"], _p(np.ascontiguousarray(prob["x0"], float)),
                    _p(xs), _p(us), _p(K), _p(vs), _p(lams), info, _p(stage0), int(cfg.max_iters if max_iters is None else max_iters),
                    int(inst_threads), int(knot_threads))
    return dict(xs=xs, us=us, K=K, vs=vs, lams=lams, info=info, stage0=stage0)


def ikid_terms(rb, x, frame_body, frame_place):
    """IKID task terms for the states x [count][57]: dict(Ag [count][6][28], dAgv [count][6], Jang [count][2][3][28], dJang [count][2][3],
    oMf [count][2][12]) of the frames (frame_body[f], frame_place[f])."""
    x = np.ascontiguousarray(x, float).reshape(-1, 57)
    B = x.shape[0]
    o = dict(Ag=np.zeros((B, 6, 28)), dAgv=np.zeros((B, 6)), Jang=np.zeros((B, 2, 3, 28)), dJang=np.zeros((B, 2, 3)), oMf=np.zeros((B, 2, 12)))
    fb, fp = np.ascontiguousarray(frame_body, np.int32), np.ascontiguousarray(frame_place, float).reshape(24)
    for i in range(B):
        lib().orc_ikid_terms(C.byref(rb), _p(x[i]), fb.ctypes.data_as(C.POINTER(C.c_int32)), _p(fp), *[_p(o[k][i]) for k in ("Ag", "dAgv", "Jang", "dJang", "oMf")])
    return o


# ---- dense QP oracle (oracle/qp.hpp; SURVEY 8f row f-3)
def qp_default_settings(**kw):
    s = _abi.QPSettings()
    lib().orc_qp_default_settings(C.byref(s))
    for k, v in kw.items():
        assert hasattr(s, k), k
        setattr(s, k, v)
    return s


def _bs(a, per):
    """(contiguous array, batch stride in doubles): arrays without the leading batch axis are shared (stride 0)."""
    a = np.ascontiguousarray(a, float)
    return a, (0 if a.size == per else per)


def qp_marshal(H, g, A, b, Cm, l, u, lb=None, ub=None, x=None, y=None, z=None):
    """Shapes, (pointer, stride) argument list and output arrays shared by the oracle and the emulation bindings."""
    g = np.ascontiguousarray(g, float)
    n = g.shape[-1]
    ne, ni = np.asarray(b).shape[-1], np.asarray(l).shape[-1]
    box = lb is not None
    nz = ni + (n if box else 0)
    keep, args, batch = [], [], 1
    for arr, per in ((H, n * n), (g, n), (A, ne * n), (b, ne), (Cm, ni * n), (l, ni), (u, ni), (lb if box else np.zeros(n), n), (ub if box else np.zeros(n), n)):
        a, s = _bs(arr, per)
        if s:
            batch = max(batch, a.size // per)
        keep.append(a)
        args += [_p(a) if a.size else None, C.c_long(s)]
    X = np.zeros((batch, n)) if x is None else np.ascontiguousarray(x, float).reshape(batch, n).copy()
    Y = np.zeros((batch, ne)) if y is None else np.ascontiguousarray(y, float).reshape(batch, ne).copy()
    Z = np.zeros((batch, nz)) if z is None else np.ascontiguousarray(z, float).reshape(batch, nz).copy()
    return (n, ne, ni, int(box), batch), args, keep, (X, Y, Z), (_abi.QPInfo * batch)()


def qp_solve(H, g, A, b, Cm, l, u, lb=None, ub=None, settings=None, x=None, y=None, z=None, threads=0):
    """Batch of QPs through the CPU oracle.  Leading axis = batch; arrays without it are shared between the QPs."""
    dims, args, keep, (X, Y, Z), info = qp_marshal(H, g, A, b, Cm, l, u, lb, ub, x, y, z)
    st = settings or qp_default_settings()
    lib().orc_qp_solve(*dims, C.byref(st), *args, _p(X), _p(Y), _p(Z), info, threads)
    return X, Y, Z, info


def qp_assemble_id(M, nle, Jc, gamma, a, forces, cs, mu, L, W):
    batch = np.asarray(M).reshape(-1, 28, 28).shape[0]
    A, b, Cm, l = np.zeros((batch, 40, 62)), np.zeros((batch, 40)), np.zeros((batch, 18, 62)), np.zeros((batch, 18))
    cs = np.ascontiguousarray(cs, np.int32)
    f = lambda v: _p(np.ascontiguousarray(v, float))
    lib().orc_qp_assemble_id(batch, f(M), f(nle), f(Jc), f(gamma), f(a), f(forces), cs.ctypes.data_as(C.POINTER(C.c_int32)), C.c_double(mu),
                             C.c_double(L), C.c_double(W), _p(A), _p(b), _p(Cm), _p(l))
    return A, b, Cm, l
