"""ctypes binding of tests/_emu/libemu.so: the CUDA kernel SOURCES (mpc_benchmark_b200/csrc/*.cuh) compiled for the host
with serial PAR_FOR loops.  TEST-ONLY: checks kernel logic on machines without a GPU; never loaded by the product."""
import ctypes as C
import os
import subprocess

import numpy as np

from mpc_benchmark_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = os.path.join(ROOT, "tests", "_emu", "libemu.so")
dp = C.POINTER(C.c_double)
_lib = None


class EmuError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "emu")], stdout=subprocess.DEVNULL)
        _lib = C.CDLL(_LIB)
        _lib.emu_last_error.restype = C.c_char_p
    return _lib


def _p(a):
    return a.ctypes.data_as(dp) if a is not None else None


def solve(prob, max_iters, dump=False, xs=None, us=None, vs=None, lams=None, robots=None, cfgs=None):
    """robots / cfgs: sequences of length batch of _abi.Robot / _abi.Config giving every instance its own model (mpc_set_instance_models),
    or None for prob's shared robot / config.  A rejected model raises EmuError with the message of the C validation."""
    cfg = prob["cfg"]
    nx, n, m, nc = _abi.DIMS[cfg.kind]
    T, B, nz = cfg.T, prob["x0"].shape[0], n + m
    for seq in (robots, cfgs):
        if seq is not None and len(seq) != B:
            raise EmuError(f"expected {B} per-instance models, got {len(seq)}")
    xs = np.ascontiguousarray(prob["xs"] if xs is None else xs, float).copy()
    us = np.ascontiguousarray(prob["us"] if us is None else us, float).copy()
    K = np.zeros((B, T, m, n))
    vs = np.zeros((B, T + 1, nc)) if vs is None else vs.copy()
    lams = np.zeros((B, T + 1, n)) if lams is None else lams.copy()
    info = (_abi.Info * B)()
    st = np.zeros((B, 68))
    d = np.zeros(T * n * nz + (T + 1) * nz * nz + (T + 1) * nz + T * n + (T + 1) * nc + (T + 1) * 8) if dump else None
    rbs = None if robots is None else (_abi.Robot * B)(*robots)
    cfs = None if cfgs is None else (_abi.Config * B)(*cfgs)
    rc = lib().emu_solve(C.byref(prob["robot"]), C.byref(cfg), rbs, cfs, B, prob["knots"], prob["terms"], _p(np.ascontiguousarray(prob["x0"], float)),
                         _p(xs), _p(us), _p(K), _p(vs), _p(lams), info, _p(st), int(max_iters), _p(d))
    if rc != 0:
        raise EmuError(lib().emu_last_error().decode())
    out = dict(xs=xs, us=us, K=K, vs=vs, lams=lams, info=info, stage0=st)
    if dump:
        o = 0

        def take(sh):
            nonlocal o
            s = int(np.prod(sh))
            a = d[o:o + s].reshape(sh)
            o += s
            return a

        out.update(AB=take((T, n, nz)), H=take((T + 1, nz, nz)), g=take((T + 1, nz)), gap=take((T, n)), h=take((T + 1, nc)), scal=take((T + 1, 8)))
    return out


def qp_solve(H, g, A, b, Cm, l, u, lb=None, ub=None, settings=None, x=None, y=None, z=None):
    """The kernel source of the batched QP solver (csrc/qp.cuh) run serially on the host."""
    import oracle_lib

    dims, args, keep, (X, Y, Z), info = oracle_lib.qp_marshal(H, g, A, b, Cm, l, u, lb, ub, x, y, z)
    st = settings or oracle_lib.qp_default_settings()
    lib().emu_qp_solve(*dims, C.byref(st), *args, _p(X), _p(Y), _p(Z), info)
    return X, Y, Z, info


def qp_assemble_id(M, nle, Jc, gamma, a, forces, cs, mu, L, W):
    batch = np.asarray(M).reshape(-1, 28, 28).shape[0]
    A, b, Cm, l = np.zeros((batch, 40, 62)), np.zeros((batch, 40)), np.zeros((batch, 18, 62)), np.zeros((batch, 18))
    cs = np.ascontiguousarray(cs, np.int32)
    f = lambda v: _p(np.ascontiguousarray(v, float))
    lib().emu_qp_assemble_id(batch, f(M), f(nle), f(Jc), f(gamma), f(a), f(forces), cs.ctypes.data_as(C.POINTER(C.c_int32)), C.c_double(mu),
                             C.c_double(L), C.c_double(W), _p(A), _p(b), _p(Cm), _p(l))
    return A, b, Cm, l


def rbd_terms(rb, cfg, x):
    """csrc/rbd_terms.cuh run serially on the host: dict(M, nle, Jc, dJv, vf) for the states x [count][57]."""
    x = np.ascontiguousarray(x, float).reshape(-1, 57)
    B = x.shape[0]
    o = dict(M=np.zeros((B, 28, 28)), nle=np.zeros((B, 28)), Jc=np.zeros((B, 12, 28)), dJv=np.zeros((B, 12)), vf=np.zeros((B, 2, 6)))
    rc = lib().emu_rbd_terms(C.byref(rb), C.byref(cfg), B, _p(x), *[_p(o[k]) for k in ("M", "nle", "Jc", "dJv", "vf")])
    assert rc == 0
    return o


def ikid_terms(rb, cfg, x, frame_body, frame_place):
    """ikid_terms_group (csrc/rbd_terms.cuh) run serially: dict(M, nle, Jc, dJv, Ag, dAgv, Jang [count][2][3][28], dJang [count][2][3])
    for the states x [count][57] and the frames (frame_body[f], frame_place[f])."""
    x = np.ascontiguousarray(x, float).reshape(-1, 57)
    B = x.shape[0]
    o = dict(M=np.zeros((B, 28, 28)), nle=np.zeros((B, 28)), Jc=np.zeros((B, 12, 28)), dJv=np.zeros((B, 12)), Ag=np.zeros((B, 6, 28)), dAgv=np.zeros((B, 6)),
             Jang=np.zeros((B, 2, 3, 28)), dJang=np.zeros((B, 2, 3)))
    fb, fp = np.ascontiguousarray(frame_body, np.int32), np.ascontiguousarray(frame_place, float).reshape(24)
    rc = lib().emu_ikid_terms(C.byref(rb), C.byref(cfg), B, _p(x), fb.ctypes.data_as(C.POINTER(C.c_int32)), _p(fp),
                              *[_p(o[k]) for k in ("M", "nle", "Jc", "dJv", "Ag", "dAgv", "Jang", "dJang")])
    assert rc == 0
    return o


def qp_assemble_ikid(M, nle, Jc, dJv, Ag, dAgv, Jang, dJang, task, forces, cs, weights, gains, mu, L, W):
    """qp_assemble_ikid_group (csrc/qp.cuh) run serially: (H, g, A, b, C, l) of the IKID QPs; gains packed [1658]."""
    batch = np.asarray(M).reshape(-1, 28, 28).shape[0]
    H, g = np.zeros((batch, 62, 62)), np.zeros((batch, 62))
    A, b, Cm, l = np.zeros((batch, 40, 62)), np.zeros((batch, 40)), np.zeros((batch, 18, 62)), np.zeros((batch, 18))
    cs = np.ascontiguousarray(cs, np.int32)
    f = lambda v: _p(np.ascontiguousarray(v, float))  # noqa: E731
    lib().emu_qp_assemble_ikid(batch, f(M), f(nle), f(Jc), f(dJv), f(Ag), f(dAgv), f(Jang), f(dJang), f(task), f(forces), cs.ctypes.data_as(C.POINTER(C.c_int32)),
                               f(weights), f(gains), C.c_double(mu), C.c_double(L), C.c_double(W), _p(H), _p(g), _p(A), _p(b), _p(Cm), _p(l))
    return H, g, A, b, Cm, l


def gait(kind, T, g, mirror, urefs, lf, rf):
    """csrc/gait.cuh run serially: lf / rf [ticks][batch][12] -> (knots [ticks][batch * T], terms [ticks][batch])."""
    lf, rf = np.ascontiguousarray(lf, float), np.ascontiguousarray(rf, float)
    ticks, batch = lf.shape[0], lf.shape[1]
    mir = np.ascontiguousarray(mirror, dtype=np.int32)
    ur = None
    if urefs is not None:
        ur = np.zeros((len(urefs), _abi.MAXU))
        ur[:, :np.asarray(urefs).shape[1]] = urefs
        g.n_uref = len(urefs)
    ks, ts = (_abi.Knot * (ticks * batch * T))(), (_abi.Term * (ticks * batch))()
    rc = lib().emu_gait(int(kind), int(T), C.byref(g), batch, mir.ctypes.data_as(C.POINTER(C.c_int32)), _p(ur), ticks, _p(lf), _p(rf), ks, ts)
    assert rc == 0
    return ks, ts
