"""ctypes bindings of the IKID test libraries built from tests/ikid/ (tests/_emu/libikid_{oracle,emu}.so): the oracle's IKID task
terms on its own rigid-body code, and the IKID kernel SOURCES (csrc/rbd_terms.cuh, csrc/qp.cuh) run serially on the host.
TEST-ONLY: never loaded by the product."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
dp = C.POINTER(C.c_double)
i32p = C.POINTER(C.c_int32)
_libs = {}


def _lib(name):
    if name not in _libs:
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "ikid")], stdout=subprocess.DEVNULL)
        _libs[name] = C.CDLL(os.path.join(ROOT, "tests", "_emu", f"lib{name}.so"))
    return _libs[name]


def _p(a):
    return a.ctypes.data_as(dp) if a is not None else None


def _frames(frame_body, frame_place):
    return np.ascontiguousarray(frame_body, np.int32), np.ascontiguousarray(frame_place, float).reshape(24)


def oracle_ikid_terms(rb, x, frame_body, frame_place):
    """The oracle's task terms for the states x [count][57]: dict(Ag [count][6][28], dAgv [count][6], Jang [count][2][3][28],
    dJang [count][2][3], oMf [count][2][12]) of the frames (frame_body[f], frame_place[f])."""
    x = np.ascontiguousarray(x, float).reshape(-1, 57)
    B = x.shape[0]
    o = dict(Ag=np.zeros((B, 6, 28)), dAgv=np.zeros((B, 6)), Jang=np.zeros((B, 2, 3, 28)), dJang=np.zeros((B, 2, 3)), oMf=np.zeros((B, 2, 12)))
    fb, fp = _frames(frame_body, frame_place)
    for i in range(B):
        _lib("ikid_oracle").orc_ikid_terms(C.byref(rb), _p(x[i]), fb.ctypes.data_as(i32p), _p(fp), *[_p(o[k][i]) for k in ("Ag", "dAgv", "Jang", "dJang", "oMf")])
    return o


def emu_ikid_terms(rb, cfg, x, frame_body, frame_place):
    """ikid_terms_group run serially: dict(M, nle, Jc, dJv, Ag, dAgv, Jang [count][2][3][28], dJang [count][2][3])."""
    x = np.ascontiguousarray(x, float).reshape(-1, 57)
    B = x.shape[0]
    o = dict(M=np.zeros((B, 28, 28)), nle=np.zeros((B, 28)), Jc=np.zeros((B, 12, 28)), dJv=np.zeros((B, 12)), Ag=np.zeros((B, 6, 28)), dAgv=np.zeros((B, 6)),
             Jang=np.zeros((B, 2, 3, 28)), dJang=np.zeros((B, 2, 3)))
    fb, fp = _frames(frame_body, frame_place)
    rc = _lib("ikid_emu").emu_ikid_terms(C.byref(rb), C.byref(cfg), B, _p(x), fb.ctypes.data_as(i32p), _p(fp),
                                         *[_p(o[k]) for k in ("M", "nle", "Jc", "dJv", "Ag", "dAgv", "Jang", "dJang")])
    assert rc == 0
    return o


def emu_qp_assemble_ikid(M, nle, Jc, dJv, Ag, dAgv, Jang, dJang, task, forces, cs, weights, gains, mu, L, W):
    """qp_assemble_ikid_group run serially: (H, g, A, b, C, l) of the IKID QPs; gains packed [1658]."""
    batch = np.asarray(M).reshape(-1, 28, 28).shape[0]
    H, g = np.zeros((batch, 62, 62)), np.zeros((batch, 62))
    A, b, Cm, l = np.zeros((batch, 40, 62)), np.zeros((batch, 40)), np.zeros((batch, 18, 62)), np.zeros((batch, 18))
    cs = np.ascontiguousarray(cs, np.int32)
    f = lambda v: _p(np.ascontiguousarray(v, float))  # noqa: E731
    _lib("ikid_emu").emu_qp_assemble_ikid(batch, f(M), f(nle), f(Jc), f(dJv), f(Ag), f(dAgv), f(Jang), f(dJang), f(task), f(forces), cs.ctypes.data_as(i32p),
                                          f(weights), f(gains), C.c_double(mu), C.c_double(L), C.c_double(W), _p(H), _p(g), _p(A), _p(b), _p(Cm), _p(l))
    return H, g, A, b, Cm, l
