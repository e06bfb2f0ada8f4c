"""ctypes binding of tests/_emu/libemu_models.so (tests/emu/emu_models.cpp): the kernel sources compiled for the host with serial PAR_FOR
loops, run with one model per instance (mpc_set_instance_models).  TEST-ONLY, like emu_lib; never loaded by the product."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

from emu_lib import _p
from mpc_benchmark_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(ROOT, "tests", "emu", "emu_models.cpp")
_LIB = os.path.join(ROOT, "tests", "_emu", "libemu_models.so")
# the flags of tests/emu/Makefile
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-Wall", "-Wno-unused-variable", "-Wno-unused-but-set-variable", "-Wno-unknown-pragmas",
          "-Wno-aggressive-loop-optimizations", "-Wno-array-bounds"]
_lib = None


class EmuError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        deps = [_SRC, os.path.join(ROOT, "tests", "emu", "emu.cpp")] + glob.glob(os.path.join(ROOT, "mpc_benchmark_b200", "csrc", "*.[ch]*")) \
            + glob.glob(os.path.join(ROOT, "include", "*.h"))
        if not os.path.exists(_LIB) or any(os.path.getmtime(d) > os.path.getmtime(_LIB) for d in deps):
            os.makedirs(os.path.dirname(_LIB), exist_ok=True)
            tmp = f"{_LIB}.{os.getpid()}.tmp"
            subprocess.check_call(["g++", *_FLAGS, "-o", tmp, _SRC])
            os.replace(tmp, _LIB)
        _lib = C.CDLL(_LIB)
        _lib.emu_models_last_error.restype = C.c_char_p
    return _lib


def solve_models(prob, robots, cfgs, max_iters, xs=None, us=None, vs=None, lams=None):
    """emu_lib.solve with per-instance models: robots / cfgs are sequences of length batch of _abi.Robot / _abi.Config, or None for prob's
    shared robot / config.  A rejected model raises EmuError with the message of the validation (build_instance_models)."""
    cfg = prob["cfg"]
    nx, n, m, nc = _abi.DIMS[cfg.kind]
    T, B = cfg.T, prob["x0"].shape[0]
    for seq in (robots, cfgs):
        if seq is not None and len(seq) != B:
            raise EmuError(f"expected {B} per-instance models, got {len(seq)}")
    xs = np.ascontiguousarray(prob["xs"] if xs is None else xs, float).copy()
    us = np.ascontiguousarray(prob["us"] if us is None else us, float).copy()
    K = np.zeros((B, T, m, n))
    vs = np.zeros((B, T + 1, nc)) if vs is None else vs.copy()
    lams = np.zeros((B, T + 1, n)) if lams is None else lams.copy()
    info = (_abi.Info * B)()
    rbs = None if robots is None else (_abi.Robot * B)(*robots)
    cfs = None if cfgs is None else (_abi.Config * B)(*cfgs)
    rc = lib().emu_solve_models(C.byref(prob["robot"]), C.byref(cfg), rbs, cfs, B, prob["knots"], prob["terms"],
                                _p(np.ascontiguousarray(prob["x0"], float)), _p(xs), _p(us), _p(K), _p(vs), _p(lams), info, int(max_iters))
    if rc != 0:
        raise EmuError(lib().emu_models_last_error().decode())
    return dict(xs=xs, us=us, K=K, vs=vs, lams=lams, info=info)
