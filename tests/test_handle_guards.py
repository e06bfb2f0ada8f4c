"""A NULL handle is an error like any other (INTEGRATION 2): every entry point of include/mpcb200.h and include/mpcqp_b200.h that
takes a handle returns a non-zero status, or the out-of-range value of a getter, with a message that names it.  No GPU needed.
Each call runs in its own interpreter, so a library that dereferences the handle fails one test instead of ending the session."""
import os
import re
import subprocess
import sys

import pytest

from mpc_benchmark_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# entry points that cannot return a status: the value a getter gives for a NULL handle, or None for a void function
NO_STATUS = {"mpc_last_launches": -1, "mpc_last_kernel_launches": -1, "mpc_last_kernel_ms": -1.0, "mpc_last_device_ms": -1.0,
             "mpc_qp_last_device_ms": -1.0, "mpc_workspace_bytes": 0, "mpc_set_profiling": None}
DESTROY = {"mpc_destroy", "mpc_qp_destroy"}  # free()-like: NULL is a no-op

# calls `name` with a NULL handle and zero / NULL for every other argument (argument types as bound in _native.py)
CALL = """
import ctypes as C, sys
sys.path.insert(0, sys.argv[1])
from mpc_benchmark_b200 import _native
L = _native.lib()
name = sys.argv[2]
f = getattr(L, name)
args = [0.0 if t is C.c_double else None if t is C.c_void_p or issubclass(t, C._Pointer) else 0 for t in f.argtypes]
r = f(*args)
err = (L.mpc_qp_last_error() if name.startswith("mpc_qp_") else L.mpc_last_error()).decode()
print(repr(r))
print(err)
"""


def _handle_entry_points():
    names = []
    for hdr in ("mpcb200.h", "mpcqp_b200.h"):
        src = open(os.path.join(ROOT, "include", hdr)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names += re.findall(r"\b(mpc_[a-z0-9_]+)\s*\(\s*(?:mpc_solver_t|mpc_qp_t)\s*\*", src)
    return sorted(names)


def test_every_handle_entry_point_is_covered():
    names = _handle_entry_points()
    assert len(names) >= 40
    assert set(NO_STATUS) | DESTROY <= set(names)


@pytest.mark.parametrize("name", _handle_entry_points())
def test_null_handle_is_an_error(name):
    if not os.path.exists(_native.LIB_PATH):
        pytest.skip("libmpcb200.so not built (run __graft_entry__.build())")
    p = subprocess.run([sys.executable, "-c", CALL, ROOT, name], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, f"{name}(NULL, ...) ended the process with code {p.returncode}: {p.stderr[-500:]}"
    ret, err = (p.stdout.split("\n") + [""])[:2]
    if name in DESTROY:
        return
    if name not in NO_STATUS:
        assert int(ret) != 0
    elif NO_STATUS[name] is not None:
        assert ret == repr(NO_STATUS[name])
    assert err == f"{name}: null handle"
