"""Runs the TOP HALF of a reference script (`*_talos.py` of a checkout of edantec/MPC_benchmark, passed as `ref_dir` — never
copied into the repo) with `aligator` / `pinocchio` replaced by this package ("switch backends with one import", SURVEY 8b)
and the plant / robot-data / spline packages stubbed (bullet_robot, example_robot_data, ndcurves, proxsuite).

The script source is executed up to (excluding) the line `solver.max_iters = 1`, i.e. model construction + setup + cold
solve (fulldynamic_talos.py:1-405).  `capture=True` replaces SolverProxDDP.setup/run by recorders so the flattening can
be checked on a machine without GPU.  tests/golden/make_golden.py stores what it captures as tests/golden/ref_flat_*.npz.
"""
import os
import sys
import types

import numpy as np


class _Stop(Exception):
    pass


def _stub_modules():
    import mpc_benchmark_b200 as pkg
    from mpc_benchmark_b200 import pin

    mods = {}
    mods["aligator"] = pkg
    mods["aligator.manifolds"], mods["aligator.dynamics"], mods["aligator.constraints"] = pkg.manifolds, pkg.dynamics, pkg.constraints
    mods["pinocchio"] = pin

    bullet = types.ModuleType("bullet_robot")

    class BulletRobot:
        def __init__(self, *a, **k):
            pass

        def initializeJoints(self, q):
            self.q = np.array(q, float)

        def changeCamera(self, *a):
            pass

        def measureState(self):
            return self.q.copy(), np.zeros(pin.Model().nv)

        def showTargetToTrack(self, *a):
            pass

    bullet.BulletRobot = BulletRobot
    mods["bullet_robot"] = bullet

    erd = types.ModuleType("example_robot_data")

    class _Wrapper:
        def __init__(self):
            self.model = pin.Model()

        def buildReducedRobot(self, locked, q):
            return _Wrapper()

    erd.load = lambda name: _Wrapper()
    erd.getModelPath = lambda sub: ""
    mods["example_robot_data"] = erd
    mods["ndcurves"] = types.ModuleType("ndcurves")
    mods["proxsuite"] = types.ModuleType("proxsuite")
    mods["pybullet"] = types.ModuleType("pybullet")
    mods["pybullet_data"] = types.ModuleType("pybullet_data")
    return mods


def run_top_half(script, ref_dir, capture=True):
    """Returns (namespace, captured) where captured = list of ('setup'|'run', FlatProblem, xs, us)."""
    import mpc_benchmark_b200 as pkg
    from mpc_benchmark_b200 import flatten

    src = open(os.path.join(ref_dir, script)).read()
    cut = src.index("solver.max_iters = 1")
    src = src[:cut]
    saved = {k: sys.modules.get(k) for k in list(_stub_modules())}
    saved_path = list(sys.path)
    captured = []
    orig_setup, orig_run = pkg.SolverProxDDP.setup, pkg.SolverProxDDP.run
    try:
        sys.modules.update(_stub_modules())
        for m in ("talos_utils", "QP_utils"):
            sys.modules.pop(m, None)
        sys.path.insert(0, ref_dir)
        if capture:
            def fake_setup(self, problem):
                self._check_options()
                captured.append(("setup", flatten.flatten_problem(problem, self.target_tol, self.mu_init, self.max_iters), None, None))

            def fake_run(self, problem, xs_init=(), us_init=(), *a):
                self._check_options()
                flat = flatten.flatten_problem(problem, self.target_tol, self.mu_init, self.max_iters)
                captured.append(("run", flat, np.array(xs_init, float), np.array(us_init, float)))
                raise _Stop()

            pkg.SolverProxDDP.setup, pkg.SolverProxDDP.run = fake_setup, fake_run
        ns = {"__name__": "__ref_script__"}
        try:
            exec(compile(src, os.path.join(ref_dir, script), "exec"), ns)
        except _Stop:
            pass
        return ns, captured
    finally:
        pkg.SolverProxDDP.setup, pkg.SolverProxDDP.run = orig_setup, orig_run
        sys.path[:] = saved_path
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        for m in ("talos_utils", "QP_utils"):
            sys.modules.pop(m, None)
