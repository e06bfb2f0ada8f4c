import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpc_benchmark_b200 import problems
from mpc_benchmark_b200.batch import BatchSolver
prob = problems.full_walk_batch(1, seed=5)
s = BatchSolver(prob["robot"], prob["cfg"], 1)
s.setup(prob["knots"], prob["terms"], prob["x0_nominal"])
w = s.run(prob["xs"], prob["us"], max_iters=20, gains=False)
s.set_x0(prob["x0"])
xs = problems.warm_tick_inputs(prob, w.xs); us = w.us.copy()
for i in range(5):
    s.reset_multipliers(); t0=time.perf_counter(); r = s.run(xs, us, max_iters=1, gains=False); dt=time.perf_counter()-t0
print("tick ms", 1e3*dt, "launches", s.last_launches, "device ms", s.last_device_ms, s.kernel_ms(), "ls", r.ls_evals)
