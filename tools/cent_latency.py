"""Warm single-instance centroidal MPC tick latency and its per-category kernel time (GPU box).  usage: python tools/cent_latency.py"""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpc_benchmark_b200 import problems  # noqa: E402
from mpc_benchmark_b200.batch import BatchSolver  # noqa: E402

prob = problems.cent_standing_problem(batch=1, T=100)
s = BatchSolver(prob["robot"], prob["cfg"], 1, device=0)
s.setup(prob["knots"], prob["terms"], prob["x0"])
warm = s.run(prob["xs"], prob["us"], max_iters=20, gains=False)
ts = []
for _ in range(60):
    t0 = time.perf_counter()
    s.reset_multipliers()
    s.run(warm.xs, warm.us, max_iters=1, gains=False)
    ts.append(1e3 * (time.perf_counter() - t0))
print("p50 ms", float(np.percentile(ts[5:], 50)), "kernel ms", s.kernel_ms(), "launches", s.last_launches)
