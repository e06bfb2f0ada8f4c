#!/usr/bin/env python
"""A population of robots with randomised link masses and torso payloads walking the REFERENCE gait in one batch, every tick on the GPU:
per-instance robot models (mpc_set_instance_models), the device gait with each robot's soles from its own kinematics (mpc_gait_tick),
the warm-start shift and one ProxDDP iteration (mpc_tick), ideal plant (x_meas = the model prediction).

    python examples/population_walk.py [kino|full] [robots] [ticks] [mass spread] [payload kg]

Robot i has every body's mass and rotational inertia scaled by a factor uniform in [1 - spread, 1 + spread], its CoMs shifted by 1 cm
(standard deviation) and a payload uniform in [0, payload] kg on the torso (problems.perturbed_robots); the kinematics are nominal.  The
gait stays uniform: every robot keeps the nominal contact-force references (m g / 2 of the nominal mass), which a heavier robot has to
correct through its own dynamics.  Prints, per robot, the total mass, ticks with a failed solve (status >= 2), ticks that ended
without an accepted step (num_iters 0: the solve stopped in its outer-loop checks), the smallest and median step length alpha over the ticks that took a
step, and how far the base advanced."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpc_benchmark_b200 import _abi, gait, problems  # noqa: E402
from mpc_benchmark_b200.batch import BatchSolver  # noqa: E402

model = sys.argv[1] if len(sys.argv) > 1 else "kino"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 32
kind = {"kino": _abi.KIND_KINO, "full": _abi.KIND_FULL}[model]
N = int(sys.argv[3]) if len(sys.argv) > 3 else (840 if kind == _abi.KIND_KINO else 1000)  # the whole reference gait
SPREAD = float(sys.argv[4]) if len(sys.argv) > 4 else 0.1
PAYLOAD = float(sys.argv[5]) if len(sys.argv) > 5 else 5.0

prob = {_abi.KIND_KINO: problems.kino_standing_problem, _abi.KIND_FULL: problems.full_standing_problem}[kind](batch=B, mu_init=1e-8)
robots = problems.perturbed_robots(prob["robot"], B, seed=0, mass=SPREAD, com=0.01, payload=PAYLOAD)
mirror = (np.arange(B) % 2).astype(bool)
s = BatchSolver(prob["robot"], prob["cfg"], B)
s.set_instance_models(robots)
s.setup(prob["knots"], prob["terms"], prob["x0"])
t0 = time.time()
cold = s.run(prob["xs"], prob["us"], max_iters=100, gains=False)
print(f"{model}: {B} robots, {N} ticks, mass spread {SPREAD}, payload up to {PAYLOAD} kg")
print(f"cold solve: {time.time() - t0:.2f} s, iterations {int(cold.num_iters.min())}..{int(cold.num_iters.max())}")
urefs = gait.force_ramp_refs(kind, prob["mass"], 34, prob["cfg"].T) if kind == _abi.KIND_KINO else None
s.set_tail_warmstart(True)  # the appended knot's control from the nearest knot of the same contact phase (DESIGN section 7)
s.gait_setup(gait.device_gait(kind, prob["lf"], prob["rf"], prob["com0"], prob["mass"]), mirror, urefs)
x_start = cold.xs[:, 0, 0].copy()
fails, nostep, alphas = np.zeros(B, int), np.zeros(B, int), []
t0 = time.time()
for t in range(N):
    s.gait_tick()
    s.tick(None, None, keep_multipliers=False, max_iters=1)
    r = s.results(gains=False, multipliers=False)
    st = np.array([i.status for i in r.info])
    stepped = r.num_iters >= 1
    fails += st >= 2
    nostep += ~stepped & (st < 2)
    alphas.append(np.where(stepped, r.alpha, np.nan))
dt = time.time() - t0
alphas = np.array(alphas)
amin, amed = np.nanmin(alphas, axis=0), np.nanmedian(alphas, axis=0)
adv = r.xs[:, 0, 0] - x_start
print(f"{N} ticks x {B} robots in {dt:.1f} s (results read back every tick)")
print(" robot  mass kg  failed ticks  no-step ticks  alpha min  alpha median  base advanced m")
for i in range(B):
    print(f"{i:6d}  {sum(robots[i].mass):7.2f}  {fails[i]:12d}  {nostep[i]:13d}  {amin[i]:9.3f}  {amed[i]:12.3f}  {adv[i]:+15.3f}")
print(f"robots with a failed tick: {int((fails > 0).sum())} of {B}; no-step ticks {int(nostep.sum())} of {B * N}; base advanced {adv.min():+.3f}..{adv.max():+.3f} m; "
      f"alpha min over the ticks with a step {np.nanmin(amin):.3f}")
s.close()
