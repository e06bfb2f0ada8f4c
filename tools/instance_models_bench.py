"""Cost of per-instance models (mpc_set_instance_models) on the bench workload: the full-dynamics reference-gait batch of bench.py
(problems.walk_batch, seed 5, T = 100) at batch 4096, one-iteration ticks (reset_multipliers + run_device(max_iters = 1), the timed
tick of bench.py) from the warm start of a 20-iteration cold solve, in three cases on ONE handle, alternated round by round:
  (a) shared   - the handle's one model, read by every instance (Ws::model_stride 0);
  (b) copies   - per-instance models, every one a copy of the shared model (the same arithmetic, 4096 x 21 KB of model reads);
  (c) random   - per-instance models with randomised masses / inertias / CoMs and a torso payload (problems.perturbed_robots).
Every tick starts from the same warm start, so each case's tick is the same computation every time.  Reports the tick's device time
(CUDA events on the launch stream; p50 / mean per case), the per-category kernel time of mpc_last_kernel_ms (eval_deriv, riccati,
eval_trial, bookkeeping), checks that (a) and (b) are bitwise equal (xs, us, K0, vs, lams, info), and reads the GPU name and power limit
in the same run.

    python tools/instance_models_bench.py [--out profiles/instance_models_b200.json] [--batch 4096] [--rounds 4] [--steps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mpc_benchmark_b200 import _abi, problems  # noqa: E402
from mpc_benchmark_b200.batch import BatchSolver  # noqa: E402

CATS = ("eval_deriv", "riccati", "eval_trial", "bookkeeping")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clk)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "instance_models_b200.json"))
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=5, help="timed ticks per case and round (after one untimed tick)")
    args = ap.parse_args()
    import torch

    B = args.batch
    t0 = time.time()
    ticks = np.random.default_rng(5).integers(0, 100, size=B)
    prob = problems.walk_batch(_abi.KIND_FULL, B, seed=5, T=100, ticks=ticks)
    cases = {"shared": None, "copies": ([prob["robot"]] * B, None),
             "random": (problems.perturbed_robots(prob["robot"], B, seed=1, mass=0.1, com=0.01, payload=5.0), None)}
    s = BatchSolver(prob["robot"], prob["cfg"], B)
    s.setup(prob["knots"], prob["terms"], prob["x0_nominal"])
    prep = s.run(prob["xs"], prob["us"], max_iters=20, gains=False)
    xs_d = torch.from_numpy(problems.warm_tick_inputs(prob, prep.xs)).cuda()
    us_d = torch.from_numpy(prep.us).cuda()
    s.set_x0(prob["x0"])
    torch.cuda.synchronize()
    print(f"setup {time.time() - t0:.1f} s", flush=True)

    def tick():
        s.reset_multipliers()
        s.run_device(xs_d.data_ptr(), us_d.data_ptr(), max_iters=1)

    def snapshot():
        r = s.results(gains=False)
        return dict(xs=r.xs, us=r.us, K0=s.feedback(0), vs=r.vs, lams=r.lams, info=b"".join(bytes(i) for i in r.info))

    ms = {c: [] for c in cases}
    cat_ms = {c: {k: [] for k in CATS} for c in cases}
    snaps = {}
    for rnd in range(args.rounds):
        for name, models in cases.items():
            s.set_instance_models(*(models or (None, None)))
            tick()  # untimed
            for _ in range(args.steps):
                tick()
                ms[name].append(s.last_device_ms)
                for k, (v, _n) in s.kernel_ms().items():
                    cat_ms[name][k].append(v)
            if rnd == 0:
                snaps[name] = snapshot()
        print(f"round {rnd}: " + ", ".join(f"{c} {np.median(ms[c][-args.steps:]):.2f} ms" for c in cases), flush=True)
    s.set_instance_models(None, None)
    a, b, c = snaps["shared"], snaps["copies"], snaps["random"]
    bitwise = {k: bool(np.array_equal(a[k], b[k])) if k != "info" else a[k] == b[k] for k in a}
    differs = {k: float(np.abs(c[k] - a[k]).max()) for k in ("xs", "us", "K0")}
    res = dict(
        gpu=gpu_info(),
        what=("full-dynamics reference-gait batch of bench.py (walk_batch seed 5, T = 100), one-iteration ticks (reset_multipliers + run_device(max_iters=1)) "
              "from one warm start; device time per tick (CUDA events around the run) and per kernel category (mpc_last_kernel_ms); the three cases "
              "alternate on one handle, round by round"),
        batch=B, rounds=args.rounds, steps_per_round=args.steps,
        cases={n: dict(tick_ms_p50=float(np.median(ms[n])), tick_ms_mean=float(np.mean(ms[n])), tick_ms_min=float(np.min(ms[n])), tick_ms_max=float(np.max(ms[n])),
                       kernel_ms_p50={k: float(np.median(cat_ms[n][k])) for k in CATS}) for n in cases},
        copies_vs_shared_bitwise=bitwise,
        random_vs_shared_max_abs_diff=differs,
    )
    res["copies_over_shared"] = res["cases"]["copies"]["tick_ms_p50"] / res["cases"]["shared"]["tick_ms_p50"]
    res["eval_deriv_copies_over_shared"] = res["cases"]["copies"]["kernel_ms_p50"]["eval_deriv"] / res["cases"]["shared"]["kernel_ms_p50"]["eval_deriv"]
    res["eval_trial_copies_over_shared"] = res["cases"]["copies"]["kernel_ms_p50"]["eval_trial"] / res["cases"]["shared"]["kernel_ms_p50"]["eval_trial"]
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    s.close()
    assert all(bitwise.values()), bitwise


if __name__ == "__main__":
    main()
