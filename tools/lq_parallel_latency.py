"""Single-instance latency of the time-parallel LQ solve (mpc_config_t.lq_legs): warm one-iteration MPC ticks on the reference walking
horizons (problems.walk_batch) of every model kind, for lq_legs in {0, 2, 4, 8, 16} at batch 1, 8 and 64.  Reports the tick's device
time (p50 / p90), the per-category kernel time of the median tick, and the largest difference of xs / us / K0 to lq_legs = 0 from the
same starting point: after the cold solve, after the first tick, and over the whole closed loop (where the model prediction feeds the
next tick, so a rounding-level difference that flips one linesearch decision carries over to all later ticks).  Reads the GPU name
and power limit in the same run.

    python tools/lq_parallel_latency.py [--out profiles/lq_parallel_latency_b200.json] [--ticks 30]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mpc_benchmark_b200 import _abi, problems  # noqa: E402
from mpc_benchmark_b200.batch import BatchSolver  # noqa: E402

KINDS = {"full": _abi.KIND_FULL, "kino": _abi.KIND_KINO, "cent": _abi.KIND_CENT}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clk)


def run_config(prob, legs, B, ticks, warmup):
    cfg = _abi.Config.from_buffer_copy(prob["cfg"])
    cfg.lq_legs = legs
    s = BatchSolver(prob["robot"], cfg, B)
    s.setup(prob["knots"], prob["terms"], prob["x0"])
    res = [s.run(prob["xs"], prob["us"], max_iters=10)]
    times, cats = [], []
    for t in range(warmup + ticks):
        s.tick(max_iters=1)
        if t >= warmup:
            times.append(s.last_device_ms)
            cats.append({k: v[0] for k, v in s.kernel_ms().items()})
        if t == 0 or t == warmup + ticks - 1:
            res.append(s.results(multipliers=False))
    s.close()
    med = int(np.argsort(times)[len(times) // 2])
    return dict(p50_ms=float(np.percentile(times, 50)), p90_ms=float(np.percentile(times, 90)), kernel_ms_median_tick=cats[med]), res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lq_parallel_latency_b200.json"))
    ap.add_argument("--ticks", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    out = dict(gpu=gpu_info(), what="warm one-iteration mpc_tick (max_iters = 1) after a 10-iteration cold solve; device time per tick (CUDA events)",
               ticks=a.ticks, warmup=a.warmup, results=[])
    for kname, kind in KINDS.items():
        for B in (1, 8, 64):
            prob = problems.walk_batch(kind, B, seed=5)
            base = None
            for legs in (0, 2, 4, 8, 16):
                row, r = run_config(prob, legs, B, a.ticks, a.warmup)
                if base is None:
                    base = r
                d = lambda x, y: float(np.abs(x - y).max() / max(1e-300, np.abs(y).max()))  # noqa: E731
                diffs = {when: dict(xs=d(x.xs, y.xs), us=d(x.us, y.us), K0=d(x.K[:, 0], y.K[:, 0]))
                         for when, x, y in zip(("cold_solve", "first_tick", "last_tick"), r, base)}
                row.update(kind=kname, batch=B, lq_legs=legs, max_rel_diff_vs_serial=diffs,
                           iters_equal=bool(all(list(x.num_iters) == list(y.num_iters) for x, y in zip(r, base))))
                out["results"].append(row)
                print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
