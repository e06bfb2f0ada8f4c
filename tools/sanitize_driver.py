"""Tiny solves of the three model kinds for compute-sanitizer (memcheck / racecheck) runs on the GPU box.
usage: compute-sanitizer --tool racecheck python tools/sanitize_driver.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mpc_benchmark_b200 import problems  # noqa: E402
from mpc_benchmark_b200.batch import BatchSolver  # noqa: E402


def run(name, prob, iters):
    b = prob["x0"].shape[0]
    s = BatchSolver(prob["robot"], prob["cfg"], b, device=0)
    s.setup(prob["knots"], prob["terms"], prob["x0"])
    r = s.run(prob["xs"], prob["us"], max_iters=iters)
    print(name, "iters", r.num_iters, "prim", r.prim_infeas, "ls", r.ls_evals)
    s.close()


def main():
    # batch 2 launches the full-dynamics Riccati kernel with 256 threads per instance; batches above the SM count use 128
    run("full walk", problems.full_walk_batch(2, seed=3, T=12), 3)
    cold = problems.full_walk_batch(2, seed=3, T=12)
    cold["x0"] = problems.perturbed_x0(cold["robot"], cold["x0"][0], __import__("numpy").random.default_rng(2), 2)  # many active rows: scratch path
    run("full walk, perturbed cold start", cold, 2)
    nl = problems.full_walk_batch(2, seed=3, T=12)
    nl["cfg"].rollout = 1
    run("full walk, nonlinear rollout kernel", nl, 2)
    run("kino standing", problems.kino_standing_problem(batch=2, T=10), 2)
    run("cent standing", problems.cent_standing_problem(batch=2, T=20), 2)
    gait_loop()


def gait_loop():
    """Device-side gait bookkeeping (k_feet_of_prediction, k_gait_tick) + closed-loop ticks, full dynamics and kinodynamic."""
    from mpc_benchmark_b200 import _abi, gait

    for kind, maker in ((_abi.KIND_FULL, problems.full_standing_problem), (_abi.KIND_KINO, problems.kino_standing_problem)):
        prob = maker(batch=2, T=12)
        s = BatchSolver(prob["robot"], prob["cfg"], 2, device=0)
        s.setup(prob["knots"], prob["terms"], prob["x0"])
        s.run(prob["xs"], prob["us"], max_iters=2)
        urefs = gait.force_ramp_refs(kind, prob["mass"], 34, 12) if kind == _abi.KIND_KINO else None
        s.gait_setup(gait.device_gait(kind, prob["lf"], prob["rf"], prob["com0"], prob["mass"]), [False, True], urefs)
        s.set_tail_warmstart(kind == _abi.KIND_FULL)  # phase-matched warm start of the appended knot (k_shift_warmstart, mode 1)
        for _ in range(3):
            s.gait_tick()
            s.tick(None, None, keep_multipliers=(kind == _abi.KIND_KINO), max_iters=1)
        print("gait loop kind", kind, "iters", s.results(gains=False).num_iters)
        s.close()


if __name__ == "__main__":
    main()
