#!/usr/bin/env python
"""Generates tests/golden/*.npz:

    python tests/golden/make_golden.py [REFERENCE_DIR]

1. ref_flat_{full,kino,cent}.npz (only with REFERENCE_DIR, a checkout of the edantec/MPC_benchmark scripts) — the flat descriptor
   obtained by executing the TOP HALF of the unmodified reference script (REFERENCE_DIR/{fulldynamic,kinodynamic,centroidal}_talos.py
   up to the cold solve) through this package's aligator/pinocchio shim (tests/ref_harness.py), plus the cold-solve result of the
   CPU ORACLE on that descriptor (without the feedback gains, which no test reads: they would take the files over 1 MB).
2. walk_full.npz — 4 instances of the synthetic random-schedule workload (bench.py) with 6 oracle iterations and one
   warm MPC tick (active cone / box constraints, non-zero multipliers).

The reference has no tests or golden vectors of its own and Aligator cannot be installed offline (SURVEY 8c), so these
fixtures pin the CUDA path to the ORACLE, not to upstream Aligator: PARITY UNPINNED.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_lib as O  # noqa: E402
import ref_harness as H  # noqa: E402
from mpc_benchmark_b200 import problems  # noqa: E402


def pack(prob):
    return dict(robot=np.frombuffer(bytes(prob["robot"]), dtype=np.uint8), cfg=np.frombuffer(bytes(prob["cfg"]), dtype=np.uint8),
                knots=np.frombuffer(bytes(prob["knots"]), dtype=np.uint8), terms=np.frombuffer(bytes(prob["terms"]), dtype=np.uint8),
                x0=prob["x0"], xs=prob["xs"], us=prob["us"])


def info_arrays(info):
    return dict(num_iters=np.array([i.num_iters for i in info]), conv=np.array([i.conv for i in info]),
                prim_infeas=np.array([i.prim_infeas for i in info]), dual_infeas=np.array([i.dual_infeas for i in info]),
                traj_cost=np.array([i.traj_cost for i in info]), ls_evals=np.array([i.ls_evals for i in info]))


def main(ref_dir=None):
    if ref_dir:
        for script, tag in [("fulldynamic_talos.py", "full"), ("kinodynamic_talos.py", "kino"), ("centroidal_talos.py", "cent")]:
            ns, cap = H.run_top_half(script, ref_dir)
            assert [c[0] for c in cap] == ["setup", "run"], script
            flat, xs, us = cap[-1][1], cap[-1][2], cap[-1][3]
            prob = dict(robot=flat.robot, cfg=flat.cfg, knots=flat.knots, terms=flat.terms, x0=flat.x0, xs=xs[None], us=us[None])
            r = O.solve(prob, knot_threads=8)
            out = pack(prob)
            out.update({"sol_" + k: r[k] for k in ["xs", "us", "vs", "lams", "stage0"]})
            out.update({"sol_" + k: v for k, v in info_arrays(r["info"]).items()})
            np.savez_compressed(os.path.join(HERE, f"ref_flat_{tag}.npz"), **out)
            print(script, "iters", out["sol_num_iters"], "conv", out["sol_conv"], "prim", out["sol_prim_infeas"])
    prob = problems.full_walk_batch(4, seed=11, T=40)
    r = O.solve(prob, max_iters=6, inst_threads=4)
    tick = O.solve(prob, max_iters=1, inst_threads=4, xs=r["xs"], us=r["us"])
    out = pack(prob)
    out.update({"sol_" + k: r[k] for k in ["xs", "us", "vs", "lams"]})
    out.update({"sol_" + k: v for k, v in info_arrays(r["info"]).items()})
    out.update({"tick_" + k: tick[k] for k in ["xs", "us", "vs", "lams", "stage0"]})
    out.update({"tick_" + k: v for k, v in info_arrays(tick["info"]).items()})
    np.savez_compressed(os.path.join(HERE, "walk_full.npz"), **out)
    print("walk: iters", out["sol_num_iters"], "ls", out["sol_ls_evals"], "max |vs|", np.abs(r["vs"]).max(), "tick ls", out["tick_ls_evals"])


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
