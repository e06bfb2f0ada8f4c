"""Throughput of the IKID whole-body QP (IKIDSolver_f6, QP_utils.py:584-768: n 62, n_eq 40, n_in 18, box; eps_abs 1e-3, 100 x 100
iterations) at batch 4096, two ways:
  solve             the cost H, g built on the host (batched numpy) from caller-supplied rigid-body and task terms, uploaded with M, nle,
                    Jc, gamma, a, forces; device constraint assembly; solve kernel; results back;
  solve_from_state  measured states, PD task errors and forces uploaded; rigid-body and task terms (k_ikid_terms), the whole assembly
                    (k_qp_assemble_ikid) and the solve kernel on the device; results back.
Workload: the committed fixture states (tests/golden/qp_id_talos.npz) tiled to the batch, PD errors and dH seeded, general gain matrices.
The host path is fed the device's own terms of those states, so both solve the same QPs.  Bytes per step are counted from the array
shapes.  Writes <out>/ikid_qp_bench.json with the GPU name and power limit read in the same run; fails without a GPU.
usage: python tools/ikid_qp_bench.py --out DIR [--batch 4096] [--steps 10] [--warmup 3]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mpc_benchmark_b200 import pin, problems, qp_utils  # noqa: E402
from mpc_benchmark_b200.batch import BatchSolver  # noqa: E402

MU, FOOT_L, FOOT_W = 0.8, 0.1, 0.075
TASK = ("q_diff", "dq_diff", "LF_diff", "dLF_diff", "RF_diff", "dRF_diff", "base_diff", "dbase_diff", "torso_diff", "dtorso_diff")


def gpu_identity():
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("ikid_qp_bench: no CUDA device (this measurement runs on the GPU only)")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else None}


def inputs(B, seed=9):
    d = np.load(os.path.join(ROOT, "tests", "golden", "qp_id_talos.npz"))
    rng = np.random.default_rng(seed)
    reps = -(-B // d["x"].shape[0])
    tile = lambda a: np.ascontiguousarray(np.tile(a, (reps,) + (1,) * (a.ndim - 1))[:B])  # noqa: E731
    t = dict(x=tile(d["x"]), cs=tile(d["cs"]), forces=tile(d["forces"]), dH=rng.normal(0, 1.0, (B, 6)))
    for k, m, s in zip(TASK, (28, 28, 6, 6, 6, 6, 3, 3, 3, 3), (0.02, 0.05, 0.01, 0.02, 0.01, 0.02, 0.02, 0.05, 0.02, 0.05)):
        t[k] = rng.normal(0, s, (B, m))
    K = lambda k, m: np.eye(m) * k + rng.normal(0, 0.1 * k, (m, m))  # noqa: E731
    t["K_gains"] = [[K(100, 28), K(20, 28)], [K(400, 6), K(40, 6)], None, [K(100, 3), K(20, 3)]]
    t["weights"] = [1.0, 100.0, 0.1, 10.0, 1e-3]
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    gpu = gpu_identity()
    B = a.batch
    t = inputs(B)
    model = pin.load_talos_like()[0]
    pr = problems.full_standing_problem(batch=1, T=4)
    dev = BatchSolver(pr["robot"], pr["cfg"], 1)
    s = qp_utils.IKIDSolver_f6(model, t["weights"], t["K_gains"], 2, MU, FOOT_L, FOOT_W, [0, 1], model.getFrameId("base_link"),
                               model.getFrameId("torso_2_link"), 6, False, batch=B)
    M, rbd = dev.ikid_terms(t["x"], s._frames())
    v = t["x"][:, 29:]
    task = [t[k] for k in TASK]

    def host():
        return s.solve(rbd, t["cs"], v, *task, t["forces"], t["dH"], M)

    def from_state():
        return s.solve_from_state(dev, t["x"], t["cs"], *task, t["forces"], t["dH"])

    res = {}
    for name, fn in (("solve", host), ("solve_from_state", from_state)):
        for _ in range(a.warmup):
            fn()
        dev_ms = []
        t0 = time.perf_counter()
        for _ in range(a.steps):
            fn()
            dev_ms.append(s.qp.results.info.run_time * 1e-3)
        step_s = (time.perf_counter() - t0) / a.steps
        info = s.qp.results.info
        res[name] = {"qps_per_s": B / step_s, "ms_per_step": 1e3 * step_s, "solve_kernel_ms": float(np.mean(dev_ms)),
                     "solved": int((info.status == 0).sum()), "max_pri_res": float(info.pri_res.max()), "max_dua_res": float(info.dua_res.max()),
                     "mean_outer_iters": float(np.mean(info.iter_ext)), "mean_newton_steps": float(np.mean(info.iter))}
    n, ne, nz = 62, 40, 18 + 62
    d2h = B * (8 * (n + ne + nz) + 48)  # x, y, z, info
    res["solve"].update(h2d_bytes_per_step=B * (8 * (n * n + n + 784 + 28 + 336 + 12 + 28 + 12) + 8) + 8 * 2 * n, d2h_bytes_per_step=d2h,
                        what="IKIDSolver_f6.solve on host arrays: H, g (numpy), M, nle, Jc, gamma, a, forces, cs and the shared box bounds up")
    res["solve_from_state"].update(h2d_bytes_per_step=B * (8 * (57 + 98 + 12) + 8) + 8 * 1658, d2h_bytes_per_step=d2h,
                                   what="IKIDSolver_f6.solve_from_state: states, task errors, forces, cs and the shared gains up; k_ikid_terms, "
                                        "k_qp_assemble_ikid and the solve kernel on the device")
    out = {"metric": f"IKID whole-body QPs/s at batch {B} (IKIDSolver_f6: n 62, n_eq 40, n_in 18, box; eps_abs 1e-3, max_iter 100 x 100)",
           "gpu": gpu, "batch": B, "steps": a.steps, "warmup": a.warmup, **res,
           "speedup_from_state_over_solve": res["solve_from_state"]["qps_per_s"] / res["solve"]["qps_per_s"]}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "ikid_qp_bench.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))
    s.qp.close()
    dev.close()


if __name__ == "__main__":
    main()
