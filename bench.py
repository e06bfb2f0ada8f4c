#!/usr/bin/env python
"""bench.py — full-dynamics Talos MPC solves/sec (BASELINE.json metric) on N GPUs of one node.

A "step" = one MPC-tick solve (SolverProxDDP.run with max_iters = 1, warm-started: fulldynamic_talos.py:407,532-540)
of EVERY instance of the GLOBAL batch.  Workload = BASELINE.json configs[4]: full-dynamics Talos, T = 100, global batch 4096
(per-instance offset into the contact schedule of fulldynamic_talos.py:256-266 + mirror flag, swing references of
talos_utils.footTrajectory, perturbed measured states; SURVEY 8d config 5) on the synthetic Talos-shaped model.
Instances are independent OCPs: the global batch is cut into contiguous shards of 4096 / N instances, one per rank (STRONG
scaling of the named configuration), and the only collective is the NCCL all-gather of xs / us / K0 / per-instance
summaries (SURVEY 8e) at the end of every step, INSIDE the timed region.  `--batch B` instead fixes the instances per GPU
(weak scaling).  `--config stairs` runs BASELINE configs[3] (stair climbing, global batch 512).

  value  : solves/s with the warm start already resident in HBM (mpc_run_device + device-side gather), whole job over all ranks
  e2e    : same metric through the host-buffer C-ABI call (mpc_run + result read-back), H2D/D2H inside the timing
  roofline: the proximal-Riccati kernel against the fp64 peak measured in this run (SURVEY 8d: fp64-bound path)
  cpu_baseline: the CPU oracle (OpenMP over instances, all host cores, -march=native) on a bounded sample — NOT upstream Aligator
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "full-dynamics Talos MPC solves/sec at batch 4096"
DUMP_INSTANCES = 512  # --dump-outputs: ~38 MB of results; every instance of batch 4096 would be ~300 MB
UNIT = "solves/s"
WORKLOADS = {
    "walk": ("BASELINE configs[4]: full-dynamics Talos MPC tick (solver.setup + 1 ProxDDP iteration), T=100, global batch 4096; instance i sits at tick "
             "t_i ~ U{0..99} of the reference loop (contact schedule of fulldynamic_talos.py:256-266 entering the horizon, swing references of "
             "talos_utils.footTrajectory), mirrored with probability 1/2; warm start = converged solve of the nominal problem, measured state x0 "
             "perturbed per instance (sigma 0.01 m / 0.02 rad / 0.05 s^-1), default_rng(5); synthetic Talos-shaped model"),
    "random": ("BASELINE configs[4] (round-1 generator): full-dynamics Talos MPC tick, T=100, one random contact schedule per instance "
               "(problems.random_schedule), warm start = converged solve of the nominal problem, perturbed measured state, synthetic Talos-shaped model"),
    "stairs": ("BASELINE configs[3]: full-dynamics Talos stair climbing (x_forward 0.3 m, z_height +0.10 m per step, talos_utils.py:187-192), MPC tick, "
               "T=100, global batch 512 perturbed initial states, default_rng(4); synthetic Talos-shaped model"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--global-batch", type=int, default=0, help="instances over ALL GPUs (default 4096; 512 for --config stairs): strong scaling")
    ap.add_argument("--batch", type=int, default=0, help="instances PER GPU (weak scaling); overrides --global-batch")
    ap.add_argument("--config", default="walk", choices=["walk", "random", "stairs"], help="walk = BASELINE configs[4] (default), stairs = configs[3]")
    ap.add_argument("--e2e-parts", type=int, default=2, help="sub-batches of the pipelined host-buffer call in the end-to-end leg (1 = no overlap)")
    ap.add_argument("--no-gather", action="store_true", help="skip the NCCL all-gather of the results (multi-GPU only)")
    ap.add_argument("--prep-iters", type=int, default=20, help="untimed cold-solve iterations that produce the warm start")
    ap.add_argument("--cpu-sample", type=int, default=0, help="instances in the CPU-baseline sample (0 = auto, ~10-30 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-qp", action="store_true", help="skip the batched whole-body QP leg (SURVEY 8f row f-3)")
    ap.add_argument("--qp-only", action="store_true", help="run only the batched whole-body QP leg and print its object")
    ap.add_argument("--latency-ticks", type=int, default=200, help="warm single-instance MPC ticks for the p50 latency (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (xs, us, K0, info) for a "
                    f"fixed, seeded sample of at most {DUMP_INSTANCES} instances of the global batch, and their indices, as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def algorithmic_lq_flops(prob):
    """SURVEY 8d dense-LQ model: sum over instances and knots of F_back + F_fwd for the knot's contact variant."""
    from mpc_benchmark_b200.problems import lq_flops

    f_ds, f_ss = lq_flops(56, 22, 78), lq_flops(56, 22, 61)
    total = 0.0
    for k in prob["knots"]:
        both = (k.cs[0] != 0.0) == (k.cs[1] != 0.0)  # [T,T] and [F,F] both use the two-contact stage (full:108-110)
        total += f_ds if both else f_ss
    return total


def make_problem(args, count=None, lo=0):
    """Instances [lo, lo + count) of the global synthetic batch of the selected configuration (every rank derives its shard from
    the SAME global draw, so the union over ranks is the single-GPU problem)."""
    from mpc_benchmark_b200 import _abi, problems

    G = global_batch(args, 1)
    count = G if count is None else count
    if args.config == "random":
        prob = problems.full_walk_batch(lo + count, seed=5, T=100, stream_ticks=args.steps + 2)
        return problems.sub_problem(prob, lo, lo + count) if lo else prob
    seed = 4 if args.config == "stairs" else 5
    rng = np.random.default_rng(seed)
    n = max(G, lo + count)
    ticks = rng.integers(0, 100, size=n)
    prob = problems.walk_batch(_abi.KIND_FULL, n, seed=seed, T=100, ticks=ticks, stairs=(args.config == "stairs"))
    return problems.sub_problem(prob, lo, lo + count) if (lo or count != n) else prob


def global_batch(args, world):
    if args.batch:
        return args.batch * world
    return args.global_batch or (512 if args.config == "stairs" else 4096)


def config_block(args, world, G, gather):
    """`config` of the JSON line: identical for both arms (the reference arm states its bounded sample in `cpu_baseline.sample`)."""
    Bl = G // world
    par = (f"global batch {G} cut into contiguous shards of {Bl} instances over {world} GPU(s); "
           + ("NCCL all-gather of xs/us/K0/info inside the timed region" if gather else "no collective on the data path"))
    return {"workload": WORKLOADS[args.config], "batch_per_gpu": Bl, "global_batch": G, "horizon": 100, "parallelism": par,
            "l2": "per-step working set (GBs of LQ blocks) >> 126 MB L2; no flush needed", "prep_iters": args.prep_iters}


def cpu_sample_size(args, cores, G):
    """Bounded CPU sample shared by `cpu_baseline` and `--impl reference`: 16 instances per host core (~1 s per step), at most the batch."""
    return int(min(G, args.cpu_sample or 16 * cores))


_NATIVE = None


def oracle_native():
    """Bind the CPU oracle built with -march=native on THIS host (first call builds it); every later oracle call of this process —
    the CPU-baseline leg, the reference arm, the CPU latency comparisons — then runs that build."""
    global _NATIVE
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    if _NATIVE is None:
        _NATIVE = oracle_lib.use_native() if oracle_lib._lib is None else False
    return oracle_lib, _NATIVE


def cpu_tick_rate(args, oracle_lib, n, cores, steps):
    """Solves/s of the CPU oracle on the first n instances of the global batch: untimed nominal solve (the warm start), then `steps`
    timed MPC ticks with OpenMP over instances on all host cores."""
    from mpc_benchmark_b200 import problems

    prob = make_problem(args, count=n)
    nominal = dict(prob, x0=prob["x0_nominal"])
    warm = oracle_lib.solve(nominal, max_iters=args.prep_iters, inst_threads=cores)
    xs, us = problems.warm_tick_inputs(prob, warm["xs"]), warm["us"]
    oracle_lib.solve(prob, max_iters=1, inst_threads=cores, xs=xs, us=us)
    t0 = time.time()
    for _ in range(steps):
        oracle_lib.solve(prob, max_iters=1, inst_threads=cores, xs=xs, us=us)
    dt = time.time() - t0
    flops = algorithmic_lq_flops(prob) + eval_flops(prob)
    return n * steps / dt, dt / steps, flops * steps / dt / 1e9 / cores


def reference_arm(args):
    """--impl reference: the reference's CPU path.  Aligator/Pinocchio are not installable here (SURVEY 8c), so this
    times the repo's CPU oracle (same algorithm, OpenMP over instances, all host cores, -march=native build made on this
    machine) on a bounded sample of the SAME configuration — stated in `cpu_baseline.kind` / `.sample`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    oracle_lib, native = oracle_native()
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cores = os.cpu_count() or 1
    G = global_batch(args, world)
    n = cpu_sample_size(args, cores, G)
    val, step_s, gf = cpu_tick_rate(args, oracle_lib, n, cores, args.steps)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * step_s, "higher_is_better": True, "scaling": "weak" if args.batch else "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config_block(args, world, G, world > 1 and not args.no_gather),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "gflops_per_core": gf,
                             "build": "-O3 -march=native -fopenmp (built on this host)" if native else "-O3 -march=x86-64-v3 -fopenmp",
                             "sample": f"first {n} instances of the global batch x {args.steps} ticks; CPU oracle (not upstream Aligator, which cannot be installed offline)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def eval_flops(prob):
    """Frozen per-knot evaluation FLOPs (BASELINE.md section 4, counted with the instrumented scalar of tools/count_eval_flops.py)."""
    try:
        with open(os.path.join(ROOT, "profiles", "eval_flops.json")) as f:
            t = json.load(f)
    except (OSError, ValueError):
        return 0.0
    total = 0.0
    for k in prob["knots"]:
        both = (k.cs[0] != 0.0) == (k.cs[1] != 0.0)
        total += t["full_ds_deriv"] if both else t["full_ss_deriv"]
    return total + t.get("full_term_deriv", 0.0) * prob["x0"].shape[0]


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)
    if args.qp_only:
        print(json.dumps({"qp": qp_leg(args, int(os.environ.get("LOCAL_RANK", "0")), not args.no_cpu_baseline)}))
        return
    import torch
    import torch.distributed as dist

    from mpc_benchmark_b200 import _native, problems
    from mpc_benchmark_b200.batch import BatchSolver
    from mpc_benchmark_b200.distributed import shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    G, T = global_batch(args, world), 100
    lo, hi = shard_range(G, rank, world)
    B = hi - lo
    if G % world:
        raise SystemExit("bench.py: the global batch must be divisible by the number of GPUs")
    gather = world > 1 and not args.no_gather
    if args.dump_outputs and world > 1 and not gather:
        raise SystemExit("bench.py: --dump-outputs needs the gather of the results when there are several GPUs")
    prob = make_problem(args, count=B, lo=lo)
    solver = BatchSolver(prob["robot"], prob["cfg"], B, device=local)
    # untimed preparation = the reference's first solve (fulldynamic_talos.py:386-397): ProxDDP from the cold start at the
    # NOMINAL state; every timed tick then re-solves from that solution with the instance's MEASURED (perturbed) state at knot 0
    solver.setup(prob["knots"], prob["terms"], prob["x0_nominal"])
    prep = solver.run(prob["xs"], prob["us"], max_iters=args.prep_iters, gains=False)
    xs_h = torch.from_numpy(problems.warm_tick_inputs(prob, prep.xs)).pin_memory()
    us_h = torch.from_numpy(prep.us).pin_memory()
    xs_d, us_d = xs_h.cuda(non_blocking=True), us_h.cuda(non_blocking=True)
    solver.set_x0(prob["x0"])
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream().cuda_stream
    L = _native.lib()
    peaks = {"dfma": L.mpc_measure_fp64_peak(local), "dmma": L.mpc_measure_fp64_peak_dmma(local), "dgemm": dgemm_peak(torch)}
    peak_tf = max(peaks.values())

    # device buffers of the gather: per rank [xs | us | K0 | info] for its shard; all_gather concatenates the rank blocks
    nx, m, n = 57, 22, 56
    per = (T + 1) * nx + T * m + m * n + 8
    pack = torch.empty(B * per, dtype=torch.float64, device="cuda")
    o_us = B * (T + 1) * nx
    o_k0 = o_us + B * T * m
    o_info = o_k0 + B * m * n
    gathered = torch.empty(world * B * per, dtype=torch.float64, device="cuda") if gather else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def export_and_gather():
        base = pack.data_ptr()
        solver.export_results_device(base, base + 8 * o_us, base + 8 * o_k0, base + 8 * o_info, stream)
        if gather:
            dist.all_gather_into_tensor(gathered, pack)

    def tick_device():
        solver.reset_multipliers(stream)  # the reference calls solver.setup(problem) inside every tick (full:539)
        solver.run_device(xs_d.data_ptr(), us_d.data_ptr(), max_iters=1, stream=stream)
        export_and_gather()

    xs_np, us_np = xs_h.numpy(), us_h.numpy()
    out_xs = torch.empty_like(xs_h).pin_memory().numpy()  # results land in pinned host buffers too
    out_us = torch.empty_like(us_h).pin_memory().numpy()

    out_k0 = torch.empty((B, 22, 56), dtype=torch.float64).pin_memory().numpy()

    def tick_e2e():
        solver.reset_multipliers()
        # solver.run on HOST buffers + read-back of what the MPC loop consumes — xs, us and the first feedback gain
        # (fulldynamic_talos.py:540,548-550) — through the pipelined C-ABI call: uploads / downloads of one half of the batch overlap
        # the solve of the other half (mpc_run_pipelined; --e2e-parts 1 = plain mpc_run + mpc_get_results ordering)
        solver.run_pipelined(xs_np, us_np, out_xs, out_us, out_k0, max_iters=1, parts=args.e2e_parts)
        if gather:
            export_and_gather()
        return out_k0

    for _ in range(max(args.warmup, 3)):
        tick_device()
    # ---- timed region 1: inputs resident in HBM
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern = {"eval_deriv": 0.0, "riccati": 0.0, "eval_trial": 0.0, "bookkeeping": 0.0}
    klaunch = {k: 0 for k in kern}
    launches = 0
    ev0.record()
    t0 = time.time()
    for _ in range(args.steps):
        tick_device()
        km = solver.kernel_ms()
        for k in kern:
            kern[k] += km[k][0]
            klaunch[k] += km[k][1]
        launches += solver.last_launches + 1 + (1 if gather else 0)
    ev1.record()
    barrier()
    wall = time.time() - t0
    dev_ms = ev0.elapsed_time(ev1)
    nric = klaunch["riccati"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gathered if gather else pack, G, world, T, nx, m, n)
    # ---- timed region 2: end to end through the host-buffer C-ABI
    tick_e2e()
    barrier()
    t1 = time.time()
    for _ in range(args.steps):
        tick_e2e()
    barrier()
    wall_e2e = time.time() - t1
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- SURVEY 8f row f-2: closed-loop ticks on the device (horizon rotation + warm-start shift + x0 from the model
    # prediction inside mpc_tick; the stage entering each horizon comes from the host), same batch, ideal plant
    stream_fn = prob.get("stream")
    if stream_fn is None:
        last = (type(prob["knots"][0]) * B)(*[prob["knots"][b * T + T - 1] for b in range(B)])
        stream_fn = lambda t: last  # noqa: E731  (the gait's last stage keeps entering the horizon)
    solver.tick(stream_fn(0), None, keep_multipliers=False, max_iters=1)
    barrier()
    t2 = time.time()
    for i in range(args.steps):
        solver.tick(stream_fn(1 + i), None, keep_multipliers=False, max_iters=1)
    barrier()
    wall_cl = time.time() - t2

    # ---- SURVEY 8f row f-4: the same closed loop with the reference's WHOLE per-tick bookkeeping on the device (mpc_gait_tick: sole placements of
    # the predicted state, update_timings, footTrajectory, the 2 x 100 reference writes and the entering stage of every robot), nothing from the host
    cl_gait = None
    try:
        cl_gait = device_gait_leg(args, solver, prob, G, world, torch)
    except Exception as e:  # noqa: BLE001  (an auxiliary leg must never cost the headline line)
        cl_gait = {"error": f"{type(e).__name__}: {e}"}

    tmax = torch.tensor([dev_ms * 1e-3, wall, wall_e2e, wall_cl], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dev_s, wall_s, e2e_s, cl_s = [float(v) for v in tmax.cpu()]
    step_s = max(dev_s, 0.0) / args.steps
    value = G * args.steps / max(dev_s, 1e-12)
    e2e = G * args.steps / e2e_s
    res_iters = solver.results(gains=False, multipliers=False).num_iters

    if rank == 0:
        flops = algorithmic_lq_flops(prob)
        ric_ms = kern["riccati"] / max(nric, 1)
        achieved = flops / (ric_ms * 1e-3) / 1e12 if ric_ms > 0 else None
        traffic, traffic_src = measured_traffic(B)
        hbm_peak, hbm_src = hbm_peak_gbs()
        hbm = None
        if traffic and ric_ms > 0:
            gbs = traffic / (ric_ms * 1e-3) / 1e9
            hbm = {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "peak_source": hbm_src,
                   "note": "secondary roofline of the same kernel: DRAM traffic / duration; far from the HBM bound, the kernel is fp64 / latency bound"}
        h2d = xs_np.nbytes + us_np.nbytes
        d2h = out_xs.nbytes + out_us.nbytes + B * 22 * 56 * 8
        cfg = config_block(args, world, G, gather)
        # (`config` is identical in both arms: what was measured about the workload goes next to it)
        workload_stats = {"tick_iters_done": int(np.min(res_iters)), "double_support_fraction": prob.get("ds_fraction")}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": 1e3 * step_s, "higher_is_better": True, "scaling": "weak" if args.batch else "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": cfg, "workload_stats": workload_stats,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": int(d2h) * world},
            "gpu_launches": int(launches),
            "gather": {"bytes_per_rank_per_step": int(B * per * 8), "bytes_total_per_step": int(world * B * per * 8), "collective": "ncclAllGather (torch.distributed.all_gather_into_tensor) of [xs|us|K0|info]"} if gather else None,
            "closed_loop": {"value": G * args.steps / cl_s, "unit": "robot-ticks/s",
                            "what": "mpc_tick (SURVEY 8f-2): horizon rotation, warm-start shift, x0 <- model prediction, 1 iteration; the next stage of every gait H2D per tick",
                            "device_gait": cl_gait},
            "wall_ms_per_step": 1e3 * wall_s / args.steps,
            "kernel_ms_per_step": {k: v / args.steps for k, v in kern.items()},
            "roofline": {"bound": "fp64", "kernel": "k_riccati (proximal Riccati backward+forward)", "achieved": achieved,
                         "peak": peak_tf, "unit": "TFLOP/s", "frac": (achieved / peak_tf) if achieved else None, "traffic": traffic, "traffic_source": traffic_src, "hbm": hbm,
                         "peak_source": "max of three fp64 micro-benchmarks measured in this run (MEASURED_PEAKS.json has no fp64 entry; SURVEY 8d): " + json.dumps(peaks),
                         "algorithmic_flops_per_launch": flops,
                         "note": "algorithmic = dense LQ model of SURVEY 8d; the kernel skips inactive constraint rows, so executed FLOPs are lower"},
            "clocks": sampler.summary(),
        }
        ef = eval_flops(prob)
        if ef and klaunch["eval_deriv"]:
            ev_ms = kern["eval_deriv"] / klaunch["eval_deriv"]
            ach = ef / (ev_ms * 1e-3) / 1e12
            line["roofline_eval"] = {"bound": "fp64", "kernel": "k_eval<FULL, derivatives>", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                                     "algorithmic_flops_per_launch": ef, "ms_per_launch": ev_ms,
                                     "note": "F_eval frozen by instrumented-scalar counting in the CPU oracle (profiles/eval_flops.json, BASELINE.md section 4)"}
        if world == 1 and not args.no_cpu_baseline:
            oracle_native()
        if args.latency_ticks > 0:
            line["latency"] = single_instance_latency(args, prob, local, not args.no_cpu_baseline and world == 1)
            line["latency"]["other_models"] = other_model_latencies(args, local, not args.no_cpu_baseline and world == 1)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, G)
        if world == 1 and not args.no_qp:
            try:  # an auxiliary leg must never cost the headline line
                line["qp"] = qp_leg(args, local, not args.no_cpu_baseline)
            except Exception as e:  # noqa: BLE001
                line["qp"] = {"error": f"{type(e).__name__}: {e}"}
        print(json.dumps(line))
    solver.close()
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, packed, G, world, T, nx, m, n):
    """Writes xs [S][T+1][nx], us [S][T][m], K0 [S][m][n] and info [S][8] of the instances `instances` [S] (a fixed, seeded sample
    of S = min(G, DUMP_INSTANCES) instances of the global batch, in ascending order) from the packed result buffer of the last
    step: one [xs | us | K0 | info] block per rank, ranks holding contiguous shards in rank order."""
    import torch

    Bl = G // world
    idx = np.sort(np.random.default_rng(0).choice(G, size=min(G, DUMP_INSTANCES), replace=False))
    sel = torch.from_numpy(idx).to(packed.device)
    blocks = packed.view(world, -1)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "instances.npy"), idx.astype(np.float64))
    off = 0
    for name, shape in (("xs", (T + 1, nx)), ("us", (T, m)), ("K0", (m, n)), ("info", (8,))):
        size = Bl * int(np.prod(shape))
        np.save(os.path.join(out_dir, name + ".npy"), blocks[:, off:off + size].reshape(G, *shape)[sel].cpu().numpy())
        off += size


def dgemm_peak(torch):
    """cuBLAS DGEMM 8192^3 (TFLOP/s, best of 3): third candidate of the fp64 roofline denominator (SURVEY 8d)."""
    try:
        n = 8192
        a = torch.randn(n, n, dtype=torch.float64, device="cuda")
        b = torch.randn(n, n, dtype=torch.float64, device="cuda")
        torch.matmul(a, b)
        best = 1e30
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        del a, b
        torch.cuda.empty_cache()
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    except Exception:
        return 0.0


def hbm_peak_gbs():
    """Measured HBM copy bandwidth of this pool (driver-written MEASURED_PEAKS.json), else the profiling recipe's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except (OSError, KeyError, ValueError):
        return 6650.0, "of fallback (B200_PROFILING.md: 6.65 TB/s)"


def measured_traffic(batch):
    """DRAM bytes of one k_riccati launch at this batch, scaled per instance from the committed `ncu --set full` capture
    (profiles/r2_traffic.json; instances are independent CTAs, so the traffic is linear in the batch)."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
        per_inst = (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["batch"]
        return per_inst * batch, f"profiles/r2_traffic.json: {per_inst / 1e6:.1f} MB/instance measured at batch {t['batch']} (algorithmic {t['algorithmic_bytes_per_instance'] / 1e6:.1f} MB), scaled to batch {batch}"
    except (OSError, KeyError, ValueError):
        return None, None


def single_instance_latency(args, prob, device, with_cpu):
    """Second half of the BASELINE metric: single-solve p50 latency (ms) of a warm MPC tick (batch 1, max_iters = 1, host buffers
    in / results out through the C-ABI call, as fulldynamic_talos.py:538-541 times it).  Instance 0 of the bench batch."""
    from mpc_benchmark_b200 import problems
    from mpc_benchmark_b200.batch import BatchSolver

    sub = problems.sub_problem(prob, 0, 1)
    s = BatchSolver(sub["robot"], sub["cfg"], 1, device=device)
    s.setup(sub["knots"], sub["terms"], sub["x0_nominal"])
    # cold solve (SURVEY 8d, config 3): from xs = [x0] * (T + 1), us = 0 to TOL = 1e-5 or 100 iterations (fulldynamic_talos.py:374-397), second run timed
    s.run(sub["xs"], sub["us"], max_iters=100, gains=False)
    s.reset_multipliers()
    t0 = time.perf_counter()
    cold = s.run(sub["xs"], sub["us"], max_iters=100, gains=False)
    cold_ms = 1e3 * (time.perf_counter() - t0)
    s.reset_multipliers()
    warm = s.run(sub["xs"], sub["us"], max_iters=args.prep_iters, gains=False)
    xs, us = problems.warm_tick_inputs(sub, warm.xs), warm.us.copy()
    s.set_x0(sub["x0"])
    ts = []
    for i in range(args.latency_ticks + 10):
        t0 = time.perf_counter()
        s.reset_multipliers()  # the reference re-runs solver.setup inside its timed region
        s.run(xs, us, max_iters=1, gains=False)
        ts.append(1e3 * (time.perf_counter() - t0))
    ts = np.array(ts[10:])
    out = {"p50_ms": float(np.percentile(ts, 50)), "p90_ms": float(np.percentile(ts, 90)), "ticks": int(len(ts)),
           "what": "warm MPC tick, batch 1, host buffers in/out (mpc_run + mpc_get_results)",
           "cold_solve": {"ms": cold_ms, "iterations": int(cold.num_iters[0]), "converged": bool(cold.conv[0]),
                          "what": "ProxDDP from xs = [x0] * (T + 1), us = 0 to TOL 1e-5 or 100 iterations on this instance's horizon (batch 1)"}}
    s.close()
    if with_cpu:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib

        cts = []
        for i in range(6):
            t0 = time.perf_counter()
            oracle_lib.solve(sub, max_iters=1, knot_threads=8, xs=xs, us=us)
            cts.append(1e3 * (time.perf_counter() - t0))
        out["cpu_oracle_8_threads_p50_ms"] = float(np.percentile(cts[1:], 50))
    return out


def other_model_latencies(args, device, with_cpu):
    """BASELINE configs[0] / configs[1] (parity-test cases, reported for reference only): warm single-instance MPC tick of the
    centroidal and kinodynamic problems of the reference scripts' cold-solve setup (standing, T = 100)."""
    from mpc_benchmark_b200 import problems
    from mpc_benchmark_b200.batch import BatchSolver

    out = {}
    for name, maker in (("centroidal", problems.cent_standing_problem), ("kinodynamic", problems.kino_standing_problem)):
        prob = maker(batch=1, T=100)
        s = BatchSolver(prob["robot"], prob["cfg"], 1, device=device)
        s.setup(prob["knots"], prob["terms"], prob["x0"])
        warm = s.run(prob["xs"], prob["us"], max_iters=args.prep_iters, gains=False)
        xs, us = warm.xs.copy(), warm.us.copy()
        ts = []
        for _ in range(min(args.latency_ticks, 50) + 5):
            t0 = time.perf_counter()
            s.reset_multipliers()
            s.run(xs, us, max_iters=1, gains=False)
            ts.append(1e3 * (time.perf_counter() - t0))
        s.close()
        out[name] = {"p50_ms": float(np.percentile(ts[5:], 50))}
        if with_cpu:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib

            cts = []
            for _ in range(4):
                t0 = time.perf_counter()
                oracle_lib.solve(prob, max_iters=1, knot_threads=8, xs=xs, us=us)
                cts.append(1e3 * (time.perf_counter() - t0))
            out[name]["cpu_oracle_8_threads_p50_ms"] = float(np.percentile(cts[1:], 50))
    return out


def device_gait_leg(args, solver, prob, G, world, torch):
    """SURVEY 8f row f-4: the closed loop with the reference's WHOLE per-tick bookkeeping on the device (mpc_gait_tick: sole placements of the predicted state,
    update_timings, footTrajectory, the 2 x 100 reference writes and the entering stage of every robot), nothing from the host."""
    import time

    if world != 1 or args.config == "random":
        return None
    from mpc_benchmark_b200 import gait as gait_mod

    stairs = args.config == "stairs"
    gkw = dict(x_forward=0.3, z_height=0.10, keep_forward=True) if stairs else {}
    solver.gait_setup(gait_mod.device_gait(prob["cfg"].kind, prob["lf"], prob["rf"], prob["com0"], prob["mass"], **gkw), prob.get("mirror"))
    solver.gait_tick()
    solver.tick(None, None, keep_multipliers=False, max_iters=1)
    torch.cuda.synchronize()
    t3 = time.time()
    for i in range(args.steps):
        solver.gait_tick()
        solver.tick(None, None, keep_multipliers=False, max_iters=1)
    torch.cuda.synchronize()
    cl_rate = G * args.steps / (time.time() - t3)
    t4 = time.time()
    for i in range(10):
        solver.gait_tick()
    torch.cuda.synchronize()
    gait_ms = 1e3 * (time.time() - t4) / 10
    cl_gait = {"value": cl_rate, "unit": "robot-ticks/s", "gpu_launches_per_tick_extra": 2, "gait_tick_ms": gait_ms,
               "what": "mpc_gait_tick + mpc_tick: every robot restarts its reference gait at tick 0 (a different workload from `value`: the warm starts "
                       "come from mid-gait horizons, so the first ticks backtrack more); forward kinematics of the predicted state, gait bookkeeping and all T "
                       "per-knot reference blocks on the device (SURVEY 8f-4), then the tick of 8f-2; no host input per tick.  gait_tick_ms = the two gait "
                       "kernels alone for the whole batch"}
    return cl_gait


def qp_leg(args, device, with_cpu, batch=4096, steps=10):
    """SURVEY 8f row f-3: the reference's whole-body inverse-dynamics QP (IDSolver_ulim, QP_utils.py:437-573: n 62, n_eq 40, n_in 18,
    eps_abs 1e-3, 10 x 10 iterations, duality-gap check) at batch 4096.  Inputs = the committed fixture tests/golden/qp_id_talos.npz
    (32 perturbed states of the synthetic Talos-shaped model, DS / left / right support) tiled to the batch, desired accelerations and
    forces perturbed per instance.  value = solve kernel on device-resident QPs; e2e = IDSolver_ulim.solve on host arrays (H2D of M, nle,
    Jc, gamma, a, forces; device assembly; solve; D2H of x, y, z, info)."""
    import time

    from mpc_benchmark_b200 import _native, pin, qp_utils

    d = np.load(os.path.join(ROOT, "tests", "golden", "qp_id_talos.npz"))
    reps = batch // d["M"].shape[0]
    rng = np.random.default_rng(7)
    tile = lambda a: np.ascontiguousarray(np.tile(a, (reps,) + (1,) * (a.ndim - 1)))  # noqa: E731
    cs = tile(d["cs"])
    a = tile(d["a"]) + rng.normal(0, 0.05, (batch, 28))
    f = tile(d["forces"]) + rng.normal(0, 1.0, (batch, 12)) * np.repeat(cs, 6, axis=1)
    M, rbd = tile(d["M"]), qp_utils.RBDTerms(nle=tile(d["nle"]), Jc=tile(d["Jc"]), dJv=tile(d["dJv"]), vf=tile(d["vf"]))
    MU, FL, FW = 0.8, 0.1, 0.075
    solver = qp_utils.IDSolver_ulim(pin.load_talos_like()[0], [1, 1], 2, MU, FL, FW, [0, 1], 6, False, batch=batch, device=device)
    for _ in range(3):
        solver.solve(rbd, cs, None, a, f, M)
    t0 = time.perf_counter()
    for _ in range(steps):
        solver.solve(rbd, cs, None, a, f, M)
    e2e_s = (time.perf_counter() - t0) / steps
    info = solver.qp.results.info
    # the same step fed from the MEASURED STATES: rigid-body terms (crba, nonLinearEffects, frame Jacobians, dJ v) on the device too
    from mpc_benchmark_b200 import problems
    from mpc_benchmark_b200.batch import BatchSolver

    pr = problems.full_standing_problem(batch=1, T=4)
    bs = BatchSolver(pr["robot"], pr["cfg"], 1, device=device)
    xs_meas = tile(d["x"])
    for _ in range(3):
        solver.solve_from_state(bs, xs_meas, cs, a, f)
    t0 = time.perf_counter()
    for _ in range(steps):
        solver.solve_from_state(bs, xs_meas, cs, a, f)
    state_s = (time.perf_counter() - t0) / steps
    solved_state = int((solver.qp.results.info.status == 0).sum())
    bs.close()
    L, h = _native.lib(), solver.qp._handle()
    st = solver.qp.settings.to_c(False)
    import ctypes as C

    ms = []
    for _ in range(3 + steps):  # device-resident: the handle's own buffers hold the assembled QPs; only the solve kernel is launched
        if L.mpc_qp_solve_device(h, batch, C.byref(st), *([0, 0] * 9), 0, 0, 0, 0, 0) != 0:
            raise RuntimeError(L.mpc_qp_last_error().decode())
        ms.append(L.mpc_qp_last_device_ms(h))
    dev_ms = float(np.mean(ms[3:]))
    n, ne, ni = 62, 40, 18
    newton = float(np.mean(info.iter))
    outer = float(np.mean(info.iter_ext))
    # algorithmic FLOPs (dense model, stated in DESIGN.md): per Newton step  K = H + A'A/mu + C'C/mu (symmetric half: n^2 (ne + ni)),
    # Cholesky n^3/3, two triangular solves 2 n^2, gradient / linesearch mat-vecs 2 * 2 n (n + ne + ni); per outer iteration the
    # residuals 2 * 2 n (n + ne + ni)
    fl_newton = n * n * (ne + ni) + n ** 3 / 3 + 2 * n * n + 4 * n * (n + ne + ni)
    fl_outer = 4 * n * (n + ne + ni)
    flops = batch * (newton * fl_newton + (outer + 1) * fl_outer)
    bytes_in = batch * 8 * (ne * n + ne + ni * n + ni) + 8 * (n * n + n + ni)  # A, b, C, l per QP; H, g, u shared
    bytes_out = batch * (8 * (n + ne + ni) + 48)
    out = {"metric": "whole-body inverse-dynamics QPs/s at batch 4096 (IDSolver_ulim: n 62, n_eq 40, n_in 18; eps_abs 1e-3, max_iter 10 x 10, duality-gap check)",
           "value": batch / (dev_ms * 1e-3), "unit": "QPs/s", "ms_per_batch": dev_ms,
           "e2e": {"value": batch / e2e_s, "unit": "QPs/s", "h2d_bytes_per_step": int(batch * 8 * (784 + 28 + 336 + 12 + 28 + 12 + 1)),
                   "d2h_bytes_per_step": int(bytes_out), "what": "IDSolver_ulim.solve on host arrays: H2D, assembly kernel, solve kernel, D2H"},
           "e2e_from_state": {"value": batch / state_s, "unit": "QPs/s", "h2d_bytes_per_step": int(batch * (8 * (57 + 28 + 12) + 8)), "d2h_bytes_per_step": int(bytes_out),
                              "solved": solved_state, "gpu_launches": 4,
                              "what": "IDSolver_ulim.solve_from_state: measured states in, rigid-body terms (k_rbd_terms), gamma, assembly and solve kernels on the device (kinodynamic_talos.py:425-445 for the whole batch)"},
           "gpu_launches": 2, "solved": int((info.status == 0).sum()), "mean_outer_iters": outer, "mean_newton_steps": newton,
           "max_pri_res": float(info.pri_res.max()), "max_dua_res": float(info.dua_res.max()),
           "roofline": {"bound": "fp64 (latency-bound in practice: one 128-thread CTA per QP, 2 QPs per SM)", "achieved": flops / (dev_ms * 1e-3) / 1e12, "unit": "TFLOP/s",
                        "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": int(bytes_in + bytes_out),
                        "hbm_gbs": (bytes_in + bytes_out) / (dev_ms * 1e-3) / 1e9}}
    solver.qp.close()
    if with_cpu:
        oracle_lib, native = oracle_native()
        cores = os.cpu_count() or 1
        nc = min(batch, 64 * cores)
        A, b, Cm, l = oracle_lib.qp_assemble_id(M[:nc], rbd.nle[:nc], rbd.Jc[:nc], _gamma(rbd, cs, nc), a[:nc], f[:nc], cs[:nc], MU, FL, FW)
        H = np.zeros((n, n)); H[:28, :28] = np.eye(28); H[28:40, 28:40] = np.eye(12)
        stc = oracle_lib.qp_default_settings(eps_abs=1e-3, eps_rel=0.0, max_iter=10, max_iter_in=10, check_duality_gap=1)
        oracle_lib.qp_solve(H, np.zeros(n), A, b, Cm, l, np.full(ni, 1e5), settings=stc)
        t0 = time.perf_counter()
        reps_c = 5
        for _ in range(reps_c):
            oracle_lib.qp_assemble_id(M[:nc], rbd.nle[:nc], rbd.Jc[:nc], _gamma(rbd, cs, nc), a[:nc], f[:nc], cs[:nc], MU, FL, FW)
            oracle_lib.qp_solve(H, np.zeros(n), A, b, Cm, l, np.full(ni, 1e5), settings=stc)
        cs_ = (time.perf_counter() - t0) / reps_c
        out["cpu_baseline"] = {"value": nc / cs_, "unit": "QPs/s", "cores": cores, "kind": "port",
                               "build": "-O3 -march=native -fopenmp (built on this host)" if native else "-O3 -march=x86-64-v3 -fopenmp",
                               "sample": f"first {nc} QPs of the batch x {reps_c} passes (assembly + solve), CPU oracle oracle/qp.hpp with OpenMP over QPs (not proxsuite: not installable offline)"}
    return out


def _gamma(rbd, cs, nc):
    g = np.array(rbd.dJv[:nc], float).reshape(nc, 2, 6).copy()
    vf = np.asarray(rbd.vf[:nc], float).reshape(nc, 2, 6)
    g[:, :, :3] += vf[:, :, :3] + vf[:, :, 3:]
    return (g * np.asarray(cs[:nc]).reshape(nc, 2, 1)).reshape(nc, 12)


def cpu_baseline(args, G):
    """CPU oracle (-march=native build made on this host) on the box's host cores over the SAME bounded sample the reference arm
    times: the first 16 x cores instances of the global batch, one warm MPC tick each."""
    oracle_lib, native = oracle_native()
    cores = os.cpu_count() or 1
    n = cpu_sample_size(args, cores, G)
    steps = 3
    val, step_s, gf = cpu_tick_rate(args, oracle_lib, n, cores, steps)
    return {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "gflops_per_core": gf,
            "build": "-O3 -march=native -fopenmp (built on this host)" if native else "-O3 -march=x86-64-v3 -fopenmp",
            "sample": f"first {n} instances of the global batch x {steps} ticks, {step_s:.2f} s per tick; CPU oracle with OpenMP over instances "
                      "(not upstream Aligator: not installable offline)"}


if __name__ == "__main__":
    main()
