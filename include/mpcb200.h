/*
 * mpcb200.h — C-ABI of the B200-native batched ProxDDP path (libmpcb200.so).
 *
 * This header is the drop-in boundary for the ONE hot path of edantec/MPC_benchmark:
 * `aligator.SolverProxDDP.setup/run` on the three Talos walking OCPs
 * (reference call sites: fulldynamic_talos.py:379-397,539-540; kinodynamic_talos.py:285-304,490;
 *  centroidal_talos.py:270-288,462).  The reference crosses Python -> C++ through
 * eigenpy/Boost.Python objects; here the Python shim (package `mpc_benchmark_b200`, importable
 * `as aligator`) flattens its object graph into the plain structs below and calls these
 * entry points through ctypes.  No torch types appear in any signature: device buffers are raw
 * device pointers (uint64 from torch.Tensor.data_ptr()), the stream is a raw cudaStream_t.
 *
 * All arithmetic is fp64.  All matrices are row-major.  SE(3) placements are 12 doubles:
 * rotation row-major (9) then translation (3).  Spatial vectors are [linear; angular].
 */
#ifndef MPCB200_H
#define MPCB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPC_KIND_CENT 0 /* centroidal_talos.py   : n=9,  m=12, nc<=34 */
#define MPC_KIND_KINO 1 /* kinodynamic_talos.py  : n=56, m=34, nc<=68 */
#define MPC_KIND_FULL 2 /* fulldynamic_talos.py  : n=56, m=22, nc<=78 */

#define MPC_NB 23  /* bodies: free-flyer base + 22 revolute (plot.py:488-490) */
#define MPC_NV 28
#define MPC_NQ 29
#define MPC_NJ 22
#define MPC_MAXU 34
#define MPC_MAXC 78

/* Robot tree = DATA (SURVEY App. B).  Body 0 is the free-flyer base; bodies must be ordered
 * parents-first.  Tangent index of body b>0 is 5+b. */
typedef struct mpc_robot {
  int32_t nb;
  int32_t parent[MPC_NB];       /* -1 for the base */
  double jplace[MPC_NB][12];    /* joint placement in the parent body frame */
  double axis[MPC_NB][3];       /* revolute axis in the joint frame (unit); unused for body 0 */
  double mass[MPC_NB];
  double com[MPC_NB][3];        /* in body frame */
  double inertia[MPC_NB][9];    /* rotational inertia about the com, body axes, row-major */
  int32_t foot_body[2];         /* left, right sole frames: parent body + placement */
  int32_t pad_;
  double foot_place[2][12];
  double q_lo[MPC_NJ], q_hi[MPC_NJ], tau_max[MPC_NJ];
  double gravity[3];            /* (0,0,-9.81) */
} mpc_robot_t;

/* Global (per problem family) constants: SURVEY App. C. */
typedef struct mpc_config {
  int32_t kind;
  int32_t T;                    /* knots in the horizon (100) */
  double dt;
  /* running costs */
  double x_ref[MPC_NQ + MPC_NV];/* QuadraticStateCost target (full:175, kino:140) */
  double wx[2 * MPC_NV];        /* diagonal of w_x */
  double wu[MPC_MAXU];          /* diagonal of w_u / w_control */
  double w_cent[6];             /* CentroidalMomentumResidual weight diag (full:141-143) */
  double w_centder[6];          /* kino:103-105 */
  double w_force[6];            /* ContactForceResidual weight diag (full:149-151) */
  /* terminal cost (full:234-245); all-zero = empty CostStack (kino:175, cent:249) */
  double wx_term[2 * MPC_NV];
  double w_cent_term[6];
  double w_foot_term[6];
  /* contact / cone parameters */
  double mu_fric, foot_L, foot_W;
  double kp[6], kd[6];          /* Baumgarte corrector (full:93-94) */
  double contact_place[2][12];  /* world placements of the two rigid contacts (full:83) */
  double mu_contact;            /* ProximalSettings mu (full:77) */
  /* centroidal model (cent:187-200) */
  double mass;
  double w_linmom[3], w_angmom[3], w_linacc[3], w_angacc[3], w_com[3], com_ref[3];
  /* solver (full:374-386) */
  double tol, mu_init;
  int32_t max_iters;
  int32_t force_initial_condition;
  int32_t rollout;              /* solver.rollout_type (full:381): 0 = ROLLOUT_LINEAR (every reference script), 1 = ROLLOUT_NONLINEAR */
  int32_t pad_;
} mpc_config_t;

/* Per-knot parameter block (one per instance per knot). */
typedef struct mpc_knot {
  double cs[2];        /* contacts in the dynamics (left, right), 0/1 */
  double fcost[2];     /* ContactForceResidual cost present (full:187-201) */
  double w_lf[6], w_rf[6]; /* FramePlacement cost weight diag; 0 = off (full:177-185) */
  double lf_ref[12], rf_ref[12];
  double f_ref[12];    /* contact-force references L,R (full:188-201) */
  double u_ref[MPC_MAXU]; /* control reference (cent:225, kino:142, full:176) */
  double cpos[6];      /* centroidal contact positions L,R (cent:209-210) */
} mpc_knot_t;

typedef struct mpc_term {
  double lf_ref[12], rf_ref[12];
  double com_ref[3];
  double has_com_cstr; /* terminal CoM equality (full:499-507, kino:176-180) */
} mpc_term_t;

/* Per-instance solve summary (mirrors aligator Results scalars). */
typedef struct mpc_info {
  double prim_infeas, dual_infeas, traj_cost, merit;
  double mu;
  double alpha;      /* step length accepted by the last linesearch */
  int32_t num_iters, al_iters, conv, status; /* status: 0 converged,1 max-iters,2 non-finite,3 reg saturated */
  int32_t ls_evals;  /* trial evaluations spent in linesearches during the run */
  int32_t pad_;
} mpc_info_t;

typedef struct mpc_solver mpc_solver_t; /* opaque */

/* Replaces SolverProxDDP(tol, mu_init) + the model carried by pin.Model (full:27-97, 379). */
mpc_solver_t *mpc_create(const mpc_robot_t *robot, const mpc_config_t *cfg, int32_t batch, int32_t device);
void mpc_destroy(mpc_solver_t *h);
const char *mpc_last_error(void);

/* solver.setup(problem): (re)allocate the device workspace for `batch` instances of T knots
 * (full:388,539).  Host pointers: knots [batch][T], terms [batch], x0 [batch][nx]. */
int32_t mpc_setup(mpc_solver_t *h, const mpc_knot_t *knots, const mpc_term_t *terms, const double *x0);
/* setReference / contact_poses / u_ref updates of knots [first, first+count) of every instance. */
int32_t mpc_update_knots(mpc_solver_t *h, const mpc_knot_t *knots, int32_t first, int32_t count);
int32_t mpc_update_terms(mpc_solver_t *h, const mpc_term_t *terms);
/* replaceStageCircular + cycleAppend (full:496-497): drop knot 0, append `last` ([batch]) at T-1. */
int32_t mpc_cycle(mpc_solver_t *h, const mpc_knot_t *last);
/* solver.cycleProblem / workspace.cycleAppend (kino:488, full:497): shift the warm multipliers by n knots — the multipliers of the
 * running knots and the co-states of x_1..x_T move left and repeat their last entry; the terminal multiplier vs[T] and the
 * initial-condition co-state lams[0] stay in place. */
int32_t mpc_shift_multipliers(mpc_solver_t *h, int32_t n);
/* New robot / weight constants for the same kind, horizon and batch (the shim re-derives them from the object graph at every run). */
int32_t mpc_reconfigure(mpc_solver_t *h, const mpc_robot_t *robot, const mpc_config_t *cfg);
/* problem.x0_init = x (full:536); host pointer [batch][nx]. */
int32_t mpc_set_x0(mpc_solver_t *h, const double *x0);

/* solver.run(problem, xs_init, us_init) with HOST buffers (full:393-397,540):
 * xs [batch][T+1][nx], us [batch][T][nu]; copies in, runs up to max_iters ProxDDP iterations
 * per instance, copies results back with mpc_get_results. */
int32_t mpc_run(mpc_solver_t *h, const double *xs_init, const double *us_init, int32_t max_iters);
/* solver.run + the results read-back (results.xs / .us / controlFeedbacks()[0], fulldynamic_talos.py:540,548-550) as ONE call on
 * HOST buffers, pipelined: the batch is cut into `parts` (1..8) contiguous sub-batches; the upload of the next part and the download
 * of the previous one overlap the solve of the current one on a second stream (pinned host memory makes the copies asynchronous;
 * pageable memory works, without overlap).  Outputs may be NULL.  Layouts: xs_out [batch][T+1][nx], us_out [batch][T][nu],
 * K0_out [batch][nu][ndx], info_out [batch].  Instance results are identical to mpc_run + mpc_get_results. */
int32_t mpc_run_pipelined(mpc_solver_t *h, const double *xs_init, const double *us_init, int32_t max_iters, int32_t parts, double *xs_out,
                          double *us_out, double *K0_out, mpc_info_t *info_out);
/* Same, with the trajectories already resident in device memory (device pointers, same layout); kernels are
 * launched on `stream` (a cudaStream_t, 0 = the handle's own).  The call returns after the solve has finished:
 * the iteration / linesearch control reads per-batch counters back between launches. */
int32_t mpc_run_device(mpc_solver_t *h, uint64_t xs_dev, uint64_t us_dev, int32_t max_iters, uint64_t stream);

/* What the per-tick solver.setup(problem) of the reference does to the solver state (full:539, cent:461) without
 * re-uploading the problem: multipliers vs / lams back to zero.  Asynchronous on `stream` (0 = the handle's own stream). */
int32_t mpc_reset_multipliers(mpc_solver_t *h, uint64_t stream);

/* One closed-loop MPC tick on the device (SURVEY 8f row f-2; the loop body of fulldynamic_talos.py:496-497,532-540):
 * append `last` ([batch], may be NULL) at the end of the horizon, shift the previous solution by one knot as warm start,
 * x0 <- x_meas ([batch][nx] host) or the model prediction xs[1] when NULL (ideal plant), multipliers reset (setup per tick)
 * or shifted (keep_multipliers, kinodynamic_talos.py:488), then max_iters ProxDDP iterations. */
int32_t mpc_tick(mpc_solver_t *h, const mpc_knot_t *last, const double *x_meas, int32_t keep_multipliers, int32_t max_iters);
/* Control warm start of the knot mpc_tick appends: 0 (default) = the previous knot's control, what the scripts pass to solver.run
 * (us = us[1:] + [us[-1]], fulldynamic_talos.py:534); 1 = the control of the nearest knot of the horizon with the SAME contact phase (not in the reference:
 * it keeps single-support torques out of the first double-support knot after a swing phase and vice versa, which is what the one-iteration full-dynamics
 * loop needs to walk, DESIGN section 7). */
int32_t mpc_set_tail_warmstart(mpc_solver_t *h, int32_t mode);

/* solver.results: xs, us, controlFeedbacks() [batch][T][nu][ndx], vs, lams; any pointer may be NULL. */
int32_t mpc_get_results(mpc_solver_t *h, double *xs, double *us, double *K, double *vs, double *lams,
                        mpc_info_t *info);
/* Device-resident result pointers (for NCCL gathers without a host bounce). */
int32_t mpc_result_ptrs(mpc_solver_t *h, uint64_t *xs, uint64_t *us, uint64_t *K, uint64_t *info);
/* Same results, packed into CALLER-OWNED device buffers for a gather over NVLink (SURVEY 8e): xs [batch][T+1][nx], us [batch][T][nu],
 * K0 [batch][nu][ndx] (controlFeedbacks()[0]), info [batch][8] doubles = prim_infeas, dual_infeas, traj_cost, merit, num_iters,
 * conv, status, alpha.  Any pointer may be 0.  Asynchronous on `stream` (0 = the handle's own); run it after mpc_run_device on the
 * same stream and hand the buffers to ncclAllGather / torch.distributed.all_gather_into_tensor. */
int32_t mpc_export_results_device(mpc_solver_t *h, uint64_t xs_dev, uint64_t us_dev, uint64_t K0_dev, uint64_t info_dev, uint64_t stream);
/* workspace.problem_data.stage_data[k].dynamics_data.continuous_data.{xdot, contact_force}
 * (full:467-480): xdot [batch][ndx], force [batch][12]. */
int32_t mpc_get_stage_data(mpc_solver_t *h, int32_t k, double *xdot, double *contact_force);

/* controlFeedbacks()[k] of every instance (fulldynamic_talos.py:405,550): K [batch][nu][ndx]. */
int32_t mpc_get_feedback(mpc_solver_t *h, int32_t k, double *K);
/* Device time (ms, CUDA events on the launch stream) and launch count of the last run per kernel category:
 * 0 evaluation+derivatives, 1 proximal Riccati, 2 trial (values-only) evaluation, 3 bookkeeping kernels. */
double mpc_last_kernel_ms(mpc_solver_t *h, int32_t category);
int32_t mpc_last_kernel_launches(mpc_solver_t *h, int32_t category);
void mpc_set_profiling(mpc_solver_t *h, int32_t on);

/* Number of kernels launched by the last mpc_run* call and device time (ms) between its first and
 * last launch as measured with CUDA events on the launch stream. */
int32_t mpc_last_launches(mpc_solver_t *h);
double mpc_last_device_ms(mpc_solver_t *h);

/* Test / measurement hook on the same kernels (parity tests call this): ONE derivative evaluation of every knot at
 * (xs, us) [batch layouts as mpc_run]; copies the LQ blocks of instance `inst` to host arrays (NULL = skip):
 * AB [T][n][n+m], H [T+1][n+m][n+m], g [T+1][n+m] (Lagrangian gradient), gap [T][n], h [T+1][nc], scal [T+1][8]. */
int32_t mpc_debug_lq(mpc_solver_t *h, const double *xs, const double *us, int32_t inst, double *AB, double *H, double *g,
                     double *gap, double *hval, double *scal);
/* Unit-test hook of the FP64 tensor-core tile GEMM used by the Riccati kernel: C (8mt x 8nt, ldc) = A^T B with
 * A [K][lda], B [K][ldb] (host pointers, K % 4 == 0). */
int32_t mpc_debug_gemm_tn(int32_t mt, int32_t nt, int32_t K, const double *A, int32_t lda, const double *B, int32_t ldb, double *C,
                          int32_t ldc);
/* Per-phase cycle counters (all zero unless built with -DMPC_PHASE_TIMING): out64 = 16 Riccati phases, 16 phases of the
 * derivative evaluation kernel, 16 phases of the values-only (linesearch trial) evaluation kernel, 16 Riccati sub-phases. */
int32_t mpc_debug_phases(mpc_solver_t *h, double *out64);
/* Rigid-body terms of the reference's whole-body QPs for `count` measured states x [count][nx] (what kinodynamic_talos.py:425-431 /
 * QP_utils.py:515-528 take from pinocchio: crba, nonLinearEffects, getFrameJacobian / getFrameJacobianTimeVariation(LOCAL) of the two
 * sole frames, getFrameVelocity): M [count][nv][nv], nle [count][nv], Jc [count][12][nv], dJv [count][12], vf [count][2][6] (LOCAL:
 * linear, angular).  Host arrays (any output may be NULL) / device pointers + stream (asynchronous).  Uses the handle's robot model only;
 * not available for MPC_KIND_CENT. */
int32_t mpc_rbd_terms(mpc_solver_t *h, int32_t count, const double *x, double *M, double *nle, double *Jc, double *dJv, double *vf);
int32_t mpc_rbd_terms_device(mpc_solver_t *h, int32_t count, uint64_t x_dev, uint64_t M_dev, uint64_t nle_dev, uint64_t Jc_dev, uint64_t dJv_dev,
                             uint64_t vf_dev, uint64_t stream);
/* The same M, nle, Jc, dJv plus the task terms of the IKID QP (IKIDSolver_f6, QP_utils.py:666-675,684,690) for `count` states:
 *   Ag [count][6][nv]      data.Ag, centroidal momentum matrix about the CoM, world axes, linear rows then angular rows;
 *   dAgv [count][6]        data.dAg @ v: rate of the centroidal momentum at zero joint acceleration, gravity EXCLUDED;
 *   Jang [count][2][3][nv] angular rows of the LOCAL frame Jacobian of the two frames (frame_body[f], frame_place[f]: parent body
 *                          in [0, nb) and placement in it, R row-major then p), in the caller's order (the IKID QP: base, then torso);
 *   dJang [count][2][3]    angular part of those frames' LOCAL acceleration at zero joint acceleration (dJ v).
 * The LOCAL frame matches the sole Jacobians; which frame the reference uses for the base / torso rows (QP_utils.py:666-675) is
 * UNPINNED.  Host arrays (any output may be NULL) / device pointers + stream (asynchronous).  Not available for MPC_KIND_CENT. */
int32_t mpc_ikid_terms(mpc_solver_t *h, int32_t count, const double *x, const int32_t frame_body[2], const double frame_place[2][12], double *M,
                       double *nle, double *Jc, double *dJv, double *Ag, double *dAgv, double *Jang, double *dJang);
int32_t mpc_ikid_terms_device(mpc_solver_t *h, int32_t count, uint64_t x_dev, const int32_t frame_body[2], const double frame_place[2][12],
                              uint64_t M_dev, uint64_t nle_dev, uint64_t Jc_dev, uint64_t dJv_dev, uint64_t Ag_dev, uint64_t dAgv_dev,
                              uint64_t Jang_dev, uint64_t dJang_dev, uint64_t stream);
/* ---- Device-side gait / swing-foot reference generation (SURVEY 8f row f-4).  Replaces, per MPC tick and for the whole batch, the
 * Python bookkeeping of the reference loops: update_timings (talos_utils.py:350-373), footTrajectory.updateTrajectory
 * (talos_utils.py:187-327), the per-stage setReference / contact_poses writes and the stage entering the horizon
 * (fulldynamic_talos.py:444-510, kinodynamic_talos.py:362-409, centroidal_talos.py:354-384,459). */
typedef struct mpc_gait {
  int32_t T_ds, T_ss, cycles, half_cycle; /* contact schedule: T_ds DS, then `cycles` x (T_ss, T_ds, T_ss, T_ds), an extra (T_ss, T_ds) if half_cycle, then 2 T DS */
  int32_t keep_forward;                   /* 1: never zero the forward step (stairs, BASELINE configs[3]) */
  int32_t n_uref;                         /* rows of the control-reference table (kino / cent: `urefs`), 0 for full dynamics */
  double x_forward, y_forward, foot_yaw, y_gap, z_height, swing_apex; /* footTrajectory(...) arguments (full:350-361) */
  double lf0[12], rf0[12], com0[3];       /* initial sole placements and CoM */
  double f_half;                          /* m g / 2: contact-force reference of the full-dynamics stages */
  double w_lfrf;                          /* foot-placement cost weight (full: 2000, kino: 1e5) */
} mpc_gait_t;
/* Create the per-robot gait state: mirror [batch] (1 = first swing with the other foot), urefs [n_uref][MPC_MAXU] (may be NULL when n_uref = 0).
 * The tick counter starts at 0 with the feet at lf0 / rf0. */
int32_t mpc_gait_setup(mpc_solver_t *h, const mpc_gait_t *gait, const int32_t *mirror, const double *urefs);
/* One tick of the bookkeeping for every robot: from the measured sole placements lf / rf ([batch][12] host; NULL = the placements of the
 * soles at the state the next mpc_tick starts from, i.e. the model prediction xs[1], computed on the device; centroidal model: the placements last
 * tick's plan wanted at this tick, i.e. exact tracking) rewrite all T knots and the
 * terminal block of every instance on the device, then advance the tick counter.  Call it before mpc_tick(h, NULL, x_meas, ...). */
int32_t mpc_gait_tick(mpc_solver_t *h, const double *lf, const double *rf);
/* Test hook: the knots [batch][T] and terminal blocks [batch] the solver currently holds. */
int32_t mpc_get_knots(mpc_solver_t *h, mpc_knot_t *knots, mpc_term_t *terms);

uint64_t mpc_workspace_bytes(mpc_solver_t *h);
int32_t mpc_abi_sizeof(int32_t which); /* 0 robot, 1 config, 2 knot, 3 term, 4 info */
/* fp64 DFMA peak micro-benchmark (TFLOP/s) used as the roofline denominator (SURVEY 8d). */
double mpc_measure_fp64_peak(int32_t device);
/* Same for the fp64 tensor pipe (independent DMMA.8x8x4 chains); the roofline denominator is the larger of the two and cuBLAS DGEMM. */
double mpc_measure_fp64_peak_dmma(int32_t device);

#ifdef __cplusplus
}
#endif
#endif
