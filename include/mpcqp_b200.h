/*
 * mpcqp_b200.h — C-ABI of the batched dense QP solver of libmpcb200.so (SURVEY 8f row f-3).
 *
 * Boundary it replaces: `proxsuite.proxqp.dense.QP(n, n_eq, n_in[, box])` + `.init / .update / .solve / .results`
 * as driven by the whole-body QPs of the reference (QP_utils.py:34-46,75-83 IKSolver; :220-233,274-287 IDSolver_velocity;
 * :355-368,412-426 IDSolver; :500-513,557-573 IDSolver_ulim; :651-664,743-760 IKIDSolver_f6; :816-830 IKIDSolver_f3; call sites
 * kinodynamic_talos.py:438-445, centroidal_talos.py:435-445 — ten solves per MPC tick at 1 kHz).  proxsuite is a pip
 * dependency that is absent here (SURVEY 8c); the algorithm restated is the published ProxQP (Bambade, El-Kazdadi, Taylor,
 * Carpentier, RSS 2022): proximal augmented Lagrangian, semismooth Newton inner loop with an exact piecewise-quadratic
 * linesearch, BCL outer loop.  One QP of the batch:
 *
 *     min_x  1/2 x'Hx + g'x   s.t.   A x = b,   l <= C x <= u,   l_box <= x <= u_box (optional)
 *
 * All arithmetic fp64, all matrices row-major, batch-major arrays: H [batch][n][n], g [batch][n], A [batch][n_eq][n],
 * b [batch][n_eq], C [batch][n_in][n], l / u [batch][n_in], l_box / u_box [batch][n], x [batch][n], y [batch][n_eq],
 * z [batch][n_in (+ n with box)].  A batch stride of 0 doubles shares one array between all QPs of the batch (the
 * reference's constant H, u, l_box, u_box).  Bounds with |value| >= 1e20 are infinite.
 */
#ifndef MPCQP_B200_H
#define MPCQP_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPC_QP_MAXN 64   /* primal variables        (reference: 62 = 2 nv - 6 + 12, QP_utils.py:451) */
#define MPC_QP_MAXEQ 64  /* equality rows           (reference: 40 = nv + 12,       QP_utils.py:452) */
#define MPC_QP_MAXIN 32  /* general inequality rows (reference: 18 = 9 nk,          QP_utils.py:453) */

/* proxsuite.proxqp Settings fields the reference sets (QP_utils.py:502-508) + the algorithm constants they leave at default. */
typedef struct mpc_qp_settings {
  double eps_abs;          /* 1e-3 (QP_utils.py:502) */
  double eps_rel;          /* 0 */
  double rho;              /* primal proximal weight, 1e-6 */
  double mu_eq;            /* initial equality penalty, 1e-3 */
  double mu_in;            /* initial inequality penalty, 1e-1 */
  double alpha_bcl;        /* 0.1 */
  double beta_bcl;         /* 0.9 */
  double mu_update_factor; /* 0.1 */
  double mu_min_eq;        /* 1e-4 (proxsuite: 1e-9; the condensed primal Newton form has a dual-residual floor ~ 1e-11 / mu_min) */
  double mu_min_in;        /* 1e-4 (proxsuite: 1e-8) */
  int32_t max_iter;        /* outer iterations (10 / 100, QP_utils.py:507,658) */
  int32_t max_iter_in;     /* Newton iterations per outer iteration (10 / 100) */
  int32_t check_duality_gap; /* QP_utils.py:505 */
  int32_t warm_start;      /* 0: start from x = y = z = 0; 1: start from the x / y / z passed in */
} mpc_qp_settings_t;

typedef struct mpc_qp_info {
  int32_t status;   /* 0 solved, 1 max_iter reached (result returned, as proxsuite does), 2 non-finite / factorisation failed */
  int32_t iter;     /* outer (BCL) iterations */
  int32_t iter_in;  /* Newton steps in total */
  int32_t mu_updates;
  double pri_res;   /* max(|Ax - b|, [Cx - u]+ + [Cx - l]-, box) in the infinity norm */
  double dua_res;   /* |Hx + g + A'y + C'z (+ z_box)| */
  double duality_gap;
  double objective;
} mpc_qp_info_t;

typedef struct mpc_qp mpc_qp_t;

/* One handle = one (n, n_eq, n_in, box) shape and a maximum batch; owns its device workspace.  NULL + mpc_qp_last_error on failure
 * (no CUDA device, dimensions above MPC_QP_MAX*).  No CPU fallback exists. */
mpc_qp_t *mpc_qp_create(int32_t n, int32_t n_eq, int32_t n_in, int32_t box, int32_t max_batch, int32_t device);
void mpc_qp_destroy(mpc_qp_t *h);
const char *mpc_qp_last_error(void);
void mpc_qp_default_settings(mpc_qp_settings_t *s);

/* qp.init / qp.update (QP_utils.py:509,557-565): upload the data of `batch` QPs from HOST arrays.  NULL = keep what the handle
 * holds (update(H=None, ...)); stride arguments are in doubles per QP, 0 = shared. */
int32_t mpc_qp_update(mpc_qp_t *h, int32_t batch, const double *H, int64_t sH, const double *g, int64_t sg, const double *A, int64_t sA,
                      const double *b, int64_t sb, const double *C, int64_t sC, const double *l, int64_t sl, const double *u, int64_t su,
                      const double *l_box, int64_t slb, const double *u_box, int64_t sub);
/* qp.solve() + qp.results.{x, y, z, info} (QP_utils.py:567-573) to HOST arrays; x / y / z are also the warm start when
 * settings->warm_start.  info may be NULL. */
int32_t mpc_qp_solve(mpc_qp_t *h, const mpc_qp_settings_t *settings, double *x, double *y, double *z, mpc_qp_info_t *info);
/* Same on DEVICE buffers the caller owns (uint64 = device pointer, 0 = the handle's own copy from mpc_qp_update for the data;
 * strides as above), asynchronous on `stream`: the device-resident number of bench.py. */
int32_t mpc_qp_solve_device(mpc_qp_t *h, int32_t batch, const mpc_qp_settings_t *settings, uint64_t H, int64_t sH, uint64_t g, int64_t sg,
                            uint64_t A, int64_t sA, uint64_t b, int64_t sb, uint64_t C, int64_t sC, uint64_t l, int64_t sl, uint64_t u,
                            int64_t su, uint64_t l_box, int64_t slb, uint64_t u_box, int64_t sub, uint64_t x, uint64_t y, uint64_t z,
                            uint64_t info, uint64_t stream);
/* Device time of the last solve kernel (ms, CUDA events on the launch stream; synchronises). */
double mpc_qp_last_device_ms(mpc_qp_t *h);
int32_t mpc_qp_abi_sizeof(int32_t which); /* 0 settings, 1 info */
/* Cycle counters per phase of the solve kernel, summed over the QPs since the last call (all zero unless built with
 * -DMPC_QP_PHASE_TIMING): load, residuals, AL gradient, Newton matrix, Cholesky, substitutions, linesearch, multiplier update. */
int32_t mpc_qp_debug_phases(mpc_qp_t *h, double *out8);

/* Whole-body inverse-dynamics QP of the reference assembled on the device (IDSolver_ulim.computeMatrice, QP_utils.py:514-552;
 * n = 2 nv - 6 + 6 nk, n_eq = nv + 6 nk, n_in = 9 nk with nv = 28, nk = 2): from HOST arrays per instance M [nv][nv], nle [nv],
 * Jc [6 nk][nv] (LOCAL contact Jacobians), gamma [6 nk] (dJ v + the Baumgarte velocity term), a [nv], forces [6 nk],
 * cs [nk] (int32 contact flags), fills the handle's A, b, C, l; H, g, u stay as uploaded.  mu / L / W: friction, half length, half width. */
int32_t mpc_qp_assemble_id(mpc_qp_t *h, int32_t batch, const double *M, const double *nle, const double *Jc, const double *gamma,
                           const double *a, const double *forces, const int32_t *cs, double mu, double L, double W);

/* The same assembly fed from MEASURED STATES instead of pinocchio results (kinodynamic_talos.py:425-445 in one call): x [batch][57]
 * host -> rigid-body terms on the device (mpc_rbd_terms_device of `solver`, a libmpcb200 solver handle created for the same robot) ->
 * gamma = (dJ v + kd (v_lin + v_ang) on the linear rows) on the active contacts (QP_utils.py:524-528) -> A, b, C, l.  Uploads 100 doubles
 * per robot instead of 1201. */
struct mpc_solver;
int32_t mpc_qp_assemble_id_from_state(mpc_qp_t *h, struct mpc_solver *solver, int32_t batch, const double *x, const double *a, const double *forces,
                                      const int32_t *cs, double mu, double L, double W, double kd);

/* The whole IKID QP of the reference (IKIDSolver_f6.computeMatrice, QP_utils.py:666-738; n 62, n_eq 40, n_in 18, box constraints)
 * assembled on the device from MEASURED STATES: x [batch][57] host -> M, nle, Jc, dJv and the task terms (mpc_ikid_terms_device of
 * `solver`, a libmpcb200 solver handle created for the same robot; frame_body / frame_place name the base and torso frames, whose
 * LOCAL angular Jacobians are used — the reference's choice of frame there is unpinned) -> the cost
 *   H[:28,:28] = w0 I + w1 (JL'JL + JR'JR) + w2 Ag'Ag + w3 (Jb'Jb + Jt'Jt),  H[28:40,28:40] = w4 I,  zeros elsewhere,
 *   g[:28] from the PD task errors, the gains, dJv, dAgv and dH (QP_utils.py:684-691),
 * and A, b, C, l as mpc_qp_assemble_id with a = 0 and gamma = dJv on the active contacts (no Baumgarte term).
 * task [batch][98]: q_diff 28, dq_diff 28, LF 6, dLF 6, RF 6, dRF 6, base 3, dbase 3, torso 3, dtorso 3, dH 6 (the argument order of
 * IKIDSolver_f6.solve); forces [batch][12]; cs [batch][2]; weights [5]; gains [1658], shared: Kp_q, Kd_q (28 x 28), Kp_f, Kd_f (6 x 6),
 * Kp_b, Kd_b (3 x 3), row-major general matrices.  Afterwards H, g, A, b, C, l hold one array per QP; u, l_box, u_box stay as uploaded.
 * Uploads 167 doubles + 8 bytes per robot (+ the gains once per call) instead of the 5,106 doubles of the host-side cost.
 * The first call allocates a scratch for the task terms and gains, freed by mpc_qp_destroy. */
int32_t mpc_qp_assemble_ikid_from_state(mpc_qp_t *h, struct mpc_solver *solver, int32_t batch, const double *x, const double *task,
                                        const double *forces, const int32_t *cs, const double weights[5], const double *gains,
                                        const int32_t frame_body[2], const double frame_place[2][12], double mu, double L, double W);

#ifdef __cplusplus
}
#endif
#endif
