"""Batched mirror of the reference's whole-body inverse-dynamics QP class `IDSolver_ulim` (QP_utils.py:437-573; call site
kinodynamic_talos.py:408-445) on the CUDA QP solver (proxqp.BatchQP -> libmpcb200.so).  SURVEY 8f row f-3.

Same constructor arguments, same `solve(...)` return values (new accelerations, new contact forces, joint torques), with a leading
batch axis on every array.  The reference reads M, nle, the LOCAL contact Jacobians, dJ v and the frame velocities out of a
`pinocchio.Data`; here they are passed as arrays (`RBDTerms`, produced by whatever plays pinocchio's part: the fixture generator
in tests/, a user's own pinocchio, ...).  Both classes also have `solve_from_state`, which computes those terms on the device from the
measured states (the kernels of csrc/rbd_terms.cuh) and assembles the whole QP there.
"""
from dataclasses import dataclass

import numpy as np

from . import proxqp


@dataclass
class RBDTerms:
    """What IDSolver_ulim.computeMatrice reads from `data` (QP_utils.py:515-528), batch-major."""
    nle: np.ndarray  # [B][nv]            data.nle
    Jc: np.ndarray   # [B][6 nk][nv]      getFrameJacobian(..., LOCAL) of every contact frame, stacked
    dJv: np.ndarray  # [B][6 nk]          getFrameJacobianTimeVariation(..., LOCAL) @ v
    vf: np.ndarray   # [B][nk][6]         getFrameVelocity(...): linear, angular


class IDSolver_ulim:
    def __init__(self, model, weights, nk, mu, L, W, contact_ids, force_size, verbose=False, batch=1, device=0):
        if force_size != 6 or nk != 2 or model.nv != 28:
            raise NotImplementedError("the device assembly covers the reference's configuration: nv = 28, two 6-D contacts (kinodynamic_talos.py:408-417)")
        kd = 1  # QP_utils.py:441
        self.baum_Kd = np.diag([kd, kd, kd])
        self.nk, self.contact_ids, self.mu, self.L, self.W, self.force_size = nk, contact_ids, mu, L, W, force_size
        self.model, self.batch = model, batch
        nv = model.nv
        n, neq, nin = 2 * nv - 6 + force_size * nk, nv + force_size * nk, 9 * nk  # QP_utils.py:451-453
        self.n, self.neq, self.nin = n, neq, nin
        u = np.ones(nin) * 100000  # QP_utils.py:486
        g = np.zeros(n)
        H = np.zeros((n, n))
        H[:nv, :nv] = np.eye(nv) * weights[0]
        H[nv:nv + force_size * nk, nv:nv + force_size * nk] = np.eye(force_size * nk) * weights[1]
        qp = proxqp.dense.BatchQP(n, neq, nin, batch, False, dense_backend=proxqp.dense.DenseBackend.PrimalDualLDLT, device=device)
        qp.settings.eps_abs = 1e-3  # QP_utils.py:502-508
        qp.settings.eps_rel = 0
        qp.settings.primal_infeasibility_solving = True
        qp.settings.check_duality_gap = True
        qp.settings.verbose = verbose
        qp.settings.max_iter = 10
        qp.settings.max_iter_in = 10
        qp.init(H, g, np.zeros((neq, n)), np.zeros(neq), np.zeros((nin, n)), np.zeros(nin), u)
        self.qp = qp

    def gamma(self, rbd, cs):
        """dJ v + Kd v_lin + Kd v_ang on the linear rows of the active contacts (QP_utils.py:524-528, as written there)."""
        B = self.batch
        g = np.array(rbd.dJv, float).reshape(B, self.nk, 6).copy()
        vf = np.asarray(rbd.vf, float).reshape(B, self.nk, 6)
        g[:, :, :3] += vf[:, :, :3] @ self.baum_Kd.T + vf[:, :, 3:] @ self.baum_Kd.T
        return (g * np.asarray(cs).reshape(B, self.nk, 1)).reshape(B, 6 * self.nk)

    def computeMatrice(self, rbd, cs, v, a, forces, M):
        """A, b, C, l of QP_utils.py:530-552, assembled by a CUDA kernel straight into the solver's device buffers."""
        self.qp.assemble_id(M, rbd.nle, rbd.Jc, self.gamma(rbd, cs), a, forces, cs, self.mu, self.L, self.W)

    def solve(self, rbd, cs, v, a, forces, M):
        self.computeMatrice(rbd, cs, v, a, forces, M)
        self.qp.solve()
        nv, nf = self.model.nv, self.force_size * self.nk
        x = self.qp.results.x
        anew = np.asarray(a, float).reshape(self.batch, nv) + x[:, :nv]
        new_forces = np.asarray(forces, float).reshape(self.batch, nf) + x[:, nv:nv + nf]
        torque = x[:, nv + nf:]
        return anew, new_forces, torque

    def solve_from_state(self, solver, x_measured, cs, a, forces):
        """kinodynamic_talos.py:425-445 in one call for the whole batch: the pinocchio step (crba, nonLinearEffects, frame Jacobians and
        their time variation at the MEASURED states x_measured [batch][57]) runs on the device through `solver` (a batch.BatchSolver of
        the same robot), then the assembly and the QP."""
        self.qp.assemble_id_from_state(solver, x_measured, a, forces, cs, self.mu, self.L, self.W, float(self.baum_Kd[0, 0]))
        self.qp.solve()
        nv, nf = self.model.nv, self.force_size * self.nk
        x = self.qp.results.x
        return np.asarray(a, float).reshape(self.batch, nv) + x[:, :nv], np.asarray(forces, float).reshape(self.batch, nf) + x[:, nv:nv + nf], x[:, nv + nf:]


@dataclass
class RBDTermsIKID:
    """What IKIDSolver_f6.computeMatrice reads from `data` (QP_utils.py:666-675,684,690), batch-major."""
    nle: np.ndarray       # [B][nv]
    Jc: np.ndarray        # [B][12][nv]   LOCAL Jacobians of the left / right contact frames
    dJv: np.ndarray       # [B][12]       their time variation times v
    J_base: np.ndarray    # [B][3][nv]    angular rows of the base frame Jacobian (getFrameJacobian(...)[3:])
    dJv_base: np.ndarray  # [B][3]
    J_torso: np.ndarray   # [B][3][nv]
    dJv_torso: np.ndarray  # [B][3]
    Ag: np.ndarray        # [B][6][nv]    centroidal momentum matrix (data.Ag)
    dAgv: np.ndarray      # [B][6]        data.dAg @ v


class IKIDSolver_f6:
    """Batched mirror of QP_utils.py:584-768 (inverse kinematics + dynamics QP, 6-D contact wrenches, torque box constraints):
    the cost `H, g` is assembled on the host with batched numpy exactly as QP_utils.py:677-691 writes it, the constraint blocks by
    the same CUDA assembly kernel as IDSolver_ulim (they coincide with a = 0 and gamma = dJ v: QP_utils.py:693-721), the solve runs
    on the batched CUDA QP solver with box constraints.  `solve_from_state` builds the same QP, cost included, on the device from the
    measured states."""

    def __init__(self, model, weights, K_gains, nk, mu, L, W, contact_ids, base_id, torso_id, force_size, verbose=False, batch=1, device=0):
        if force_size != 6 or nk != 2 or model.nv != 28:
            raise NotImplementedError("reference configuration only: nv = 28, two 6-D contacts")
        self.K_gains, self.weights = K_gains, weights
        self.nk, self.contact_ids, self.base_id, self.torso_id = nk, contact_ids, base_id, torso_id
        self.mu, self.L, self.W, self.force_size, self.model, self.batch = mu, L, W, force_size, model, batch
        nv = model.nv
        n, neq, nin = 2 * nv - 6 + force_size * nk, nv + force_size * nk, 9 * nk
        self.n, self.neq, self.nin = n, neq, nin
        eff = np.asarray(model.effortLimit, float)[6:]
        self.l_box = -np.ones(n) * 100000  # QP_utils.py:612-615
        self.l_box[nv + force_size * nk:] = -eff
        self.u_box = np.ones(n) * 100000
        self.u_box[nv + force_size * nk:] = eff
        self.g = np.zeros((batch, n))
        self.H = np.zeros((batch, n, n))
        i = np.arange(nv, nv + force_size * nk)
        self.H[:, i, i] = weights[4]  # QP_utils.py:648
        qp = proxqp.dense.BatchQP(n, neq, nin, batch, True, dense_backend=proxqp.dense.DenseBackend.PrimalDualLDLT, device=device)
        qp.settings.eps_abs = 1e-3  # QP_utils.py:653-659
        qp.settings.eps_rel = 0.0
        qp.settings.primal_infeasibility_solving = True
        qp.settings.check_duality_gap = True
        qp.settings.verbose = verbose
        qp.settings.max_iter = 100
        qp.settings.max_iter_in = 100
        qp.init(self.H, self.g, np.zeros((neq, n)), np.zeros(neq), np.zeros((nin, n)), np.zeros(nin), np.ones(nin) * 100000, self.l_box, self.u_box)
        self.qp = qp

    def computeMatrice(self, rbd, cs, v, q_diff, dq_diff, LF_diff, dLF_diff, RF_diff, dRF_diff, base_diff, dbase_diff, torso_diff, dtorso_diff, forces, dH, M):
        B, nv, w, K = self.batch, self.model.nv, self.weights, self.K_gains
        arr = lambda a, *sh: np.broadcast_to(np.asarray(a, float), (B,) + sh)  # noqa: E731
        Jc = arr(rbd.Jc, 12, nv)
        JL, JR, Jb, Jt, Ag = Jc[:, :6], Jc[:, 6:], arr(rbd.J_base, 3, nv), arr(rbd.J_torso, 3, nv), arr(rbd.Ag, 6, nv)
        dJv = arr(rbd.dJv, 12)
        gram = lambda J: np.einsum("bki,bkj->bij", J, J)  # noqa: E731
        Hq = w[0] * np.eye(nv) + w[1] * (gram(JL) + gram(JR)) + w[2] * gram(Ag) + w[3] * (gram(Jb) + gram(Jt))  # QP_utils.py:677-682
        self.H[:, :nv, :nv] = Hq
        mv = lambda Kmat, d: np.einsum("ij,bj->bi", np.asarray(Kmat, float), d)  # noqa: E731
        jt = lambda r, J: np.einsum("bk,bki->bi", r, J)  # noqa: E731  (r' J)
        g = w[0] * (-mv(K[0][0], arr(q_diff, nv)) - mv(K[0][1], arr(dq_diff, nv)))  # QP_utils.py:684-691
        g = g + w[1] * jt(dJv[:, :6] - mv(K[1][0], arr(LF_diff, 6)) - mv(K[1][1], arr(dLF_diff, 6)), JL)
        g = g + w[1] * jt(dJv[:, 6:] - mv(K[1][0], arr(RF_diff, 6)) - mv(K[1][1], arr(dRF_diff, 6)), JR)
        g = g - w[2] * jt(arr(dH, 6) - arr(rbd.dAgv, 6), Ag)
        g = g + w[3] * jt(arr(rbd.dJv_base, 3) - mv(K[3][0], arr(base_diff, 3)) - mv(K[3][1], arr(dbase_diff, 3)), Jb)
        g = g + w[3] * jt(arr(rbd.dJv_torso, 3) - mv(K[3][0], arr(torso_diff, 3)) - mv(K[3][1], arr(dtorso_diff, 3)), Jt)
        self.g[:, :nv] = g
        csb = np.asarray(cs).reshape(-1, self.nk)
        gamma = dJv * np.repeat(np.broadcast_to(csb, (B, self.nk)), 6, axis=1)
        # A, b, C, l of QP_utils.py:693-738 = the IDSolver_ulim blocks with a = 0, gamma = dJ v
        self.qp.assemble_id(M, rbd.nle, Jc, gamma, np.zeros((B, nv)), forces, cs, self.mu, self.L, self.W)

    def solve(self, rbd, cs, v, q_diff, dq_diff, LF_diff, dLF_diff, RF_diff, dRF_diff, base_diff, dbase_diff, torso_diff, dtorso_diff, forces, dH, M):
        self.computeMatrice(rbd, cs, v, q_diff, dq_diff, LF_diff, dLF_diff, RF_diff, dRF_diff, base_diff, dbase_diff, torso_diff, dtorso_diff, forces, dH, M)
        self.qp.update(H=self.H, g=self.g, l_box=self.l_box, u_box=self.u_box, update_preconditioner=False)
        self.qp.solve()
        nv, nf = self.model.nv, self.force_size * self.nk
        x = self.qp.results.x
        anew = x[:, :nv]
        new_forces = np.asarray(forces, float).reshape(self.batch, nf) + x[:, nv:nv + nf]
        torque = x[:, nv + nf:]
        return anew, new_forces, torque

    def _frames(self):
        """(parent body, placement 12) of the base and torso frames named by base_id / torso_id."""
        return [(self.model.frames[i].parentJoint - 1, self.model.frames[i].placement.to12()) for i in (self.base_id, self.torso_id)]

    def _packed_gains(self):
        """K_gains packed as the device assembly reads them: Kp_q, Kd_q (nv x nv), Kp_f, Kd_f (6 x 6), Kp_b, Kd_b (3 x 3), row-major."""
        K, nv = self.K_gains, self.model.nv
        return np.concatenate([np.broadcast_to(np.asarray(k, float), (m, m)).ravel() for k, m in
                               ((K[0][0], nv), (K[0][1], nv), (K[1][0], 6), (K[1][1], 6), (K[3][0], 3), (K[3][1], 3))])

    def solve_from_state(self, solver, x_measured, cs, q_diff, dq_diff, LF_diff, dLF_diff, RF_diff, dRF_diff, base_diff, dbase_diff, torso_diff,
                         dtorso_diff, forces, dH):
        """centroidal_talos.py:435-445 in one call for the whole batch: the pinocchio step (crba, nonLinearEffects, the contact, base and
        torso frame Jacobians with their time variation, the centroidal momentum matrix and dAg v at the MEASURED states x_measured
        [batch][57]) runs on the device through `solver` (a kinodynamic or full-dynamics batch.BatchSolver of the same robot), then the
        whole cost and constraint assembly and the QP.  Only x, the task errors, forces and cs are uploaded per robot.  Returns what
        `solve` returns.  The base / torso rows use the LOCAL frame."""
        B = self.batch
        f = lambda a, per: np.broadcast_to(np.asarray(a, float).reshape(-1, per), (B, per))  # noqa: E731
        nv = self.model.nv
        task = np.concatenate([f(q_diff, nv), f(dq_diff, nv), f(LF_diff, 6), f(dLF_diff, 6), f(RF_diff, 6), f(dRF_diff, 6), f(base_diff, 3), f(dbase_diff, 3),
                               f(torso_diff, 3), f(dtorso_diff, 3), f(dH, 6)], axis=1)
        self.qp.assemble_ikid_from_state(solver, x_measured, task, forces, cs, self.weights, self._packed_gains(), self._frames(), self.mu, self.L, self.W)
        self.qp.solve()
        nf = self.force_size * self.nk
        x = self.qp.results.x
        return x[:, :nv], np.asarray(forces, float).reshape(B, nf) + x[:, nv:nv + nf], x[:, nv + nf:]
