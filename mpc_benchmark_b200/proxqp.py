"""Drop-in for the slice of `proxsuite.proxqp` the reference's whole-body QPs use (SURVEY 8f row f-3), on the batched CUDA QP
solver of libmpcb200.so (include/mpcqp_b200.h, csrc/qp.cuh).

Reference usage (QP_utils.py:34-46, 220-233, 355-368, 500-513, 651-664, 816-830 and the `update` / `solve` / `results.x` calls
next to them):

    import proxsuite
    qp = proxsuite.proxqp.dense.QP(n, neq, nin[, box], dense_backend=proxsuite.proxqp.dense.DenseBackend.PrimalDualLDLT)
    qp.settings.eps_abs = 1e-3; qp.settings.max_iter = 10; ...
    qp.init(H, g, A, b, C, l, u[, l_box, u_box]);  qp.update(A=..., b=..., update_preconditioner=False);  qp.solve();  qp.results.x

`from mpc_benchmark_b200 import proxqp as _p; proxsuite = _p.proxsuite` (or `import mpc_benchmark_b200.proxqp as proxsuite` and
`proxsuite.proxqp.dense.QP`) keeps that code unchanged.  `dense.BatchQP` is the same object over a leading batch axis: one CUDA
launch solves every QP of the batch, one CTA each.  There is no CPU fallback: without the library / a GPU `solve()` raises.
The algorithm is the published ProxQP restated (oracle/qp.hpp is normative); parity with proxsuite itself is unpinned
(it is not installable here), see DESIGN.md.
"""
import ctypes as C
import types

import numpy as np

from . import _abi, _native


class Settings:
    """proxsuite.proxqp.Settings fields the reference sets, plus the algorithm constants it leaves at their defaults."""

    def __init__(self):
        self.eps_abs = 1e-5
        self.eps_rel = 0.0
        self.default_rho = 1e-6
        self.default_mu_eq = 1e-3
        self.default_mu_in = 1e-1
        self.alpha_bcl = 0.1
        self.beta_bcl = 0.9
        self.mu_update_factor = 0.1
        self.mu_min_eq = 1e-4  # proxsuite: 1e-9 / 1e-8 (primal-dual form); the condensed primal form evaluates multiplier
        self.mu_min_in = 1e-4  # estimates as residual / mu, so its dual-residual floor is ~1e-11 / mu_min (DESIGN.md, QP section)
        self.max_iter = 10000
        self.max_iter_in = 1500
        self.check_duality_gap = False
        self.primal_infeasibility_solving = False  # accepted and recorded only (closest-feasible solves are not restated)
        self.verbose = False
        self.compute_timings = False
        self.initial_guess = "NO_INITIAL_GUESS"  # or "WARM_START"

    def to_c(self, warm):
        s = _abi.QPSettings()
        s.eps_abs, s.eps_rel, s.rho, s.mu_eq, s.mu_in = self.eps_abs, self.eps_rel, self.default_rho, self.default_mu_eq, self.default_mu_in
        s.alpha_bcl, s.beta_bcl, s.mu_update_factor = self.alpha_bcl, self.beta_bcl, self.mu_update_factor
        s.mu_min_eq, s.mu_min_in = self.mu_min_eq, self.mu_min_in
        s.max_iter, s.max_iter_in = int(self.max_iter), int(self.max_iter_in)
        s.check_duality_gap, s.warm_start = int(bool(self.check_duality_gap)), int(bool(warm))
        return s


class Info:
    def __init__(self):
        self.status = None
        self.iter = self.iter_ext = self.mu_updates = 0
        self.pri_res = self.dua_res = self.duality_gap = self.objValue = 0.0
        self.run_time = 0.0  # device time of the solve kernel, microseconds (proxsuite reports microseconds)


class Results:
    def __init__(self):
        self.x = self.y = self.z = None
        self.info = Info()


class QPSolverOutput:
    PROXQP_SOLVED, PROXQP_MAX_ITER_REACHED, PROXQP_NOT_RUN = 0, 1, 2


class DenseBackend:
    Automatic, PrimalDualLDLT, PrimalLDLT = 0, 1, 2


class BatchQP:
    """`batch` QPs of one shape solved together.  Arrays carry a leading batch axis; an array without it is shared."""

    def __init__(self, n, n_eq, n_in, batch=1, box_constraints=False, dense_backend=DenseBackend.PrimalDualLDLT, device=0):
        self.n, self.n_eq, self.n_in, self.batch, self.box = int(n), int(n_eq), int(n_in), int(batch), bool(box_constraints)
        self.nz = self.n_in + (self.n if self.box else 0)
        self.settings = Settings()
        self.results = Results()
        self.dense_backend = dense_backend  # recorded only: the kernel factors the condensed primal Newton matrix
        self._h = None
        self._device = device
        self._initialised = False

    # -- native handle
    def _handle(self):
        if self._h is None:
            L = _native.lib()
            h = L.mpc_qp_create(self.n, self.n_eq, self.n_in, int(self.box), self.batch, self._device)
            if not h:
                raise _native.NativeError(f"mpc_qp_create failed: {L.mpc_qp_last_error().decode()}")
            self._h = h
        return self._h

    def close(self):
        if self._h is not None:
            _native.lib().mpc_qp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _arg(self, a, per, name):
        """(pointer, stride) of one data array; None keeps what the handle holds."""
        if a is None or per == 0:
            return None, 0, None
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.size == per:
            return _native.ptr(a), 0, a
        if a.size != per * self.batch:
            raise ValueError(f"{name}: expected {per} or {self.batch} x {per} values, got {a.size}")
        return _native.ptr(a), per, a

    def _upload(self, H, g, A, b, C_, l, u, l_box, u_box):
        n, ne, ni = self.n, self.n_eq, self.n_in
        spec = [(H, n * n, "H"), (g, n, "g"), (A, ne * n, "A"), (b, ne, "b"), (C_, ni * n, "C"), (l, ni, "l"), (u, ni, "u"),
                (l_box if self.box else None, n, "l_box"), (u_box if self.box else None, n, "u_box")]
        args, keep = [], []
        for a, per, name in spec:
            p, s, arr = self._arg(a, per, name)
            args += [p, s]
            keep.append(arr)
        L = _native.lib()
        if L.mpc_qp_update(self._handle(), self.batch, *args) != 0:
            raise _native.NativeError(f"mpc_qp_update failed: {L.mpc_qp_last_error().decode()}")

    def init(self, H=None, g=None, A=None, b=None, C=None, l=None, u=None, l_box=None, u_box=None, *_, **__):  # noqa: E741
        if H is None or g is None:
            raise ValueError("init needs H and g")
        if self.n_eq and (A is None or b is None):
            raise ValueError("init needs A and b for n_eq > 0")
        if self.n_in and (C is None or l is None or u is None):
            raise ValueError("init needs C, l and u for n_in > 0")
        if self.box and (l_box is None or u_box is None):
            raise ValueError("init needs l_box and u_box with box constraints")
        self._upload(H, g, A, b, C, l, u, l_box, u_box)
        self._initialised = True

    def update(self, H=None, g=None, A=None, b=None, C=None, l=None, u=None, l_box=None, u_box=None, update_preconditioner=False, **__):  # noqa: E741
        if not self._initialised:
            raise RuntimeError("update before init")
        self._upload(H, g, A, b, C, l, u, l_box, u_box)

    def solve(self, x=None, y=None, z=None):
        if not self._initialised:
            raise RuntimeError("solve before init")
        warm = x is not None or self.settings.initial_guess == "WARM_START" and self.results.x is not None
        B = self.batch
        X = np.zeros((B, self.n)) if not warm else np.ascontiguousarray(x if x is not None else self.results.x, float).reshape(B, self.n).copy()
        Y = np.zeros((B, max(self.n_eq, 1))) if not warm else np.ascontiguousarray(y if y is not None else self.results.y, float).reshape(B, -1).copy()
        Z = np.zeros((B, max(self.nz, 1))) if not warm else np.ascontiguousarray(z if z is not None else self.results.z, float).reshape(B, -1).copy()
        info = (_abi.QPInfo * B)()
        st = self.settings.to_c(warm)
        L = _native.lib()
        if L.mpc_qp_solve(self._handle(), C.byref(st), _native.ptr(X), _native.ptr(Y), _native.ptr(Z), info) != 0:
            raise _native.NativeError(f"mpc_qp_solve failed: {L.mpc_qp_last_error().decode()}")
        self._store(X, Y[:, :self.n_eq], Z[:, :self.nz], info)
        return self.results

    def _store(self, X, Y, Z, info):
        r = self.results
        r.x, r.y, r.z = X, Y, Z
        r.info.status = np.array([i.status for i in info])
        r.info.iter_ext = np.array([i.iter for i in info])
        r.info.iter = np.array([i.iter_in for i in info])
        r.info.mu_updates = np.array([i.mu_updates for i in info])
        r.info.pri_res = np.array([i.pri_res for i in info])
        r.info.dua_res = np.array([i.dua_res for i in info])
        r.info.duality_gap = np.array([i.duality_gap for i in info])
        r.info.objValue = np.array([i.objective for i in info])
        r.info.run_time = 1e3 * _native.lib().mpc_qp_last_device_ms(self._handle())

    # -- whole-body inverse-dynamics assembly on the device (IDSolver_ulim.computeMatrice, QP_utils.py:514-552)
    def assemble_id(self, M, nle, Jc, gamma, a, forces, cs, mu, L, W):
        f = lambda v, per: _native.ptr(np.ascontiguousarray(np.broadcast_to(np.asarray(v, float).reshape(-1, per), (self.batch, per))))  # noqa: E731
        cs = np.ascontiguousarray(np.broadcast_to(np.asarray(cs).reshape(-1, 2), (self.batch, 2)), dtype=np.int32)
        lib = _native.lib()
        rc = lib.mpc_qp_assemble_id(self._handle(), self.batch, f(M, 784), f(nle, 28), f(Jc, 336), f(gamma, 12), f(a, 28), f(forces, 12),
                                    cs.ctypes.data_as(C.POINTER(C.c_int32)), float(mu), float(L), float(W))
        if rc != 0:
            raise _native.NativeError(f"mpc_qp_assemble_id failed: {lib.mpc_qp_last_error().decode()}")


    def assemble_id_from_state(self, solver, x, a, forces, cs, mu, L, W, kd):
        """Same blocks from MEASURED STATES x [batch][57]: the rigid-body terms are computed on the device by `solver` (a
        batch.BatchSolver created for the same robot), nothing but x, a, forces, cs is uploaded."""
        B = self.batch
        f = lambda v, per: np.ascontiguousarray(np.broadcast_to(np.asarray(v, float).reshape(-1, per), (B, per)))  # noqa: E731
        xs, aa, ff = f(x, 57), f(a, 28), f(forces, 12)
        cs = np.ascontiguousarray(np.broadcast_to(np.asarray(cs).reshape(-1, 2), (B, 2)), dtype=np.int32)
        lib = _native.lib()
        rc = lib.mpc_qp_assemble_id_from_state(self._handle(), solver._h, B, _native.ptr(xs), _native.ptr(aa), _native.ptr(ff),
                                               cs.ctypes.data_as(C.POINTER(C.c_int32)), float(mu), float(L), float(W), float(kd))
        if rc != 0:
            raise _native.NativeError(f"mpc_qp_assemble_id_from_state failed: {lib.mpc_qp_last_error().decode()}")

    def assemble_ikid_from_state(self, solver, x, task, forces, cs, weights, gains, frames, mu, L, W):
        """The whole IKID QP (IKIDSolver_f6.computeMatrice, QP_utils.py:666-738) from MEASURED STATES x [batch][57]: rigid-body and task
        terms on the device by `solver` (a batch.BatchSolver of the same robot), then H, g, A, b, C, l.  task [batch][98] packs the PD
        errors in the argument order of IKIDSolver_f6.solve; gains [1658] packs Kp_q, Kd_q, Kp_f, Kd_f, Kp_b, Kd_b row-major;
        frames = ((body, placement 12), (body, placement 12)) of the base and torso frames."""
        B = self.batch
        f = lambda v, per: np.ascontiguousarray(np.broadcast_to(np.asarray(v, float).reshape(-1, per), (B, per)))  # noqa: E731
        xs, tk, ff = f(x, 57), f(task, 98), f(forces, 12)
        cs = np.ascontiguousarray(np.broadcast_to(np.asarray(cs).reshape(-1, 2), (B, 2)), dtype=np.int32)
        wt, gn = np.ascontiguousarray(weights, float).reshape(5), np.ascontiguousarray(gains, float).reshape(1658)
        fb = np.ascontiguousarray([fr[0] for fr in frames], dtype=np.int32)
        fp = np.ascontiguousarray([fr[1] for fr in frames], dtype=np.float64).reshape(2, 12)
        i32p = C.POINTER(C.c_int32)
        lib = _native.lib()
        rc = lib.mpc_qp_assemble_ikid_from_state(self._handle(), solver._h, B, _native.ptr(xs), _native.ptr(tk), _native.ptr(ff), cs.ctypes.data_as(i32p),
                                                 _native.ptr(wt), _native.ptr(gn), fb.ctypes.data_as(i32p), _native.ptr(fp), float(mu), float(L), float(W))
        if rc != 0:
            raise _native.NativeError(f"mpc_qp_assemble_ikid_from_state failed: {lib.mpc_qp_last_error().decode()}")


class QP(BatchQP):
    """proxsuite.proxqp.dense.QP(n, n_eq, n_in[, box_constraints], dense_backend=...): one QP (a batch of one)."""

    def __init__(self, n, n_eq, n_in, box_constraints=False, dense_backend=DenseBackend.PrimalDualLDLT, **kw):
        super().__init__(n, n_eq, n_in, 1, box_constraints, dense_backend, **kw)

    def _store(self, X, Y, Z, info):
        super()._store(X, Y, Z, info)
        r = self.results
        r.x, r.y, r.z = X[0], Y[0], Z[0]
        i = r.info
        for k in ("status", "iter_ext", "iter", "mu_updates", "pri_res", "dua_res", "duality_gap", "objValue"):
            setattr(i, k, getattr(i, k)[0].item())


# namespace mirrors: proxsuite.proxqp.dense.QP / .DenseBackend / proxsuite.proxqp.QPSolverOutput
dense = types.SimpleNamespace(QP=QP, BatchQP=BatchQP, DenseBackend=DenseBackend)
proxqp = types.SimpleNamespace(dense=dense, Settings=Settings, Results=Results, QPSolverOutput=QPSolverOutput)
proxsuite = types.SimpleNamespace(proxqp=proxqp)
