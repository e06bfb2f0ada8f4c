"""BatchSolver — batched ProxDDP over flat problem descriptors (the layer under the aligator-compatible shim).

One BatchSolver = one `mpc_solver_t` handle = one batch of independent MPC instances on one GPU
(SURVEY 8e: instances are the data-parallel axis).  Mirrors SolverProxDDP.setup / run / results
(fulldynamic_talos.py:379-405) for a whole batch at once.
"""
import ctypes as C

import numpy as np

from . import _abi, _native
from .qp_utils import RBDTermsIKID


class BatchResults:
    def __init__(self, xs, us, K, vs, lams, info):
        self.xs, self.us, self.K, self.vs, self.lams, self.info = xs, us, K, vs, lams, info

    @property
    def num_iters(self):
        return np.array([i.num_iters for i in self.info])

    @property
    def conv(self):
        return np.array([bool(i.conv) for i in self.info])

    @property
    def prim_infeas(self):
        return np.array([i.prim_infeas for i in self.info])

    @property
    def dual_infeas(self):
        return np.array([i.dual_infeas for i in self.info])

    @property
    def traj_cost(self):
        return np.array([i.traj_cost for i in self.info])

    @property
    def ls_evals(self):
        return np.array([i.ls_evals for i in self.info])

    @property
    def alpha(self):
        return np.array([i.alpha for i in self.info])


class BatchSolver:
    def __init__(self, robot, cfg, batch, device=0, **_unused):
        self.robot, self.cfg, self.batch, self.device = robot, cfg, int(batch), int(device)
        self.nx, self.n, self.m, self.nc = _abi.DIMS[cfg.kind]
        self.T = cfg.T
        L = _native.lib()
        self._h = L.mpc_create(C.byref(robot), C.byref(cfg), self.batch, self.device)
        if not self._h:
            raise _native.NativeError("mpc_create failed: " + _native.last_error())

    def close(self):
        if getattr(self, "_h", None):
            _native.lib().mpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # solver.setup(problem)
    def setup(self, knots, terms, x0):
        x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(self.batch, self.nx)
        assert len(knots) == self.batch * self.T and len(terms) == self.batch
        _native.check(_native.lib().mpc_setup(self._h, C.cast(knots, C.c_void_p), C.cast(terms, C.c_void_p), _native.ptr(x0)), "mpc_setup")

    def update_knots(self, knots, first, count):
        assert len(knots) == self.batch * count
        _native.check(_native.lib().mpc_update_knots(self._h, C.cast(knots, C.c_void_p), first, count), "mpc_update_knots")

    def update_terms(self, terms):
        _native.check(_native.lib().mpc_update_terms(self._h, C.cast(terms, C.c_void_p)), "mpc_update_terms")

    def cycle(self, last_knots):
        assert len(last_knots) == self.batch
        _native.check(_native.lib().mpc_cycle(self._h, C.cast(last_knots, C.c_void_p)), "mpc_cycle")

    def reconfigure(self, robot, cfg):
        self.robot, self.cfg = robot, cfg
        _native.check(_native.lib().mpc_reconfigure(self._h, C.byref(robot), C.byref(cfg)), "mpc_reconfigure")

    def set_instance_models(self, robots=None, cfgs=None):
        """Per-instance robot parameters and cost constants: instance i is solved with robots[i] / cfgs[i] (sequences of length batch of
        _abi.Robot / _abi.Config; None = the shared robot / config for every instance; both None = back to the shared model).  Kind,
        horizon, dt, solver constants and the tree topology stay those of the handle (`mpc_set_instance_models`, include/mpcb200.h)."""
        B = self.batch
        arrs = []
        for seq, typ in ((robots, _abi.Robot), (cfgs, _abi.Config)):
            if seq is None:
                arrs.append(None)
                continue
            if len(seq) != B:
                raise ValueError(f"set_instance_models: expected {B} {typ.__name__} blocks (one per instance), got {len(seq)}")
            arrs.append((typ * B)(*seq))
        _native.check(_native.lib().mpc_set_instance_models(self._h, *[None if a is None else C.cast(a, C.c_void_p) for a in arrs]),
                      "mpc_set_instance_models")

    def shift_multipliers(self, n=1):
        _native.check(_native.lib().mpc_shift_multipliers(self._h, int(n)), "mpc_shift_multipliers")

    def reset_multipliers(self, stream=0):
        """The solver-state part of a per-tick `solver.setup` (full:539): multipliers back to zero, problem kept."""
        _native.check(_native.lib().mpc_reset_multipliers(self._h, int(stream)), "mpc_reset_multipliers")

    def set_x0(self, x0):
        x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(self.batch, self.nx)
        _native.check(_native.lib().mpc_set_x0(self._h, _native.ptr(x0)), "mpc_set_x0")

    # solver.run(problem, xs_init, us_init) with host arrays
    def run(self, xs, us, max_iters=None, fetch=True, gains=True):
        xs = np.ascontiguousarray(xs, dtype=np.float64).reshape(self.batch, self.T + 1, self.nx)
        us = np.ascontiguousarray(us, dtype=np.float64).reshape(self.batch, self.T, self.m)
        mi = self.cfg.max_iters if max_iters is None else int(max_iters)
        _native.check(_native.lib().mpc_run(self._h, _native.ptr(xs), _native.ptr(us), mi), "mpc_run")
        return self.results(gains=gains) if fetch else None

    def run_pipelined(self, xs, us, xs_out, us_out, K0_out=None, max_iters=None, parts=2, info=False):
        """solver.run + read-back of xs / us / K0 as one pipelined call on host buffers (pinned buffers give the overlap): the upload of
        the next sub-batch and the download of the previous one run beside the solve of the current one (`mpc_run_pipelined`)."""
        xs = np.ascontiguousarray(xs, dtype=np.float64).reshape(self.batch, self.T + 1, self.nx)
        us = np.ascontiguousarray(us, dtype=np.float64).reshape(self.batch, self.T, self.m)
        for a in (xs_out, us_out, K0_out):
            assert a is None or (a.dtype == np.float64 and a.flags["C_CONTIGUOUS"])
        mi = self.cfg.max_iters if max_iters is None else int(max_iters)
        inf = (_abi.Info * self.batch)() if info else None
        _native.check(_native.lib().mpc_run_pipelined(self._h, _native.ptr(xs), _native.ptr(us), mi, int(parts), _native.ptr(xs_out), _native.ptr(us_out),
                                                      _native.ptr(K0_out), C.cast(inf, C.c_void_p) if info else None), "mpc_run_pipelined")
        return inf

    def tick(self, last_knots=None, x_meas=None, keep_multipliers=False, max_iters=1):
        """One closed-loop MPC tick on the device: rotate the horizon, shift the warm start, new x0, solve (SURVEY 8f f-2)."""
        if last_knots is not None:
            assert len(last_knots) == self.batch
        xm = None if x_meas is None else np.ascontiguousarray(x_meas, dtype=np.float64).reshape(self.batch, self.nx)
        _native.check(_native.lib().mpc_tick(self._h, C.cast(last_knots, C.c_void_p) if last_knots is not None else None, _native.ptr(xm),
                                             int(bool(keep_multipliers)), int(max_iters)), "mpc_tick")

    # same with trajectories already in HBM (torch tensors or raw device pointers)
    def run_device(self, xs_ptr, us_ptr, max_iters=None, stream=0):
        mi = self.cfg.max_iters if max_iters is None else int(max_iters)
        _native.check(_native.lib().mpc_run_device(self._h, int(xs_ptr), int(us_ptr), mi, int(stream)), "mpc_run_device")

    def results(self, gains=True, multipliers=True):
        B, T = self.batch, self.T
        xs = np.empty((B, T + 1, self.nx))
        us = np.empty((B, T, self.m))
        K = np.empty((B, T, self.m, self.n)) if gains else None
        vs = np.empty((B, T + 1, self.nc)) if multipliers else None
        lams = np.empty((B, T + 1, self.n)) if multipliers else None
        info = (_abi.Info * B)()
        _native.check(_native.lib().mpc_get_results(self._h, _native.ptr(xs), _native.ptr(us), _native.ptr(K), _native.ptr(vs), _native.ptr(lams),
                                                    C.cast(info, C.c_void_p)), "mpc_get_results")
        return BatchResults(xs, us, K, vs, lams, info)

    def export_results_device(self, xs_ptr=0, us_ptr=0, K0_ptr=0, info_ptr=0, stream=0):
        """Pack xs / us / K0 / per-instance summary into caller-owned device buffers (raw pointers) for a gather over NVLink."""
        _native.check(_native.lib().mpc_export_results_device(self._h, int(xs_ptr), int(us_ptr), int(K0_ptr), int(info_ptr), int(stream)),
                      "mpc_export_results_device")

    def result_ptrs(self):
        p = [C.c_uint64(0) for _ in range(4)]
        _native.check(_native.lib().mpc_result_ptrs(self._h, *[C.byref(x) for x in p]), "mpc_result_ptrs")
        return tuple(x.value for x in p)

    def stage_data(self, k=0):
        nd = 9 if self.cfg.kind == _abi.KIND_CENT else 56
        xdot = np.empty((self.batch, nd))
        force = np.empty((self.batch, 12))
        _native.check(_native.lib().mpc_get_stage_data(self._h, k, _native.ptr(xdot), _native.ptr(force)), "mpc_get_stage_data")
        return xdot, force

    def set_tail_warmstart(self, phase_matched):
        """Control warm start of the knot `tick` appends: False = the previous knot's (the reference scripts' us[1:] + [us[-1]]), True = the control of the
        nearest knot of the horizon with the same contact phase (what the one-iteration full-dynamics loop needs to walk, DESIGN section 7)."""
        _native.check(_native.lib().mpc_set_tail_warmstart(self._h, int(bool(phase_matched))), "mpc_set_tail_warmstart")

    # -- device-side gait / swing-foot references (SURVEY 8f row f-4; mirrors gait.GaitPlan)
    def gait_setup(self, gait, mirror=None, urefs=None):
        """gait: _abi.Gait (see gait.device_gait); mirror [batch] bools; urefs [n][34] control references of the schedule (kino / cent)."""
        B = self.batch
        mir = np.ascontiguousarray(np.zeros(B) if mirror is None else mirror, dtype=np.int32)
        ur = None
        if urefs is not None:
            ur = np.zeros((len(urefs), _abi.MAXU))
            ur[:, :np.asarray(urefs).shape[1]] = urefs
            gait.n_uref = len(urefs)
        _native.check(_native.lib().mpc_gait_setup(self._h, C.byref(gait), mir.ctypes.data_as(C.POINTER(C.c_int32)), _native.ptr(ur)), "mpc_gait_setup")

    def gait_tick(self, lf=None, rf=None):
        """One tick of the reference's per-tick bookkeeping for the whole batch on the device: all T knots and the terminal block of every
        robot are rewritten from the measured sole placements lf / rf [batch][12] (None: soles at the model prediction xs[1])."""
        f = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64).reshape(self.batch, 12)  # noqa: E731
        l, r = f(lf), f(rf)
        _native.check(_native.lib().mpc_gait_tick(self._h, _native.ptr(l), _native.ptr(r)), "mpc_gait_tick")

    def knots(self):
        """The per-knot parameter blocks [batch * T] and terminal blocks [batch] the solver currently holds (test hook)."""
        T = self.cfg.T
        ks, ts = (_abi.Knot * (self.batch * T))(), (_abi.Term * self.batch)()
        _native.check(_native.lib().mpc_get_knots(self._h, C.cast(ks, C.c_void_p), C.cast(ts, C.c_void_p)), "mpc_get_knots")
        return ks, ts

    def rbd_terms(self, x):
        """Rigid-body terms of the whole-body QPs for the states x [count][nx] (what kinodynamic_talos.py:425-431 takes from pinocchio):
        dict(M, nle, Jc, dJv, vf).  With per-instance models set, state i uses instance i's robot and count must equal the batch."""
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 57)
        B = x.shape[0]
        o = dict(M=np.zeros((B, 28, 28)), nle=np.zeros((B, 28)), Jc=np.zeros((B, 12, 28)), dJv=np.zeros((B, 12)), vf=np.zeros((B, 2, 6)))
        _native.check(_native.lib().mpc_rbd_terms(self._h, B, _native.ptr(x), *[_native.ptr(o[k]) for k in ("M", "nle", "Jc", "dJv", "vf")]), "mpc_rbd_terms")
        return o

    def ikid_terms(self, x, frames):
        """Rigid-body terms and task terms of the IKID QP (IKIDSolver_f6, QP_utils.py:666-675) for the states x [count][nx]:
        (M, qp_utils.RBDTermsIKID).  frames = ((body, placement 12), (body, placement 12)) of the base and torso frames, whose LOCAL
        angular Jacobians and dJ v are returned.  With per-instance models set, state i uses instance i's robot and count must equal the batch."""
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 57)
        B = x.shape[0]
        fb = np.ascontiguousarray([f[0] for f in frames], dtype=np.int32)
        fp = np.ascontiguousarray([f[1] for f in frames], dtype=np.float64).reshape(2, 12)
        o = dict(M=np.zeros((B, 28, 28)), nle=np.zeros((B, 28)), Jc=np.zeros((B, 12, 28)), dJv=np.zeros((B, 12)), Ag=np.zeros((B, 6, 28)),
                 dAgv=np.zeros((B, 6)), Jang=np.zeros((B, 2, 3, 28)), dJang=np.zeros((B, 2, 3)))
        _native.check(_native.lib().mpc_ikid_terms(self._h, B, _native.ptr(x), fb.ctypes.data_as(C.POINTER(C.c_int32)), _native.ptr(fp),
                                                   *[_native.ptr(o[k]) for k in ("M", "nle", "Jc", "dJv", "Ag", "dAgv", "Jang", "dJang")]), "mpc_ikid_terms")
        return o["M"], RBDTermsIKID(nle=o["nle"], Jc=o["Jc"], dJv=o["dJv"], J_base=o["Jang"][:, 0], dJv_base=o["dJang"][:, 0], J_torso=o["Jang"][:, 1],
                                    dJv_torso=o["dJang"][:, 1], Ag=o["Ag"], dAgv=o["dAgv"])

    def feedback(self, k=0):
        """results.controlFeedbacks()[k] for every instance: [batch, nu, ndx]."""
        K = np.empty((self.batch, self.m, self.n))
        _native.check(_native.lib().mpc_get_feedback(self._h, k, _native.ptr(K)), "mpc_get_feedback")
        return K

    def kernel_ms(self):
        L = _native.lib()
        names = ["eval_deriv", "riccati", "eval_trial", "bookkeeping"]
        return {n: (L.mpc_last_kernel_ms(self._h, i), L.mpc_last_kernel_launches(self._h, i)) for i, n in enumerate(names)}

    def debug_lq(self, xs, us, inst=0):
        B, T, n, nz, nc = self.batch, self.T, self.n, self.n + self.m, self.nc
        xs = np.ascontiguousarray(xs, dtype=np.float64).reshape(B, T + 1, self.nx)
        us = np.ascontiguousarray(us, dtype=np.float64).reshape(B, T, self.m)
        o = dict(AB=np.empty((T, n, nz)), H=np.empty((T + 1, nz, nz)), g=np.empty((T + 1, nz)), gap=np.empty((T, n)), h=np.empty((T + 1, nc)),
                 scal=np.empty((T + 1, 8)))
        _native.check(_native.lib().mpc_debug_lq(self._h, _native.ptr(xs), _native.ptr(us), inst, _native.ptr(o["AB"]), _native.ptr(o["H"]),
                                                 _native.ptr(o["g"]), _native.ptr(o["gap"]), _native.ptr(o["h"]), _native.ptr(o["scal"])), "mpc_debug_lq")
        return o

    @property
    def last_launches(self):
        return _native.lib().mpc_last_launches(self._h)

    @property
    def last_device_ms(self):
        return _native.lib().mpc_last_device_ms(self._h)

    @property
    def workspace_bytes(self):
        return _native.lib().mpc_workspace_bytes(self._h)
