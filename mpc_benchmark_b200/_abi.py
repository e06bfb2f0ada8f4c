"""ctypes mirrors of the plain structs in include/mpcb200.h (the C-ABI boundary, SURVEY 8b).

The reference crosses Python -> C++ through eigenpy/Boost.Python (fulldynamic_talos.py:8-25);
here the boundary is a flat C ABI so that any FFI can bind it.  Field order and sizes must match
include/mpcb200.h exactly; tests/test_abi.py checks sizeof() against the library.
"""
import ctypes as C

KIND_CENT, KIND_KINO, KIND_FULL = 0, 1, 2
NB, NV, NQ, NJ, MAXU, MAXC = 23, 28, 29, 22, 34, 78
d = C.c_double
i32 = C.c_int32


class Robot(C.Structure):
    _fields_ = [
        ("nb", i32),
        ("parent", i32 * NB),
        ("jplace", (d * 12) * NB),
        ("axis", (d * 3) * NB),
        ("mass", d * NB),
        ("com", (d * 3) * NB),
        ("inertia", (d * 9) * NB),
        ("foot_body", i32 * 2),
        ("pad_", i32),
        ("foot_place", (d * 12) * 2),
        ("q_lo", d * NJ),
        ("q_hi", d * NJ),
        ("tau_max", d * NJ),
        ("gravity", d * 3),
    ]


class Config(C.Structure):
    _fields_ = [
        ("kind", i32),
        ("T", i32),
        ("dt", d),
        ("x_ref", d * (NQ + NV)),
        ("wx", d * (2 * NV)),
        ("wu", d * MAXU),
        ("w_cent", d * 6),
        ("w_centder", d * 6),
        ("w_force", d * 6),
        ("wx_term", d * (2 * NV)),
        ("w_cent_term", d * 6),
        ("w_foot_term", d * 6),
        ("mu_fric", d),
        ("foot_L", d),
        ("foot_W", d),
        ("kp", d * 6),
        ("kd", d * 6),
        ("contact_place", (d * 12) * 2),
        ("mu_contact", d),
        ("mass", d),
        ("w_linmom", d * 3),
        ("w_angmom", d * 3),
        ("w_linacc", d * 3),
        ("w_angacc", d * 3),
        ("w_com", d * 3),
        ("com_ref", d * 3),
        ("tol", d),
        ("mu_init", d),
        ("max_iters", i32),
        ("force_initial_condition", i32),
        ("rollout", i32),
        ("lq_legs", i32),
    ]


class Knot(C.Structure):
    _fields_ = [
        ("cs", d * 2),
        ("fcost", d * 2),
        ("w_lf", d * 6),
        ("w_rf", d * 6),
        ("lf_ref", d * 12),
        ("rf_ref", d * 12),
        ("f_ref", d * 12),
        ("u_ref", d * MAXU),
        ("cpos", d * 6),
    ]


class Term(C.Structure):
    _fields_ = [
        ("lf_ref", d * 12),
        ("rf_ref", d * 12),
        ("com_ref", d * 3),
        ("has_com_cstr", d),
    ]


class Info(C.Structure):
    _fields_ = [
        ("prim_infeas", d),
        ("dual_infeas", d),
        ("traj_cost", d),
        ("merit", d),
        ("mu", d),
        ("alpha", d),
        ("num_iters", i32),
        ("al_iters", i32),
        ("conv", i32),
        ("status", i32),
        ("ls_evals", i32),
        ("pad_", i32),
    ]


KNOT_DOUBLES = C.sizeof(Knot) // 8
TERM_DOUBLES = C.sizeof(Term) // 8

DIMS = {  # kind -> (nx, ndx, nu, ncmax)
    KIND_CENT: (9, 9, 12, 34),
    KIND_KINO: (57, 56, 34, 68),
    KIND_FULL: (57, 56, 22, 78),
}


# ---- include/mpcqp_b200.h (batched dense QP, SURVEY 8f row f-3)
class QPSettings(C.Structure):
    _fields_ = [
        ("eps_abs", d), ("eps_rel", d), ("rho", d), ("mu_eq", d), ("mu_in", d), ("alpha_bcl", d), ("beta_bcl", d),
        ("mu_update_factor", d), ("mu_min_eq", d), ("mu_min_in", d),
        ("max_iter", i32), ("max_iter_in", i32), ("check_duality_gap", i32), ("warm_start", i32),
    ]


class QPInfo(C.Structure):
    _fields_ = [
        ("status", i32), ("iter", i32), ("iter_in", i32), ("mu_updates", i32),
        ("pri_res", d), ("dua_res", d), ("duality_gap", d), ("objective", d),
    ]


# ---- device-side gait generator (include/mpcb200.h mpc_gait_t, SURVEY 8f row f-4)
class Gait(C.Structure):
    _fields_ = [
        ("T_ds", i32), ("T_ss", i32), ("cycles", i32), ("half_cycle", i32), ("keep_forward", i32), ("n_uref", i32),
        ("x_forward", d), ("y_forward", d), ("foot_yaw", d), ("y_gap", d), ("z_height", d), ("swing_apex", d),
        ("lf0", d * 12), ("rf0", d * 12), ("com0", d * 3), ("f_half", d), ("w_lfrf", d),
    ]
