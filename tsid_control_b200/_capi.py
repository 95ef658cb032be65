"""ctypes view of include/tsidb.h plus the conf/model marshalling.

The product path has no CPU fallback: :func:`load_library` raises if
``libtsidb.so`` has not been built (``python -c 'import __graft_entry__ as g; g.build()'``)
and every compute entry point fails without a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Optional

import numpy as np

from .model_compiler import CompiledModel

MAX_BODIES = 24
MAX_NA = 23
MAX_NV = 29

c_double_p = C.POINTER(C.c_double)


class TsidbModel(C.Structure):
    _fields_ = [
        ("nb", C.c_int32),
        ("parent", C.c_int32 * MAX_BODIES),
        ("jR", (C.c_double * 9) * MAX_BODIES),
        ("jp", (C.c_double * 3) * MAX_BODIES),
        ("mass", C.c_double * MAX_BODIES),
        ("com", (C.c_double * 3) * MAX_BODIES),
        ("inertia", (C.c_double * 9) * MAX_BODIES),
        ("foot_body", C.c_int32 * 2),
        ("fR", (C.c_double * 9) * 2),
        ("fp", (C.c_double * 3) * 2),
        ("gravity", C.c_double * 3),
    ]


class TsidbConf(C.Structure):
    _fields_ = [
        ("contact_points", (C.c_double * 4) * 3),
        ("contact_normal", C.c_double * 3),
        ("mu", C.c_double),
        ("fmin", C.c_double),
        ("fmax", C.c_double),
        ("kp_contact", C.c_double * 6),
        ("kd_contact", C.c_double * 6),
        ("w_force_reg", C.c_double),
        ("force_reg_weights", C.c_double * 6),
        ("w_foot", C.c_double),
        ("kp_foot", C.c_double * 6),
        ("kd_foot", C.c_double * 6),
        ("w_com", C.c_double),
        ("kp_com", C.c_double * 3),
        ("kd_com", C.c_double * 3),
        ("w_posture", C.c_double),
        ("kp_posture", C.c_double * MAX_NA),
        ("kd_posture", C.c_double * MAX_NA),
        ("w_am", C.c_double),
        ("kp_am", C.c_double * 3),
        ("use_torque_bounds", C.c_int32),
        ("tau_min", C.c_double * MAX_NA),
        ("tau_max", C.c_double * MAX_NA),
        ("use_joint_bounds", C.c_int32),
        ("v_min", C.c_double * MAX_NA),
        ("v_max", C.c_double * MAX_NA),
        ("joint_bounds_dt", C.c_double),
        ("hessian_reg", C.c_double),
        ("max_iter", C.c_int32),
        ("pad_", C.c_int32),
    ]


class TsidbRefs(C.Structure):
    _fields_ = [
        ("com", C.c_void_p),
        ("foot_lf", C.c_void_p),
        ("foot_rf", C.c_void_p),
        ("contact_lf", C.c_void_p),
        ("contact_rf", C.c_void_p),
        ("posture", C.c_void_p),
    ]


class TsidbGaitConf(C.Structure):
    _fields_ = [("dt", C.c_double), ("step_duration", C.c_double), ("step_length", C.c_double),
                ("step_height", C.c_double), ("com_height", C.c_double)]


class TsidbAuxOut(C.Structure):
    _fields_ = [
        ("com", C.c_void_p),
        ("foot_lf", C.c_void_p),
        ("foot_rf", C.c_void_p),
        ("wrench", C.c_void_p),
        ("lambda_", C.c_void_p),
        ("lambda_row", C.c_void_p),
    ]


class TsidbProblemOut(C.Structure):
    # TA, ta0 were appended to the C struct; ctypes leaves unnamed fields NULL, so older callers are unchanged
    _fields_ = [(k, C.c_void_p) for k in ("H", "g", "CE", "ce0", "CI", "ci0", "sizes", "TA", "ta0")]


class TsidbQpOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("x", "status", "iters", "active", "lambda", "lambda_eq", "tau")]


class TsidbRefsOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("com", "foot_lf", "foot_rf", "contact_lf", "contact_rf", "posture")]


def _fill(arr, values) -> None:
    v = np.asarray(values, dtype=np.float64).ravel()
    for i, x in enumerate(v):
        arr[i] = float(x)


def model_to_c(m: CompiledModel, lf_frame: str, rf_frame: str) -> TsidbModel:
    """CompiledModel + the two sole-frame names of the conf -> tsidb_model."""
    cm = TsidbModel()
    cm.nb = m.nb
    for b in range(m.nb):
        cm.parent[b] = m.parent[b]
        _fill(cm.jR[b], m.jR[b])
        _fill(cm.jp[b], m.jp[b])
        cm.mass[b] = float(m.mass[b])
        _fill(cm.com[b], m.com[b])
        _fill(cm.inertia[b], m.inertia[b])
    for s, name in enumerate((lf_frame, rf_frame)):
        if name not in m.frames:
            raise KeyError(f"frame {name!r} not in model {m.name!r}; has {sorted(m.frames)}")
        fr = m.frames[name]
        cm.foot_body[s] = fr["body"]
        _fill(cm.fR[s], fr["R"])
        _fill(cm.fp[s], fr["p"])
    _fill(cm.gravity, [0.0, 0.0, -9.81])
    return cm


def conf_to_c(conf, m: CompiledModel, legacy: bool = False) -> TsidbConf:
    """Freeze the task constants exactly as the reference constructors compute them.

    WalkController: ref:ctrl/WalkController.py:55-184 with ref:ctrl/conf.py:21-72.
    Biped:          ref:legacy/biped.py:31-130 with ref:legacy/op3_conf.py:4-50.
    """
    na = m.na
    cc = TsidbConf()
    # contact_points (ref:ctrl/WalkController.py:55-57)
    pts = np.ones((3, 4)) * (-conf.lz)
    pts[0, :] = [-conf.lxn, -conf.lxn, conf.lxp, conf.lxp]
    pts[1, :] = [-conf.lyn, conf.lyp, -conf.lyn, conf.lyp]
    for r in range(3):
        for c in range(4):
            cc.contact_points[r][c] = float(pts[r, c])
    _fill(cc.contact_normal, conf.contactNormal)
    cc.mu, cc.fmin, cc.fmax = float(conf.mu), float(conf.fMin), float(conf.fMax)
    _fill(cc.kp_contact, conf.kp_contact * np.ones(6))
    _fill(cc.kd_contact, 2.0 * np.sqrt(conf.kp_contact) * np.ones(6))
    cc.w_force_reg = float(conf.w_forceRef)
    _fill(cc.force_reg_weights, [1.0, 1.0, 1e-3, 2.0, 2.0, 2.0])  # [UPSTREAM Contact6d::init]
    cc.w_foot = float(conf.w_foot)
    _fill(cc.kp_foot, conf.kp_foot * np.ones(6))
    _fill(cc.kd_foot, 2.0 * np.sqrt(conf.kp_foot) * np.ones(6))
    cc.w_com = float(conf.w_com)
    _fill(cc.kp_com, conf.kp_com * np.ones(3))
    _fill(cc.kd_com, 2.0 * np.sqrt(conf.kp_com) * np.ones(3))
    cc.w_posture = float(conf.w_posture)
    gv = np.asarray(conf.gain_vector, dtype=np.float64)
    if gv.shape != (na,):
        raise ValueError(f"gain_vector has {gv.shape[0]} entries, model has {na} actuated joints")
    mask = np.asarray(conf.masks_posture, dtype=np.float64)
    if not np.all(mask == 1.0):
        raise NotImplementedError("masks_posture other than all-ones (both reference confs use ones)")
    _fill(cc.kp_posture, conf.kp_posture * gv)
    _fill(cc.kd_posture, 2.0 * np.sqrt(conf.kp_posture * gv))
    if legacy and getattr(conf, "w_am", 0.0) > 0.0:
        cc.w_am = float(conf.w_am)
        _fill(cc.kp_am, conf.kp_am * np.array([1.0, 1.0, 0.0]))  # ref:legacy/biped.py:83
    else:
        cc.w_am = 0.0
    # actuation bounds (ref:ctrl/WalkController.py:168-176)
    cc.use_torque_bounds = 1 if conf.w_torque_bounds > 0.0 else 0
    tau_max = conf.tau_max_scaling * m.effort
    _fill(cc.tau_max, tau_max)
    _fill(cc.tau_min, -tau_max)
    # joint (velocity) bounds (ref:ctrl/WalkController.py:178-184)
    cc.use_joint_bounds = 1 if conf.w_joint_bounds > 0.0 else 0
    v_max = conf.v_max_scaling * m.velocity
    _fill(cc.v_max, v_max)
    _fill(cc.v_min, -v_max)
    cc.joint_bounds_dt = 2.0 * float(conf.dt)  # [UPSTREAM TaskJointBounds ctor: m_dt(2*dt)]
    cc.hessian_reg = 1e-8  # [UPSTREAM SolverHQuadProgFast DEFAULT_HESSIAN_REGULARIZATION]
    cc.max_iter = 1000
    return cc


# ---------------------------------------------------------------------------------
_LIB: Optional[C.CDLL] = None
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libtsidb.so")


class TsidbError(RuntimeError):
    pass


def load_library() -> C.CDLL:
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise TsidbError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "There is no CPU fallback for the TSID tick."
        )
    lib = C.CDLL(LIB_PATH)
    vp, ip, dp = C.c_void_p, C.c_int, c_double_p
    lib.tsidb_create.argtypes = [C.POINTER(TsidbModel), C.POINTER(TsidbConf), ip, ip, C.POINTER(vp)]
    lib.tsidb_create.restype = ip
    lib.tsidb_destroy.argtypes = [vp]
    lib.tsidb_destroy.restype = None
    lib.tsidb_last_error.argtypes = []
    lib.tsidb_last_error.restype = C.c_char_p
    lib.tsidb_sizes.argtypes = [vp, C.POINTER(ip), C.POINTER(ip), C.POINTER(ip)]
    lib.tsidb_sizes.restype = ip
    lib.tsidb_set_default_refs.argtypes = [vp, dp, dp, dp, dp, dp, dp]
    lib.tsidb_set_default_refs.restype = ip
    lib.tsidb_compute.argtypes = [vp, ip, ip, vp, vp, vp, C.POINTER(TsidbRefs), vp, vp, vp, vp, vp, vp,
                                  C.POINTER(TsidbAuxOut), vp]
    lib.tsidb_compute.restype = ip
    lib.tsidb_compute_host.argtypes = [vp, ip, vp, vp, vp, C.POINTER(TsidbRefs), vp, vp, vp, vp, vp, vp]
    lib.tsidb_compute_host.restype = ip
    lib.tsidb_compute_host_devrefs.argtypes = [vp, ip, vp, vp, vp, C.POINTER(TsidbRefs), vp, vp, vp, vp, vp, vp]
    lib.tsidb_compute_host_devrefs.restype = ip
    lib.tsidb_integrate.argtypes = [vp, ip, ip, vp, vp, vp, C.c_double, vp]
    lib.tsidb_integrate.restype = ip
    lib.tsidb_kinematics.argtypes = [vp, ip, ip, vp, vp, C.POINTER(TsidbAuxOut), vp]
    lib.tsidb_kinematics.restype = ip
    lib.tsidb_ci_row.argtypes = [vp, ip, ip, ip]
    lib.tsidb_ci_row.restype = ip
    lib.tsidb_fp64_peak.argtypes = [ip, dp]
    lib.tsidb_fp64_peak.restype = ip
    lib.tsidb_launch_count.argtypes = [vp]
    lib.tsidb_launch_count.restype = C.c_int64
    lib.tsidb_set_timing.argtypes = [vp, ip]
    lib.tsidb_set_timing.restype = ip
    lib.tsidb_set_sched_hint.argtypes = [vp, ip]
    lib.tsidb_set_sched_hint.restype = ip
    lib.tsidb_last_tick_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.tsidb_last_tick_ms.restype = ip
    lib.tsidb_gait_reset.argtypes = [vp, ip, C.POINTER(TsidbGaitConf), vp, vp, vp]
    lib.tsidb_gait_reset.restype = ip
    lib.tsidb_foot_trajectory.argtypes = [vp, ip, C.c_double, C.c_double, vp, vp, C.c_double, C.c_double, vp, vp, vp]
    lib.tsidb_foot_trajectory.restype = ip
    lib.tsidb_footstep_plan.argtypes = [vp, ip, vp, vp, ip, vp, C.c_double, C.c_double, vp, vp, ip, vp]
    lib.tsidb_footstep_plan.restype = ip
    lib.tsidb_gait_set_plan.argtypes = [vp, ip, vp, vp, ip, C.c_double, vp]
    lib.tsidb_gait_set_plan.restype = ip
    lib.tsidb_gait_state.argtypes = [vp, C.POINTER(TsidbRefs), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.tsidb_gait_state.restype = ip
    lib.tsidb_gait_step.argtypes = [vp, ip, vp, vp, vp, vp]
    lib.tsidb_gait_step.restype = ip
    lib.tsidb_rollout.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp, vp, vp, ip, vp]
    lib.tsidb_rollout.restype = ip
    lib.tsidb_diagnostics.argtypes = [vp, ip, C.POINTER(TsidbAuxOut), vp, C.c_double, vp, vp, vp, vp]
    lib.tsidb_diagnostics.restype = ip
    lib.tsidb_debug_terms.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp]
    lib.tsidb_debug_terms.restype = ip
    lib.tsidb_problem_sizes.argtypes = [vp, C.POINTER(ip), C.POINTER(ip), C.POINTER(ip)]
    lib.tsidb_problem_sizes.restype = ip
    lib.tsidb_problem_data.argtypes = [vp, ip, ip, vp, vp, vp, C.POINTER(TsidbRefs), C.POINTER(TsidbProblemOut), vp]
    lib.tsidb_problem_data.restype = ip
    lib.tsidb_qp_solve.argtypes = [vp, ip, ip, ip, ip, C.POINTER(TsidbProblemOut), C.POINTER(TsidbQpOut), vp]
    lib.tsidb_qp_solve.restype = ip
    lib.tsidb_qp_grad.argtypes = [vp, ip, ip, ip, ip, C.POINTER(TsidbProblemOut), C.POINTER(TsidbQpOut), C.POINTER(TsidbQpOut),
                                  C.POINTER(TsidbProblemOut), vp, vp]
    lib.tsidb_qp_grad.restype = ip
    lib.tsidb_refs_grad.argtypes = [vp, ip, ip, vp, vp, vp, C.POINTER(TsidbRefs), ip, ip, vp, vp, C.POINTER(TsidbRefsOut), vp]
    lib.tsidb_refs_grad.restype = ip
    lib.tsidb_state_grad.argtypes = [vp, ip, ip, vp, vp, vp, C.POINTER(TsidbRefs), ip, ip, ip, C.POINTER(TsidbProblemOut), vp,
                                     vp, vp]
    lib.tsidb_state_grad.restype = ip
    _LIB = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load_library().tsidb_last_error()
        raise TsidbError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")


EXPORTED_SYMBOLS = [
    "tsidb_create", "tsidb_destroy", "tsidb_last_error", "tsidb_sizes", "tsidb_set_default_refs",
    "tsidb_compute", "tsidb_compute_host", "tsidb_compute_host_devrefs", "tsidb_integrate", "tsidb_kinematics", "tsidb_ci_row",
    "tsidb_fp64_peak", "tsidb_launch_count", "tsidb_set_timing", "tsidb_set_sched_hint", "tsidb_last_tick_ms",
    "tsidb_gait_reset", "tsidb_gait_state", "tsidb_gait_step", "tsidb_rollout", "tsidb_diagnostics",
    "tsidb_foot_trajectory", "tsidb_footstep_plan", "tsidb_gait_set_plan", "tsidb_debug_terms",
    "tsidb_problem_sizes", "tsidb_problem_data", "tsidb_qp_solve", "tsidb_qp_grad",
    "tsidb_refs_grad", "tsidb_state_grad",
]
