"""ctypes driver of the host warp emulator build of the generic QP solve (tests/emu/emu_qp.cpp): the kernel header's
qp_env runs with 32 lock-step fibers per env, so tsidb_qp_solve can be compared with the oracle on a box without a GPU.
Also the emulated QP export with the actuation map (TA, ta0).  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from emu_problem import EmuProblem
from emu_py import EMU_DIR, SRC_DIR, TickArgs
from tsid_control_b200._capi import TsidbProblemOut, TsidbQpOut


def build_emu_qp() -> str:
    so = os.path.join(EMU_DIR, "libtsidb_emu_qp.so")
    srcs = [os.path.join(EMU_DIR, "emu_qp.cpp"), os.path.join(EMU_DIR, "emu_cuda.h")] + [
        os.path.join(SRC_DIR, f) for f in ("tsidb_kernels.cuh", "tsidb_const.h", "tsidb_host_const.h")] + [
        os.path.join(SRC_DIR, "..", "..", "include", "tsidb.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-Wno-enum-compare", "-o", so, os.path.join(EMU_DIR, "emu_qp.cpp")], check=True)
    return so


QP_PARTS = ("H", "g", "CE", "ce0", "CI", "ci0", "TA", "ta0")


def emu_qp_solve(problem: dict, max_iter: int, na: int = 0) -> dict:
    """problem: padded [N, ...] float64 arrays H, g, CE, ce0, CI, ci0 (TA, ta0 optional) and sizes [N,3] int32, the strides
    taken from the shapes -> x, status, iters, active, lambda, lambda_eq (and tau with TA/ta0), NaN/garbage-filled
    before the call so that anything left unwritten shows."""
    lib = C.CDLL(build_emu_qp())
    lib.emu_qp_solve.argtypes = [C.c_int] * 6 + [C.POINTER(TsidbProblemOut), C.POINTER(TsidbQpOut)]
    N, nm = problem["g"].shape
    neqm = problem["ce0"].shape[1] if "ce0" in problem else 0
    ninm = problem["ci0"].shape[1] if "ci0" in problem else 0
    p = {k: np.ascontiguousarray(problem[k], dtype=np.float64) for k in QP_PARTS if k in problem}
    p["sizes"] = np.ascontiguousarray(problem["sizes"], dtype=np.int32)
    out = {"x": np.full((N, nm), np.nan), "status": np.full(N, -7, np.int32), "iters": np.full(N, -7, np.int32),
           "active": np.full((N, nm), -7, np.int32), "lambda": np.full((N, nm), np.nan), "lambda_eq": np.full((N, neqm), np.nan)}
    if "TA" in p:
        na = p["TA"].shape[1]
        out["tau"] = np.full((N, na), np.nan)
    po = TsidbProblemOut(**{k: a.ctypes.data for k, a in p.items()})
    qo = TsidbQpOut(**{k: a.ctypes.data for k, a in out.items()})
    rc = lib.emu_qp_solve(N, nm, neqm, ninm, na, int(max_iter), C.byref(po), C.byref(qo))
    assert rc == 0, rc
    return out


class EmuProblemTA(EmuProblem):
    """The emulated export (tests/emu_problem.py) with the actuation map TA [N,na,n_max], ta0 [N,na] as well."""

    def problem_ta(self, q, v, mask, refs: dict) -> dict:
        N = q.shape[0]
        na, nv, cc = self.na, self.nv, self.cc
        nx, nin = nv + 24, 2 * (34 + (na if cc.use_torque_bounds else 0) + (nv if cc.use_joint_bounds else 0))
        out = {"H": np.full((N, nx, nx), np.nan), "g": np.full((N, nx), np.nan), "CE": np.full((N, 18, nx), np.nan),
               "ce0": np.full((N, 18), np.nan), "CI": np.full((N, nin, nx), np.nan), "ci0": np.full((N, nin), np.nan),
               "sizes": np.full((N, 3), -1, np.int32), "TA": np.full((N, na, nx), np.nan), "ta0": np.full((N, na), np.nan)}
        keep = [np.ascontiguousarray(q, dtype=np.float64), np.ascontiguousarray(v, dtype=np.float64),
                np.ascontiguousarray(mask, dtype=np.uint8)]
        arrs = {k: np.ascontiguousarray(refs[k], dtype=np.float64) for k in self.REF_KEYS}
        a = TickArgs()
        a.n_envs, a.layout, a.slot = N, 0, 0
        a.q, a.v, a.mask = (x.ctypes.data for x in keep)
        a.r_com, a.r_posture = arrs["com"].ctypes.data, arrs["posture"].ctypes.data
        a.r_foot[0], a.r_foot[1] = arrs["foot_lf"].ctypes.data, arrs["foot_rf"].ctypes.data
        a.r_contact[0], a.r_contact[1] = arrs["contact_lf"].ctypes.data, arrs["contact_rf"].ctypes.data
        po = TsidbProblemOut(**{k: x.ctypes.data for k, x in out.items()})
        assert self.lib.emu_problem(C.byref(a), C.byref(po)) == 0
        return out
