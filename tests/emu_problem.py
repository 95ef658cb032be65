"""ctypes driver of the host warp emulator build of the QP export (tests/emu/emu_problem.cpp): the kernel header's
dynamics_env and problem_env run with 32 lock-step fibers per env, so the export can be compared with the oracle on a
box without a GPU.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from emu_py import EMU_DIR, SRC_DIR, TickArgs
from tsid_control_b200._capi import TsidbConf, TsidbModel, TsidbProblemOut


def build_emu_problem() -> str:
    so = os.path.join(EMU_DIR, "libtsidb_emu_problem.so")
    srcs = [os.path.join(EMU_DIR, "emu_problem.cpp"), os.path.join(EMU_DIR, "emu_cuda.h")] + [
        os.path.join(SRC_DIR, f) for f in ("tsidb_kernels.cuh", "tsidb_const.h", "tsidb_host_const.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-Wno-enum-compare", "-o", so, os.path.join(EMU_DIR, "emu_problem.cpp")], check=True)
    return so


class EmuProblem:
    REF_KEYS = ("com", "foot_lf", "foot_rf", "contact_lf", "contact_rf", "posture")

    def __init__(self, cm: TsidbModel, cc: TsidbConf):
        self.lib = C.CDLL(build_emu_problem())
        self.lib.emu_problem_fill_const.argtypes = [C.POINTER(TsidbModel), C.POINTER(TsidbConf)]
        self.lib.emu_problem.argtypes = [C.POINTER(TickArgs), C.POINTER(TsidbProblemOut)]
        assert self.lib.emu_problem_fill_const(C.byref(cm), C.byref(cc)) == 0
        self.cc = cc
        self.na, self.nv = cm.nb - 1, cm.nb + 5

    def problem(self, q, v, mask, refs: dict) -> dict:
        """q [N,nq], v [N,nv], mask [N], refs: per-env [N,k] arrays -> the padded [N, ...] arrays and sizes [N,3]
        (NaN-filled before the call: anything left unwritten shows)."""
        N = q.shape[0]
        na, nv, cc = self.na, self.nv, self.cc
        nx, nin = nv + 24, 2 * (34 + (na if cc.use_torque_bounds else 0) + (nv if cc.use_joint_bounds else 0))
        out = {"H": np.full((N, nx, nx), np.nan), "g": np.full((N, nx), np.nan), "CE": np.full((N, 18, nx), np.nan),
               "ce0": np.full((N, 18), np.nan), "CI": np.full((N, nin, nx), np.nan), "ci0": np.full((N, nin), np.nan),
               "sizes": np.full((N, 3), -1, np.int32)}
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
