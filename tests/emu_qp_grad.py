"""ctypes driver of the host warp emulator build of the QP gradient (tests/emu/emu_qp_grad.cpp): the kernel header's
qp_grad_env runs with 32 lock-step fibers per env and NaN-poisoned shared memory, so tsidb_qp_grad can be compared with
the numpy reference on a box without a GPU.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from emu_py import EMU_DIR, SRC_DIR
from tsid_control_b200._capi import TsidbProblemOut, TsidbQpOut

FLOAT_PARTS = ("H", "g", "CE", "ce0", "CI", "ci0", "TA", "ta0")


def build_emu_qp_grad() -> str:
    so = os.path.join(EMU_DIR, "libtsidb_emu_qp_grad.so")
    srcs = [os.path.join(EMU_DIR, "emu_qp_grad.cpp"), os.path.join(EMU_DIR, "emu_cuda.h")] + [
        os.path.join(SRC_DIR, f) for f in ("tsidb_kernels.cuh", "tsidb_const.h", "tsidb_host_const.h")] + [
        os.path.join(SRC_DIR, "..", "..", "include", "tsidb.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-Wno-enum-compare", "-o", so, os.path.join(EMU_DIR, "emu_qp_grad.cpp")], check=True)
    return so


def emu_qp_grad(problem: dict, sol: dict, grads: dict, parts=None, na: int = 0) -> dict:
    """problem: padded [N, ...] float64 arrays (H, CE, CI, TA as present) and sizes [N,3]; sol: x, status, active, lambda,
    lambda_eq of a solve; grads: any of x, lambda, lambda_eq, tau -> the requested parts (default: the float parts of
    `problem`) at the problem's shapes and status [N], all filled with NaN / -7 before the call so that anything left
    unwritten shows."""
    lib = C.CDLL(build_emu_qp_grad())
    lib.emu_qp_grad.argtypes = [C.c_int] * 5 + [C.POINTER(TsidbProblemOut), C.POINTER(TsidbQpOut), C.POINTER(TsidbQpOut),
                                                C.POINTER(TsidbProblemOut), C.c_void_p]
    N, nm = problem["g"].shape
    neqm = problem["ce0"].shape[1] if "ce0" in problem else 0
    ninm = problem["ci0"].shape[1] if "ci0" in problem else 0
    if "TA" in problem:
        na = problem["TA"].shape[1]
    p = {k: np.ascontiguousarray(problem[k], dtype=np.float64) for k in FLOAT_PARTS if k in problem}
    p["sizes"] = np.ascontiguousarray(problem["sizes"], dtype=np.int32)
    s = {k: np.ascontiguousarray(sol[k], dtype=np.int32 if k in ("status", "active") else np.float64)
         for k in ("x", "status", "active", "lambda", "lambda_eq")}
    g = {k: np.ascontiguousarray(a, dtype=np.float64) for k, a in grads.items()}
    parts = tuple(k for k in FLOAT_PARTS if k in problem) if parts is None else tuple(parts)
    out = {k: np.full(p[k].shape, np.nan) for k in parts}
    status = np.full(N, -7, np.int32)
    keep = (p, s, g, out)  # noqa: F841 (the arrays outlive the call)
    po = TsidbProblemOut(**{k: a.ctypes.data for k, a in p.items()})
    so = TsidbQpOut(**{k: a.ctypes.data for k, a in s.items() if a.size})
    gi = TsidbQpOut(**{k: a.ctypes.data for k, a in g.items() if a.size})
    go = TsidbProblemOut(**{k: a.ctypes.data for k, a in out.items() if a.size})
    rc = lib.emu_qp_grad(N, nm, neqm, ninm, na, C.byref(po), C.byref(so), C.byref(gi), C.byref(go), status.ctypes.data)
    assert rc == 0, rc
    out["status"] = status
    return out
