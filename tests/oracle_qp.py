"""ctypes wrapper of tests/oracle_qp/oracle_qp.c: the CPU oracle's eiquadprog-fast on a caller-supplied dense QP, the
reference of the generic QP kernel (tsidb_qp_solve).  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle_py import NINMAX, NMAX, ORACLE_DIR

QP_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_qp")
NEQMAX = 18

_LIB = None


def _lib() -> C.CDLL:
    """Built like liboracle.so (strict IEEE fp64, no FMA contraction) from the oracle's unchanged source."""
    global _LIB
    if _LIB is None:
        so = os.path.join(QP_DIR, "liboracle_qp.so")
        srcs = [os.path.join(QP_DIR, "oracle_qp.c"), os.path.join(ORACLE_DIR, "tsid_oracle.c"),
                os.path.join(ORACLE_DIR, "tsid_oracle.h")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
            subprocess.run(["gcc", "-std=gnu11", "-fPIC", "-shared", "-Wall", "-Wno-unused-function", "-pthread", "-O2",
                            "-ffp-contract=off", "-o", so, os.path.join(QP_DIR, "oracle_qp.c"), "-lm"], check=True)
        lib = C.CDLL(so)
        vp, ip = C.c_void_p, C.c_int
        lib.oracle_qp_solve.argtypes = [ip, ip, ip, vp, vp, vp, vp, vp, vp, ip, vp, C.POINTER(ip), vp, vp, vp]
        lib.oracle_qp_solve.restype = ip
        _LIB = lib
    return _LIB


def oracle_qp_solve(H, g, CE, ce0, CI, ci0, max_iter: int) -> dict:
    """Dense, unpadded arrays of one QP -> status, iters, x [n], active [n] (-1 padded), lambda [n], lambda_eq [neq]."""
    n, neq, nin = len(g), len(ce0), len(ci0)
    a = {k: np.ascontiguousarray(v, dtype=np.float64).reshape(-1) for k, v in
         (("H", H), ("g", g), ("CE", CE), ("ce0", ce0), ("CI", CI), ("ci0", ci0))}
    x, lam, lam_eq = np.zeros(n), np.zeros(n), np.zeros(max(neq, 1))
    active = np.full(n, -1, np.int32)
    it = C.c_int(0)
    st = _lib().oracle_qp_solve(n, neq, nin, *(a[k].ctypes.data for k in ("H", "g", "CE", "ce0", "CI", "ci0")),
                                int(max_iter), x.ctypes.data, C.byref(it), active.ctypes.data, lam.ctypes.data,
                                lam_eq.ctypes.data)
    if st < 0:
        raise ValueError(f"oracle_qp_solve: sizes ({n}, {neq}, {nin}) beyond the oracle's ({NMAX}, {NEQMAX}, {NINMAX})")
    return {"status": st, "iters": it.value, "x": x, "active": active, "lambda": lam, "lambda_eq": lam_eq[:neq]}
