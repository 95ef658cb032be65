"""ctypes driver of the host warp emulator build of the adjoint of the export in the gains and weights
(tests/emu/emu_gains_grad.cpp): the kernel header's gains_grad_env runs with 32 lock-step fibers per env, so
tsidb_gains_grad can be checked against the oracle on a box without a GPU.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from emu_py import EMU_DIR, SRC_DIR, TickArgs
from tsid_control_b200._capi import GAINS_LEN, TsidbConf, TsidbModel

REF_KEYS = ("com", "foot_lf", "foot_rf", "contact_lf", "contact_rf", "posture")


class GainsGradArgs(C.Structure):
    _fields_ = [("n_max", C.c_int32), ("neq_max", C.c_int32), ("dH", C.c_void_p), ("dg", C.c_void_p), ("dce0", C.c_void_p),
                ("frg", C.c_void_p), ("out", C.c_void_p)]


def build_emu_gains_grad() -> str:
    so = os.path.join(EMU_DIR, "libtsidb_emu_gains_grad.so")
    srcs = [os.path.join(EMU_DIR, "emu_gains_grad.cpp"), os.path.join(EMU_DIR, "emu_cuda.h")] + [
        os.path.join(SRC_DIR, f) for f in ("tsidb_kernels.cuh", "tsidb_const.h", "tsidb_host_const.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-Wno-enum-compare", "-o", so, os.path.join(EMU_DIR, "emu_gains_grad.cpp")], check=True)
    return so


class EmuGainsGrad:
    """One emulated handle: the constants of (cm, cc) with the default references `defaults`."""

    def __init__(self, cm: TsidbModel, cc: TsidbConf, defaults: dict):
        self.lib = C.CDLL(build_emu_gains_grad())
        self.lib.emu_gains_grad_fill_const.argtypes = [C.POINTER(TsidbModel), C.POINTER(TsidbConf), C.c_void_p]
        self.lib.emu_gains_grad.argtypes = [C.POINTER(TickArgs), C.POINTER(GainsGradArgs)]
        self.na, self.nv = cm.nb - 1, cm.nb + 5
        self.cm, self.defaults = cm, defaults
        self.set_conf(cc)

    def set_conf(self, cc: TsidbConf) -> None:
        flat = np.ascontiguousarray(np.concatenate([np.asarray(self.defaults[k], np.float64).ravel() for k in REF_KEYS]))
        assert self.lib.emu_gains_grad_fill_const(C.byref(self.cm), C.byref(cc), flat.ctypes.data) == 0

    def gains_grad(self, q, v, mask, refs: dict, dH, dg, dce0, layout: int = 0, fill=np.nan) -> np.ndarray:
        """q [N,nq], v [N,nv], mask [N] (None: double support), refs: {name: [N,k]} (a missing name: the default),
        dH [N,n_max,n_max] / dg [N,n_max] / dce0 [N,neq_max] (None: zero) -> dL/d(gains) [N, GAINS_LEN].  layout 1
        passes every per-env array transposed ([k][N]) and transposes the output back.  The output starts filled with
        `fill`."""
        N = q.shape[0]
        tr = (lambda x: np.ascontiguousarray(np.asarray(x, np.float64).T)) if layout else \
            (lambda x: np.ascontiguousarray(x, dtype=np.float64))
        keep = [tr(q), tr(v)]
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        a = TickArgs()
        a.n_envs, a.layout, a.slot = N, layout, 0
        a.q, a.v = keep[0].ctypes.data, keep[1].ctypes.data
        a.mask = None if m is None else m.ctypes.data
        fields = {"com": ("r_com", None), "foot_lf": ("r_foot", 0), "foot_rf": ("r_foot", 1), "contact_lf": ("r_contact", 0),
                  "contact_rf": ("r_contact", 1), "posture": ("r_posture", None)}
        for k, arr in refs.items():
            x = tr(arr)
            keep.append(x)
            f, i = fields[k]
            if i is None:
                setattr(a, f, x.ctypes.data)
            else:
                getattr(a, f)[i] = x.ctypes.data
        r = GainsGradArgs()
        parts = [None if x is None else np.ascontiguousarray(x, dtype=np.float64) for x in (dH, dg, dce0)]
        r.n_max = next((x.shape[1] for x in parts[:2] if x is not None), self.nv + 24)
        r.neq_max = 18 if parts[2] is None else parts[2].shape[1]
        r.dH, r.dg, r.dce0 = (None if x is None else x.ctypes.data for x in parts)
        out = np.full((GAINS_LEN, N) if layout else (N, GAINS_LEN), fill)
        r.out = out.ctypes.data
        assert self.lib.emu_gains_grad(C.byref(a), C.byref(r)) == 0
        return np.ascontiguousarray(out.T) if layout else out
