"""ctypes driver of the host warp emulator build of the adjoint of the reference terms (tests/emu/emu_refs_grad.cpp): the
kernel header's refs_grad_env runs with 32 lock-step fibers per env, so tsidb_refs_grad can be checked against the
oracle on a box without a GPU.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from emu_py import EMU_DIR, SRC_DIR, TickArgs
from tsid_control_b200._capi import TsidbConf, TsidbModel

REF_KEYS = ("com", "foot_lf", "foot_rf", "contact_lf", "contact_rf", "posture")


class RefsGradArgs(C.Structure):
    _fields_ = [("n_max", C.c_int32), ("neq_max", C.c_int32), ("dg", C.c_void_p), ("dce0", C.c_void_p),
                ("out", C.c_void_p * 6)]


def build_emu_refs_grad() -> str:
    so = os.path.join(EMU_DIR, "libtsidb_emu_refs_grad.so")
    srcs = [os.path.join(EMU_DIR, "emu_refs_grad.cpp"), os.path.join(EMU_DIR, "emu_cuda.h")] + [
        os.path.join(SRC_DIR, f) for f in ("tsidb_kernels.cuh", "tsidb_const.h", "tsidb_host_const.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-Wno-enum-compare", "-o", so, os.path.join(EMU_DIR, "emu_refs_grad.cpp")], check=True)
    return so


class EmuRefsGrad:
    def __init__(self, cm: TsidbModel, cc: TsidbConf, defaults: dict):
        self.lib = C.CDLL(build_emu_refs_grad())
        self.lib.emu_refs_grad_fill_const.argtypes = [C.POINTER(TsidbModel), C.POINTER(TsidbConf), C.c_void_p]
        self.lib.emu_refs_grad.argtypes = [C.POINTER(TickArgs), C.POINTER(RefsGradArgs)]
        self.na, self.nv = cm.nb - 1, cm.nb + 5
        flat = np.ascontiguousarray(np.concatenate([np.asarray(defaults[k], np.float64).ravel() for k in REF_KEYS]))
        assert self.lib.emu_refs_grad_fill_const(C.byref(cm), C.byref(cc), flat.ctypes.data) == 0
        self.dims = dict(zip(REF_KEYS, (9, 24, 24, 12, 12, self.na)))

    def refs_grad(self, q, v, mask, refs: dict, dg, dce0, parts=REF_KEYS, layout: int = 0, fill=np.nan) -> dict:
        """q [N,nq], v [N,nv], mask [N] (None: double support), refs: {name: [N,k]} (a missing name: the default),
        dg [N,n_max] / dce0 [N,neq_max] (None: zero) -> {name: [N,k]} for `parts`.  layout 1 passes every per-env array
        transposed ([k][N]) and transposes the outputs back.  Outputs start filled with `fill`."""
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
        r = RefsGradArgs()
        dgc = None if dg is None else np.ascontiguousarray(dg, dtype=np.float64)
        dcc = None if dce0 is None else np.ascontiguousarray(dce0, dtype=np.float64)
        r.n_max = 0 if dgc is None else dgc.shape[1]
        r.neq_max = 0 if dcc is None else dcc.shape[1]
        r.dg = None if dgc is None else dgc.ctypes.data
        r.dce0 = None if dcc is None else dcc.ctypes.data
        out = {k: np.full((self.dims[k], N) if layout else (N, self.dims[k]), fill) for k in parts}
        for i, k in enumerate(REF_KEYS):
            r.out[i] = out[k].ctypes.data if k in out else None
        assert self.lib.emu_refs_grad(C.byref(a), C.byref(r)) == 0
        return {k: np.ascontiguousarray(x.T) if layout else x for k, x in out.items()}
