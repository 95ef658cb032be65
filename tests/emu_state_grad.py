"""ctypes driver of the host warp emulator build of the adjoint of the QP export in q and v (tests/emu/emu_state_grad.cpp):
the kernel header's state_grad_env runs with 32 lock-step fibers per env, so tsidb_state_grad can be checked against
the oracle on a box without a GPU.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from emu_py import EMU_DIR, SRC_DIR, TickArgs
from emu_refs_grad import REF_KEYS
from tsid_control_b200._capi import TsidbConf, TsidbModel

PARTS = ("H", "g", "CE", "ce0", "CI", "ci0", "TA", "ta0")


class StateGradArgs(C.Structure):
    _fields_ = [("n_max", C.c_int32), ("neq_max", C.c_int32), ("nin_max", C.c_int32), ("pad_", C.c_int32)] + \
        [(k, C.c_void_p) for k in PARTS] + [("dq", C.c_void_p), ("dv", C.c_void_p)]


def build_emu_state_grad() -> str:
    so = os.path.join(EMU_DIR, "libtsidb_emu_state_grad.so")
    srcs = [os.path.join(EMU_DIR, "emu_state_grad.cpp"), os.path.join(EMU_DIR, "emu_cuda.h")] + [
        os.path.join(SRC_DIR, f) for f in ("tsidb_kernels.cuh", "tsidb_const.h", "tsidb_host_const.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-Wno-enum-compare", "-o", so, os.path.join(EMU_DIR, "emu_state_grad.cpp")], check=True)
    return so


class EmuStateGrad:
    def __init__(self, cm: TsidbModel, cc: TsidbConf, defaults: dict):
        self.lib = C.CDLL(build_emu_state_grad())
        self.lib.emu_state_grad_fill_const.argtypes = [C.POINTER(TsidbModel), C.POINTER(TsidbConf), C.c_void_p]
        self.lib.emu_state_grad.argtypes = [C.POINTER(TickArgs), C.POINTER(StateGradArgs)]
        self.na, self.nv, self.nq = cm.nb - 1, cm.nb + 5, cm.nb + 6
        flat = np.ascontiguousarray(np.concatenate([np.asarray(defaults[k], np.float64).ravel() for k in REF_KEYS]))
        assert self.lib.emu_state_grad_fill_const(C.byref(cm), C.byref(cc), flat.ctypes.data) == 0

    def state_grad(self, q, v, mask, refs: dict, grads: dict, strides, layout: int = 0, parts=("q", "v"),
                   fill=np.nan) -> dict:
        """q [N,nq], v [N,nv], mask [N] (None: double support), refs: {name: [N,k]} (a missing name: the default),
        grads: {part: array} in the export's layout with strides (n_max, neq_max, nin_max) (a missing part: NULL) ->
        {"q": [N,nq], "v": [N,nv]} for `parts`.  layout 1 passes q, v and the references transposed ([k][N]) and
        transposes the outputs back.  Outputs start filled with `fill`."""
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
        r = StateGradArgs()
        r.n_max, r.neq_max, r.nin_max = strides
        for k in PARTS:
            if grads.get(k) is not None:
                x = np.ascontiguousarray(grads[k], dtype=np.float64)
                keep.append(x)
                setattr(r, k, x.ctypes.data)
        dims = {"q": self.nq, "v": self.nv}
        out = {k: np.full((dims[k], N) if layout else (N, dims[k]), fill) for k in parts}
        r.dq = out["q"].ctypes.data if "q" in out else None
        r.dv = out["v"].ctypes.data if "v" in out else None
        assert self.lib.emu_state_grad(C.byref(a), C.byref(r)) == 0
        return {k: np.ascontiguousarray(x.T) if layout else x for k, x in out.items()}
