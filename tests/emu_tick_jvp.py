"""ctypes driver of the host warp emulator build of the forward derivative of export + solve (tests/emu/emu_tick_jvp.cpp):
the kernel header's tick_jvp_env runs with 32 lock-step fibers per env, so tsidb_tick_jvp can be checked against the
adjoints and the oracle on a box without a GPU.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from emu_py import EMU_DIR, SRC_DIR, TickArgs
from emu_refs_grad import REF_KEYS
from tsid_control_b200._capi import TsidbConf, TsidbModel


class JvpArgs(C.Structure):
    _fields_ = [("n_max", C.c_int32), ("neq_max", C.c_int32), ("nin_max", C.c_int32), ("n_dirs", C.c_int32),
                ("shared", C.c_int32)] + \
        [(k, C.c_void_p) for k in ("H", "CE", "CI", "TA", "sizes", "x", "lambda_", "lambda_eq", "sol_status", "active",
                                    "dq", "dv")] + \
        [("dref", C.c_void_p * 6), ("ox", C.c_void_p), ("otau", C.c_void_p), ("status", C.c_void_p)]


def build_emu_tick_jvp() -> str:
    so = os.path.join(EMU_DIR, "libtsidb_emu_tick_jvp.so")
    srcs = [os.path.join(EMU_DIR, "emu_tick_jvp.cpp"), os.path.join(EMU_DIR, "emu_cuda.h")] + [
        os.path.join(SRC_DIR, f) for f in ("tsidb_kernels.cuh", "tsidb_const.h", "tsidb_host_const.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas",
                        "-Wno-enum-compare", "-o", so, os.path.join(EMU_DIR, "emu_tick_jvp.cpp")], check=True)
    return so


class EmuTickJvp:
    def __init__(self, cm: TsidbModel, cc: TsidbConf, defaults: dict):
        self.lib = C.CDLL(build_emu_tick_jvp())
        self.lib.emu_tick_jvp_fill_const.argtypes = [C.POINTER(TsidbModel), C.POINTER(TsidbConf), C.c_void_p]
        self.lib.emu_tick_jvp.argtypes = [C.POINTER(TickArgs), C.POINTER(JvpArgs)]
        self.na, self.nv, self.nq = cm.nb - 1, cm.nb + 5, cm.nb + 6
        flat = np.ascontiguousarray(np.concatenate([np.asarray(defaults[k], np.float64).ravel() for k in REF_KEYS]))
        assert self.lib.emu_tick_jvp_fill_const(C.byref(cm), C.byref(cc), flat.ctypes.data) == 0

    def tick_jvp(self, q, v, mask, refs: dict, prob: dict, sol: dict, dirs: dict, shared: bool = False, layout: int = 0,
                 outs=("x", "tau")) -> dict:
        """q [N,nq], v [N,nv], mask [N] (None: double support), refs {name: [N,k]} (a missing name: the default), prob
        the export (H, CE, CI, TA, sizes; strides from the shapes) and sol its solve (x, status, active, lambda,
        lambda_eq); dirs {"q"/"v"/reference name: [N,D,k] or, shared, [D,k]} (a missing name: NULL) -> {"x": [N,D,n_max],
        "tau": [N,D,na] for `outs`, "status": [N]}, the outputs NaN-filled before the call.  layout 1 passes q, v and
        the references transposed ([k][N])."""
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
        nm = prob["H"].shape[1]
        j = JvpArgs()
        j.n_max, j.neq_max, j.nin_max = nm, prob["CE"].shape[1], prob["CI"].shape[1]
        D = next(iter(dirs.values())).shape[0 if shared else 1]
        j.n_dirs, j.shared = D, int(shared)

        def put(name, arr, dtype=np.float64):
            x = np.ascontiguousarray(arr, dtype=dtype)
            keep.append(x)
            setattr(j, name, x.ctypes.data)

        for k in ("H", "CE", "CI", "TA"):
            if k in prob:
                put(k, prob[k])
        put("sizes", prob["sizes"], np.int32)
        put("x", sol["x"]); put("lambda_", sol["lambda"]); put("lambda_eq", sol["lambda_eq"])
        put("sol_status", sol["status"], np.int32); put("active", sol["active"], np.int32)
        if "q" in dirs:
            put("dq", dirs["q"])
        if "v" in dirs:
            put("dv", dirs["v"])
        for i, k in enumerate(REF_KEYS):
            if k in dirs:
                x = np.ascontiguousarray(dirs[k], dtype=np.float64)
                keep.append(x)
                j.dref[i] = x.ctypes.data
        out = {"x": np.full((N, D, nm), np.nan), "tau": np.full((N, D, self.na), np.nan)}
        out = {k: o for k, o in out.items() if k in outs}
        out["status"] = np.full(N, -7, np.int32)
        j.ox = out["x"].ctypes.data if "x" in out else None
        j.otau = out["tau"].ctypes.data if "tau" in out else None
        j.status = out["status"].ctypes.data
        assert self.lib.emu_tick_jvp(C.byref(a), C.byref(j)) == 0
        return out
