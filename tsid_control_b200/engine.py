"""TsidEngine — torch-tensor front of libtsidb.so (one handle = one model+conf on one GPU).

PyTorch is plumbing here: device memory, streams, and (in sharding.py) torch.distributed.
All arithmetic happens in the CUDA library; nothing in this module computes a tick on the CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _capi
from ._capi import TsidbAuxOut, TsidbGaitConf, TsidbRefs, check, conf_to_c, load_library, model_to_c
from .model_compiler import CompiledModel

REF_KEYS = ("com", "foot_lf", "foot_rf", "contact_lf", "contact_rf", "posture")


class TickOutput:
    """Result of one batched tick: what `sol` + the decode calls give in the reference
    (ref:main.py:121-127), for N envs."""

    __slots__ = ("tau", "ddq", "f", "status", "iters", "active_set", "com", "foot_lf", "foot_rf", "wrench", "lam", "lam_row")

    def __init__(self, **kw):
        for k in self.__slots__:
            setattr(self, k, kw.get(k))


class TsidEngine:
    def __init__(self, model: CompiledModel, conf, lf_frame: str, rf_frame: str, legacy: bool = False,
                 max_envs: int = 65536, device: int = 0):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise _capi.TsidbError("no CUDA device: the TSID tick has no CPU fallback")
        self.model = model
        self.cm = model_to_c(model, lf_frame, rf_frame)
        self.cc = conf_to_c(conf, model, legacy=legacy)
        self.na, self.nv, self.nq = model.na, model.nv, model.nq
        self._ref_dims = tuple(zip(REF_KEYS, (9, 24, 24, 12, 12, model.na)))
        self.device = torch.device("cuda", device)
        self._dev_index = int(device)
        self._tick_cache: Dict[tuple, TickOutput] = {}
        self._refs_struct, self._aux_struct = TsidbRefs(), TsidbAuxOut()
        self._refs_ref, self._aux_ref = C.byref(self._refs_struct), C.byref(self._aux_struct)
        self.max_envs = int(max_envs)
        h = C.c_void_p()
        check(self.lib.tsidb_create(C.byref(self.cm), C.byref(self.cc), self.max_envs, device, C.byref(h)), "tsidb_create")
        self.h = h
        self._out_cache: Dict[int, dict] = {}
        self._gains_version = 0  # bumped by every set_gains(); tick_layer's backward checks it
        self._gain_dims = tuple((k, model.na if k in ("kp_posture", "kd_posture") else n) for k, n in _capi.GAIN_FIELDS)

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.tsidb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _stream(self) -> int:
        """Raw handle of torch's current stream on the engine's device (the private fast getter when torch has it: the
        public one builds a Stream object per call, 4 us of a 75 us single-robot tick)."""
        try:
            return torch._C._cuda_getCurrentRawStream(self._dev_index)
        except AttributeError:
            return torch.cuda.current_stream(self.device).cuda_stream

    def _chk(self, t: torch.Tensor, n: int, nd: int, name: str, dtype=torch.float64) -> torch.Tensor:
        try:
            ok = t.is_cuda and t.dtype is dtype and t.get_device() == self._dev_index
        except AttributeError:
            ok = False
        if not ok:
            raise TypeError(f"{name}: expected a {dtype} tensor on {self.device}")
        if t.shape != (n, nd) or not t.is_contiguous():
            raise ValueError(f"{name}: expected a contiguous [{n}, {nd}] tensor, got {tuple(t.shape)}")
        return t

    def _outputs(self, n: int, aux: bool) -> dict:
        o = self._out_cache.get(n)
        if o is None:
            f64 = dict(dtype=torch.float64, device=self.device)
            o = {
                "tau": torch.empty((n, self.na), **f64), "ddq": torch.empty((n, self.nv), **f64),
                "f": torch.empty((n, 24), **f64),
                "status": torch.empty(n, dtype=torch.int32, device=self.device),
                "iters": torch.empty(n, dtype=torch.int32, device=self.device),
                "active_set": torch.empty((3, n), dtype=torch.int64, device=self.device),
                "com": torch.empty((n, 9), **f64), "foot_lf": torch.empty((n, 12), **f64),
                "foot_rf": torch.empty((n, 12), **f64), "wrench": torch.empty((n, 12), **f64),
                "lam": torch.empty((n, 32), **f64), "lam_row": torch.empty((n, 32), dtype=torch.int32, device=self.device),
            }
            # a few sizes stay resident (a single-robot kinematics()/solve() call between two batched ticks must
            # not evict the batch's buffers); the least recently created goes first
            while len(self._out_cache) >= 4:
                old_n = next(iter(self._out_cache))
                self._out_cache.pop(old_n)
                for key in [k for k in self._tick_cache if k[0] == old_n]:
                    self._tick_cache.pop(key)
            self._out_cache[n] = o
        return o

    def _tick_output(self, o: dict, aux: bool, want_active: bool) -> TickOutput:
        """Fields the call did not write are None (never a stale or uninitialised buffer).  The view object is cached with
        the buffers it wraps (the same tensors come back for the same batch size anyway)."""
        key = (o["tau"].shape[0], aux, want_active)
        t = self._tick_cache.get(key)
        if t is None or t.tau is not o["tau"]:
            keys = ["tau", "ddq", "f", "status", "iters"] + (["active_set"] if want_active else []) + \
                   (["com", "foot_lf", "foot_rf", "wrench", "lam", "lam_row"] if aux else [])
            t = TickOutput(**{k: o[k] for k in keys})
            self._tick_cache[key] = t
        return t

    # ------------------------------------------------------------------ API
    def set_default_refs(self, refs: Dict[str, np.ndarray]) -> None:
        arrs = [np.ascontiguousarray(refs[k], dtype=np.float64) for k in REF_KEYS]
        sizes = (9, 24, 24, 12, 12, self.na)
        for a, s, k in zip(arrs, sizes, REF_KEYS):
            if a.shape != (s,):
                raise ValueError(f"default ref {k}: expected [{s}], got {a.shape}")
        ptrs = [a.ctypes.data_as(_capi.c_double_p) for a in arrs]
        check(self.lib.tsidb_set_default_refs(self.h, *ptrs), "tsidb_set_default_refs")

    def compute(self, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor] = None,
                refs: Optional[Dict[str, torch.Tensor]] = None, aux: bool = False, want_active: bool = True) -> TickOutput:
        """One batched tick.  The returned tensors are the engine's cached output buffers for this batch size: the
        NEXT compute()/rollout()/kinematics() call with the same size overwrites them in place (clone what must
        survive).  aux=False leaves com/foot_lf/foot_rf/wrench None, want_active=False leaves active_set None.
        All calls on one engine must be ordered on one CUDA stream (the handle has one set of workspaces)."""
        n = q.shape[0]
        self._chk(q, n, self.nq, "q")
        self._chk(v, n, self.nv, "v")
        if contact_mask is not None:
            if contact_mask.dtype is not torch.uint8 or not contact_mask.is_cuda or contact_mask.get_device() != self._dev_index \
                    or contact_mask.shape != (n,):
                raise TypeError("contact_mask: expected a uint8 [N] tensor on the engine's device")
        # the argument structs are reused from call to call (a single-robot tick is ~75 us: every microsecond of
        # marshalling shows)
        r = self._refs_struct
        for k, nd in self._ref_dims:
            t = refs.get(k) if refs else None
            setattr(r, k, None if t is None else self._chk(t, n, nd, k).data_ptr())
        o = self._outputs(n, aux)
        if aux:
            a = self._aux_struct
            a.com, a.foot_lf, a.foot_rf, a.wrench = (o[k].data_ptr() for k in ("com", "foot_lf", "foot_rf", "wrench"))
            a.lambda_, a.lambda_row = o["lam"].data_ptr(), o["lam_row"].data_ptr()
        ptrs = o.get("_ptrs")
        if ptrs is None:
            ptrs = o["_ptrs"] = tuple(o[k].data_ptr() for k in ("tau", "ddq", "f", "status", "iters", "active_set"))
        check(self.lib.tsidb_compute(
            self.h, n, 0, q.data_ptr(), v.data_ptr(), contact_mask.data_ptr() if contact_mask is not None else None,
            self._refs_ref, ptrs[0], ptrs[1], ptrs[2], ptrs[3], ptrs[4], ptrs[5] if want_active else None,
            self._aux_ref if aux else None, self._stream()), "tsidb_compute")
        return self._tick_output(o, aux, want_active)

    def host_buffers(self, n: int, pinned: bool = True) -> Dict[str, np.ndarray]:
        """Output buffers for :meth:`compute_host`.  Pinned buffers (the default) are DMA targets themselves;
        pageable ones go through the library's staging copy."""
        shapes = {"tau": ((n, self.na), torch.float64), "ddq": ((n, self.nv), torch.float64), "f": ((n, 24), torch.float64),
                  "status": ((n,), torch.int32), "iters": ((n,), torch.int32), "active_set": ((3, n), torch.int64)}
        out = {}
        self._pinned_keep = getattr(self, "_pinned_keep", [])
        for k, (shp, dt) in shapes.items():
            t = torch.empty(shp, dtype=dt, pin_memory=pinned)
            self._pinned_keep.append(t)
            a = t.numpy()
            out[k] = a.view(np.uint64) if k == "active_set" else a
        return out

    @staticmethod
    def pin(a: np.ndarray) -> np.ndarray:
        """A pinned copy of a host array (so that compute_host can DMA straight from it)."""
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        TsidEngine._pins.append(t)  # the numpy view does not own the pinned allocation
        return t.numpy()

    _pins: list = []

    def compute_host(self, q: np.ndarray, v: np.ndarray, contact_mask: Optional[np.ndarray] = None,
                     refs: Optional[Dict[str, np.ndarray]] = None, want_active: bool = True,
                     out: Optional[Dict[str, np.ndarray]] = None, tau_only: bool = False) -> Dict[str, np.ndarray]:
        """The same tick with HOST numpy buffers in and out (H2D, kernels, D2H inside the call, chunked so that
        the copies overlap the kernels).  `out` = buffers from :meth:`host_buffers` to avoid per-call allocation.
        tau_only=True brings back only tau, status and iters (what ref:main.py:126 sends to the actuators): ddq and f
        stay on the device and out["ddq"], out["f"] are left untouched."""
        q = np.ascontiguousarray(q, dtype=np.float64)
        v = np.ascontiguousarray(v, dtype=np.float64)
        n = q.shape[0]
        if q.shape != (n, self.nq) or v.shape != (n, self.nv):
            raise ValueError("q/v: expected [N,nq] / [N,nv]")
        r = TsidbRefs()
        keep = []
        if refs:
            for k, nd in zip(REF_KEYS, (9, 24, 24, 12, 12, self.na)):
                if refs.get(k) is not None:
                    arr = np.ascontiguousarray(refs[k], dtype=np.float64)
                    if arr.shape != (n, nd):
                        raise ValueError(f"refs[{k}]: expected [{n},{nd}]")
                    keep.append(arr)
                    setattr(r, k, arr.ctypes.data)
        m = None
        if contact_mask is not None:
            m = np.ascontiguousarray(contact_mask, dtype=np.uint8)
        if out is None:
            out = self.host_buffers(n, pinned=False)
        elif out["tau"].shape[0] != n:
            raise ValueError("out: buffers were allocated for a different batch size")
        check(self.lib.tsidb_compute_host(
            self.h, n, q.ctypes.data, v.ctypes.data, m.ctypes.data if m is not None else None, C.byref(r),
            out["tau"].ctypes.data, None if tau_only else out["ddq"].ctypes.data, None if tau_only else out["f"].ctypes.data,
            out["status"].ctypes.data, out["iters"].ctypes.data, out["active_set"].ctypes.data if want_active else None),
            "tsidb_compute_host")
        return out

    def compute_host_devrefs(self, q: np.ndarray, v: np.ndarray, contact_mask: Optional[torch.Tensor] = None,
                             refs: Optional[Dict[str, torch.Tensor]] = None, want_active: bool = True,
                             out: Optional[Dict[str, np.ndarray]] = None, tau_only: bool = False) -> Dict[str, np.ndarray]:
        """compute_host with the references and the contact phases resident on the DEVICE (CUDA tensors, e.g. the
        views of gait_state()): only q and v cross PCIe on the way in (tsidb_compute_host_devrefs); tau_only as in
        :meth:`compute_host`."""
        q = np.ascontiguousarray(q, dtype=np.float64)
        v = np.ascontiguousarray(v, dtype=np.float64)
        n = q.shape[0]
        if q.shape != (n, self.nq) or v.shape != (n, self.nv):
            raise ValueError("q/v: expected [N,nq] / [N,nv]")
        r = TsidbRefs()
        if refs:
            for k, nd in zip(REF_KEYS, (9, 24, 24, 12, 12, self.na)):
                t = refs.get(k)
                if t is not None:
                    setattr(r, k, self._chk(t, n, nd, f"refs[{k}]").data_ptr())
        if contact_mask is not None:
            if contact_mask.dtype != torch.uint8 or contact_mask.device != self.device or tuple(contact_mask.shape) != (n,):
                raise TypeError("contact_mask: expected a uint8 [N] tensor on the engine's device")
        if out is None:
            out = self.host_buffers(n, pinned=False)
        elif out["tau"].shape[0] != n:
            raise ValueError("out: buffers were allocated for a different batch size")
        torch.cuda.current_stream(self.device).synchronize()  # the device arrays must be final: the call uses its own streams
        check(self.lib.tsidb_compute_host_devrefs(
            self.h, n, q.ctypes.data, v.ctypes.data, contact_mask.data_ptr() if contact_mask is not None else None, C.byref(r),
            out["tau"].ctypes.data, None if tau_only else out["ddq"].ctypes.data, None if tau_only else out["f"].ctypes.data,
            out["status"].ctypes.data, out["iters"].ctypes.data, out["active_set"].ctypes.data if want_active else None),
            "tsidb_compute_host_devrefs")
        return out

    def kinematics(self, q: torch.Tensor, v: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """(com9, foot_lf12, foot_rf12): robot.com / robot.framePosition without a solve."""
        n = q.shape[0]
        self._chk(q, n, self.nq, "q")
        if v is not None:
            self._chk(v, n, self.nv, "v")
        o = self._outputs(n, True)
        a = TsidbAuxOut()
        a.com, a.foot_lf, a.foot_rf = o["com"].data_ptr(), o["foot_lf"].data_ptr(), o["foot_rf"].data_ptr()
        check(self.lib.tsidb_kinematics(self.h, n, 0, q.data_ptr(), v.data_ptr() if v is not None else None,
                                        C.byref(a), self._stream()), "tsidb_kinematics")
        return o["com"], o["foot_lf"], o["foot_rf"]

    def integrate(self, q: torch.Tensor, v: torch.Tensor, dv: torch.Tensor, dt: float) -> None:
        """In place: v_mean = v + dt/2 dv; v += dt dv; q = q (+) dt v_mean (ref:ctrl/WalkController.py:291-295)."""
        n = q.shape[0]
        self._chk(q, n, self.nq, "q")
        self._chk(v, n, self.nv, "v")
        self._chk(dv, n, self.nv, "dv")
        check(self.lib.tsidb_integrate(self.h, n, 0, q.data_ptr(), v.data_ptr(), dv.data_ptr(), float(dt), self._stream()),
              "tsidb_integrate")

    # ------------------------------------------------------------------ gait phase machine / closed-loop rollout
    def gait_reset(self, n: int, dt: float, step_duration: float, step_length: float, step_height: float, com_height: float,
                   phase0: Optional[torch.Tensor] = None, vcmd: Optional[torch.Tensor] = None) -> None:
        """(Re)start the device gait of n envs from the default references (tsidb_gait_reset).  phase0 [n] in
        [0,1) and vcmd [n,2] are CUDA fp64 tensors (None = zeros)."""
        gc = TsidbGaitConf(float(dt), float(step_duration), float(step_length), float(step_height), float(com_height))
        if phase0 is not None:
            self._chk(phase0.reshape(n, 1), n, 1, "phase0")
        if vcmd is not None:
            self._chk(vcmd, n, 2, "vcmd")
        self._gait_n = n
        check(self.lib.tsidb_gait_reset(self.h, n, C.byref(gc), phase0.data_ptr() if phase0 is not None else None,
                                        vcmd.data_ptr() if vcmd is not None else None, self._stream()), "tsidb_gait_reset")

    def gait_set_plan(self, steps: Optional[torch.Tensor], n_steps: Optional[torch.Tensor] = None, rise_ratio: float = 0.5) -> None:
        """Footstep plan [N,S,4] (x, y, yaw, side) + n_steps [N] int32 (e.g. from footstep_plan) for the device gait: the
        swing foot follows FootTrajectory(rise_ratio) to the env's next footstep of its side.  None: straight steps."""
        if steps is None:
            check(self.lib.tsidb_gait_set_plan(self.h, 0, None, None, 0, 0.5, self._stream()), "tsidb_gait_set_plan")
            return
        n, S = steps.shape[0], steps.shape[1]
        self._chk(steps.reshape(n, 4 * S), n, 4 * S, "steps")
        if n_steps.dtype != torch.int32 or tuple(n_steps.shape) != (n,) or n_steps.device != self.device:
            raise TypeError("n_steps: expected an int32 [N] tensor on the engine's device")
        check(self.lib.tsidb_gait_set_plan(self.h, n, steps.data_ptr(), n_steps.data_ptr(), S, float(rise_ratio), self._stream()),
              "tsidb_gait_set_plan")

    def _view(self, ptr: int, shape, dtype: torch.dtype) -> torch.Tensor:
        """A torch view of a library-owned device array (no copy)."""
        np_dt = {torch.float64: "<f8", torch.int32: "<i4", torch.uint8: "|u1"}[dtype]

        class _Arr:
            __cuda_array_interface__ = {"shape": tuple(shape), "typestr": np_dt, "data": (int(ptr), False), "version": 2}

        return torch.as_tensor(_Arr(), device=self.device)

    def gait_state(self) -> Dict[str, torch.Tensor]:
        """Views of the gait's device state: references (com, foot_lf, foot_rf, contact_lf, contact_rf), mask,
        phase and the per-env count of failed ticks."""
        n = self._gait_n
        r = TsidbRefs()
        m, ph, fl = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(self.lib.tsidb_gait_state(self.h, C.byref(r), C.byref(m), C.byref(ph), C.byref(fl)), "tsidb_gait_state")
        out = {k: self._view(getattr(r, k), (n, nd), torch.float64)
               for k, nd in (("com", 9), ("foot_lf", 24), ("foot_rf", 24), ("contact_lf", 12), ("contact_rf", 12))}
        out["mask"] = self._view(m.value, (n,), torch.uint8)
        out["phase"] = self._view(ph.value, (n,), torch.float64)
        out["fails"] = self._view(fl.value, (n,), torch.int32)
        return out

    def gait_step(self, foot_lf_now: torch.Tensor, foot_rf_now: torch.Tensor, status: Optional[torch.Tensor] = None) -> None:
        n = self._gait_n
        self._chk(foot_lf_now, n, 12, "foot_lf_now")
        self._chk(foot_rf_now, n, 12, "foot_rf_now")
        check(self.lib.tsidb_gait_step(self.h, n, foot_lf_now.data_ptr(), foot_rf_now.data_ptr(),
                                       status.data_ptr() if status is not None else None, self._stream()), "tsidb_gait_step")

    def foot_trajectory(self, t0: float, t1: float, start: torch.Tensor, target: torch.Tensor, step_height: float,
                        rise_ratio: float, t: torch.Tensor) -> torch.Tensor:
        """FootTrajectory([t0, t1], start, target, step_height, rise_ratio) of ref:ctrl/Foot_Trajectory.py:6-43 evaluated
        per env on the device: start/target [N,4] = (x, y, z, yaw), t [N]; returns [N,4,4]: value and the first three
        derivatives (axis 1) of (x, y, z, yaw) (axis 2)."""
        n = start.shape[0]
        self._chk(start, n, 4, "start")
        self._chk(target, n, 4, "target")
        self._chk(t.reshape(n, 1), n, 1, "t")
        out = torch.empty((n, 16), dtype=torch.float64, device=self.device)
        check(self.lib.tsidb_foot_trajectory(self.h, n, float(t0), float(t1), start.data_ptr(), target.data_ptr(), float(step_height),
                                             float(rise_ratio), t.data_ptr(), out.data_ptr(), self._stream()), "tsidb_foot_trajectory")
        return out.reshape(n, 4, 4)

    def footstep_plan(self, path: torch.Tensor, init_supports: torch.Tensor, step_length: float, step_width: float,
                      n_pts: Optional[torch.Tensor] = None, max_steps: int = 64) -> Tuple[torch.Tensor, torch.Tensor]:
        """FootstepPlanner(step_width, step_length).plan(path, init_supports) of ref:ctrl/Footstep_Planner.py:92-125 per env
        on the device: path [N,P,2], init_supports [N,2,4] = (x, y, yaw, side); returns (steps [N,max_steps,4],
        n_steps [N] int32)."""
        n, P = path.shape[0], path.shape[1]
        self._chk(path.reshape(n, 2 * P), n, 2 * P, "path")
        self._chk(init_supports.reshape(n, 8), n, 8, "init_supports")
        steps = torch.zeros((n, max_steps, 4), dtype=torch.float64, device=self.device)
        ns = torch.zeros(n, dtype=torch.int32, device=self.device)
        check(self.lib.tsidb_footstep_plan(self.h, n, path.data_ptr(), n_pts.data_ptr() if n_pts is not None else None, P,
                                           init_supports.data_ptr(), float(step_length), float(step_width), steps.data_ptr(),
                                           ns.data_ptr(), int(max_steps), self._stream()), "tsidb_footstep_plan")
        return steps, ns

    def rollout(self, q: torch.Tensor, v: torch.Tensor, n_steps: int, use_graph: bool = True) -> TickOutput:
        """n_steps closed-loop ticks on the device (tick -> integrate_dv -> gait step), q and v advanced in place;
        returns the last step's outputs (tau, ddq, f, status, iters; the engine's cached buffers, overwritten by the
        next call of the same batch size).  Needs gait_reset first."""
        n = q.shape[0]
        self._chk(q, n, self.nq, "q")
        self._chk(v, n, self.nv, "v")
        o = self._outputs(n, False)
        check(self.lib.tsidb_rollout(self.h, n, int(n_steps), q.data_ptr(), v.data_ptr(), o["tau"].data_ptr(), o["ddq"].data_ptr(),
                                     o["f"].data_ptr(), o["status"].data_ptr(), o["iters"].data_ptr(), int(use_graph),
                                     self._stream()), "tsidb_rollout")
        return self._tick_output(o, False, False)

    def diagnostics(self, out: TickOutput, contact_mask: Optional[torch.Tensor], omega: float) -> Dict[str, torch.Tensor]:
        """CoP [N,3], capture point [N,3] and support (lf.xy, rf.xy) [N,4] of a tick computed with aux=True
        (tsidb_diagnostics; ref:ctrl/WalkController.py:255-289, ref:legacy/biped.py:224-234)."""
        if out.wrench is None or out.com is None:
            raise RuntimeError("diagnostics needs a tick computed with aux outputs")
        n = out.com.shape[0]
        f64 = dict(dtype=torch.float64, device=self.device)
        res = {"cop": torch.empty((n, 3), **f64), "capture_point": torch.empty((n, 3), **f64), "support": torch.empty((n, 4), **f64)}
        a = TsidbAuxOut()
        a.com, a.foot_lf, a.foot_rf, a.wrench = out.com.data_ptr(), out.foot_lf.data_ptr(), out.foot_rf.data_ptr(), out.wrench.data_ptr()
        check(self.lib.tsidb_diagnostics(self.h, n, C.byref(a), contact_mask.data_ptr() if contact_mask is not None else None,
                                         float(omega), res["cop"].data_ptr(), res["capture_point"].data_ptr(),
                                         res["support"].data_ptr(), self._stream()), "tsidb_diagnostics")
        return res

    PROBLEM_PARTS = ("H", "g", "CE", "ce0", "CI", "ci0")
    ACTUATION_PARTS = ("TA", "ta0")

    def problem_sizes(self) -> Tuple[int, int, int]:
        """(n_max, neq_max, nin_max): the padding of :meth:`problem_data`'s arrays (tsidb_problem_sizes)."""
        n, neq, nin = C.c_int(), C.c_int(), C.c_int()
        check(self.lib.tsidb_problem_sizes(self.h, C.byref(n), C.byref(neq), C.byref(nin)), "tsidb_problem_sizes")
        return n.value, neq.value, nin.value

    def problem_data(self, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor] = None,
                     refs: Optional[Dict[str, torch.Tensor]] = None, parts=PROBLEM_PARTS) -> Dict[str, torch.Tensor]:
        """computeProblemData without the solve (tsidb_problem_data): for every env the QP SolverHQuadProgFast hands to
        eiquadprog, min 1/2 x'Hx + g'x s.t. CE x + ce0 = 0, CI x + ci0 >= 0, in x = [dv; f of the feet in contact, LF
        first].  Returns new CUDA tensors H [N,n,n], g [N,n], CE [N,18,n], ce0 [N,18], CI [N,nin,n], ci0 [N,nin] (the
        requested `parts`, padded with zeros to problem_sizes()) and sizes [N,3] int32 = (n, neq, nin) of each env.
        `parts` may also name the actuation map TA [N,na,n], ta0 [N,na]: tau = TA x + ta0 (getActuatorForces).
        Inputs as in :meth:`compute`; a later tick's results do not depend on this call."""
        n = q.shape[0]
        self._chk(q, n, self.nq, "q")
        self._chk(v, n, self.nv, "v")
        if contact_mask is not None:
            if contact_mask.dtype is not torch.uint8 or not contact_mask.is_cuda or contact_mask.get_device() != self._dev_index \
                    or contact_mask.shape != (n,):
                raise TypeError("contact_mask: expected a uint8 [N] tensor on the engine's device")
        unknown = set(parts) - set(self.PROBLEM_PARTS + self.ACTUATION_PARTS)
        if unknown:
            raise ValueError(f"parts: unknown {sorted(unknown)}; choose from {self.PROBLEM_PARTS + self.ACTUATION_PARTS}")
        r = TsidbRefs()
        for k, nd in self._ref_dims:
            t = refs.get(k) if refs else None
            setattr(r, k, None if t is None else self._chk(t, n, nd, k).data_ptr())
        nx, neq, nin = self.problem_sizes()
        shapes = {"H": (n, nx, nx), "g": (n, nx), "CE": (n, neq, nx), "ce0": (n, neq), "CI": (n, nin, nx), "ci0": (n, nin),
                  "TA": (n, self.na, nx), "ta0": (n, self.na)}
        out = {k: torch.empty(shapes[k], dtype=torch.float64, device=self.device) for k in parts}
        out["sizes"] = torch.empty((n, 3), dtype=torch.int32, device=self.device)
        po = _capi.TsidbProblemOut(**{k: t.data_ptr() for k, t in out.items()})
        check(self.lib.tsidb_problem_data(self.h, n, 0, q.data_ptr(), v.data_ptr(),
                                          contact_mask.data_ptr() if contact_mask is not None else None, C.byref(r),
                                          C.byref(po), self._stream()), "tsidb_problem_data")
        return out

    def qp_solve(self, problem: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """eiquadprog-fast with this controller's max_iter on every env of `problem` (tsidb_qp_solve): a dict in the
        layout :meth:`problem_data` returns, possibly modified or enlarged.  H [N,n_max,n_max], g [N,n_max] and sizes
        [N,3] int32 are required; CE [N,neq_max,n_max] with ce0 [N,neq_max], CI [N,nin_max,n_max] with ci0 [N,nin_max]
        and TA [N,na,n_max] with ta0 [N,na] are optional (absent = no such rows / no tau).  The strides come from the
        shapes.  Returns new CUDA tensors x [N,n_max], status, iters [N] int32, active [N,n_max] int32 (CI rows of the
        working set in working-set order, -1 padded), lambda [N,n_max] (their multipliers), lambda_eq [N,neq_max] and,
        with TA and ta0, tau [N,na]."""
        n, nx, neq, nin = self._qp_problem("qp_solve", problem)
        f64 = dict(dtype=torch.float64, device=self.device)
        i32 = dict(dtype=torch.int32, device=self.device)
        out = {"x": torch.empty((n, nx), **f64), "status": torch.empty(n, **i32), "iters": torch.empty(n, **i32),
               "active": torch.empty((n, nx), **i32), "lambda": torch.empty((n, nx), **f64),
               "lambda_eq": torch.empty((n, neq), **f64)}
        if "TA" in problem:
            out["tau"] = torch.empty((n, self.na), **f64)
        po = _capi.TsidbProblemOut(**{k: t.data_ptr() for k, t in problem.items()})
        qo = _capi.TsidbQpOut(**{k: t.data_ptr() for k, t in out.items()})
        check(self.lib.tsidb_qp_solve(self.h, n, nx, neq, nin, C.byref(po), C.byref(qo), self._stream()), "tsidb_qp_solve")
        return out

    def _qp_problem(self, what: str, problem: Dict[str, torch.Tensor]) -> Tuple[int, int, int, int]:
        """Checks a problem dict in the layout of :meth:`problem_data` -> (N, n_max, neq_max, nin_max) from its shapes."""
        for k in ("H", "g", "sizes"):
            if k not in problem:
                raise ValueError(f"{what}: {k} is required")
        for a, b in (("CE", "ce0"), ("CI", "ci0"), ("TA", "ta0")):
            if (a in problem) != (b in problem):
                raise ValueError(f"{what}: {a} and {b} go together")
        unknown = set(problem) - set(self.PROBLEM_PARTS + self.ACTUATION_PARTS + ("sizes",))
        if unknown:
            raise ValueError(f"{what}: unknown parts {sorted(unknown)}")
        n, nx = problem["g"].shape if problem["g"].dim() == 2 else (-1, -1)
        neq = problem["ce0"].shape[-1] if "ce0" in problem else 0
        nin = problem["ci0"].shape[-1] if "ci0" in problem else 0
        shapes = {"H": (n, nx, nx), "g": (n, nx), "CE": (n, neq, nx), "ce0": (n, neq), "CI": (n, nin, nx), "ci0": (n, nin),
                  "TA": (n, self.na, nx), "ta0": (n, self.na), "sizes": (n, 3)}
        self._qp_tensors(what, problem, shapes)
        return n, nx, neq, nin

    def _qp_tensors(self, what: str, tensors: Dict[str, torch.Tensor], shapes: Dict[str, tuple]) -> None:
        for k, t in tensors.items():
            dt = torch.int32 if k in ("sizes", "status", "iters", "active") else torch.float64
            if not isinstance(t, torch.Tensor) or t.dtype is not dt or not t.is_cuda or t.get_device() != self._dev_index \
                    or not t.is_contiguous() or tuple(t.shape) != shapes[k]:
                raise TypeError(f"{what}: {k}: expected a contiguous {dt} tensor of shape {shapes[k]} on the engine's device")

    def qp_grad(self, problem: Dict[str, torch.Tensor], sol: Dict[str, torch.Tensor], grads: Dict[str, torch.Tensor],
                parts: Optional[Tuple[str, ...]] = None) -> Dict[str, torch.Tensor]:
        """Adjoint of :meth:`qp_solve` (tsidb_qp_grad): the gradient of a loss with respect to the problem's parts from its
        gradient with respect to the solve's outputs.  `problem` is what qp_solve was given and `sol` what it returned
        (x, status, active, lambda, lambda_eq are read).  `grads` holds any of x [N,n_max], lambda [N,n_max],
        lambda_eq [N,neq_max] and tau [N,na] (absent = zero; tau needs TA).  `parts` names the gradients to compute among
        the float parts of `problem` (default: all of them).  Returns new CUDA tensors of those parts' shapes and status
        [N] int32: 0 where the env was differentiated, 4 (zero gradients) where it was not (a solve status other than 0,
        an invalid working set, H not positive definite or dependent working-set rows).  The gradient is the one of the
        final working set's KKT system, and that of H is lower triangular (the solve reads only that triangle); see
        INTEGRATION.md, "Differentiating a QP"."""
        n, nx, neq, nin = self._qp_problem("qp_grad", problem)
        floats = tuple(k for k in self.PROBLEM_PARTS + self.ACTUATION_PARTS if k in problem)
        parts = floats if parts is None else tuple(parts)
        if set(parts) - set(floats):
            raise ValueError(f"qp_grad: parts {sorted(set(parts) - set(floats))} are not float parts of the problem")
        need = ("x", "status", "active", "lambda", "lambda_eq")
        if set(need) - set(sol):
            raise ValueError(f"qp_grad: sol needs {need}")
        if set(grads) - {"x", "lambda", "lambda_eq", "tau"}:
            raise ValueError(f"qp_grad: unknown gradients {sorted(set(grads) - {'x', 'lambda', 'lambda_eq', 'tau'})}")
        if "tau" in grads and "TA" not in problem:
            raise ValueError("qp_grad: a tau gradient needs TA")
        shapes = {"x": (n, nx), "status": (n,), "active": (n, nx), "lambda": (n, nx), "lambda_eq": (n, neq), "tau": (n, self.na)}
        sol = {k: sol[k] for k in need}
        self._qp_tensors("qp_grad", sol, shapes)
        self._qp_tensors("qp_grad", grads, shapes)
        out = {k: torch.empty_like(problem[k]) for k in parts}
        out["status"] = torch.empty(n, dtype=torch.int32, device=self.device)
        po = _capi.TsidbProblemOut(**{k: t.data_ptr() for k, t in problem.items()})
        so = _capi.TsidbQpOut(**{k: t.data_ptr() for k, t in sol.items()})
        gi = _capi.TsidbQpOut(**{k: t.data_ptr() for k, t in grads.items()})
        go = _capi.TsidbProblemOut(**{k: out[k].data_ptr() for k in parts})
        check(self.lib.tsidb_qp_grad(self.h, n, nx, neq, nin, C.byref(po), C.byref(so), C.byref(gi), C.byref(go),
                                     out["status"].data_ptr(), self._stream()), "tsidb_qp_grad")
        return out

    def qp_layer(self, problem: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """:meth:`qp_solve` as a differentiable layer: the same result, with x, lambda, lambda_eq and tau carrying a
        grad_fn for every float tensor of `problem` that requires grad; the backward pass is :meth:`qp_grad` (first
        order only).  sizes gets no gradient, and an env that was not differentiated contributes zero."""
        keys = tuple(k for k in self.PROBLEM_PARTS + self.ACTUATION_PARTS if k in problem)
        outs = _QpLayer.apply(self, problem["sizes"], keys, *(problem[k] for k in keys))
        names = ("x", "lambda", "lambda_eq", "status", "iters", "active") + (("tau",) if "TA" in problem else ())
        return dict(zip(names, outs))

    def _state_args(self, what: str, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor],
                    refs: Optional[Dict[str, torch.Tensor]]) -> TsidbRefs:
        """Checks q, v, contact_mask and refs as :meth:`problem_data` does -> the refs struct (a missing name: the default)."""
        n = q.shape[0]
        self._chk(q, n, self.nq, "q")
        self._chk(v, n, self.nv, "v")
        if contact_mask is not None:
            if contact_mask.dtype is not torch.uint8 or not contact_mask.is_cuda or contact_mask.get_device() != self._dev_index \
                    or contact_mask.shape != (n,):
                raise TypeError("contact_mask: expected a uint8 [N] tensor on the engine's device")
        unknown = set(refs or ()) - set(REF_KEYS)
        if unknown:
            raise ValueError(f"{what}: unknown references {sorted(unknown)}; choose from {REF_KEYS}")
        r = TsidbRefs()
        for k, nd in self._ref_dims:
            t = refs.get(k) if refs else None
            setattr(r, k, None if t is None else self._chk(t, n, nd, k).data_ptr())
        return r

    def refs_grad(self, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor] = None,
                  refs: Optional[Dict[str, torch.Tensor]] = None, dg: Optional[torch.Tensor] = None,
                  dce0: Optional[torch.Tensor] = None, parts: Optional[Tuple[str, ...]] = None) -> Dict[str, torch.Tensor]:
        """Adjoint of the references' part of :meth:`problem_data` (tsidb_refs_grad): from dg = dL/dg [N,n_max] and
        dce0 = dL/dce0 [N,neq_max] (None = zero; n_max, neq_max at least those of problem_sizes(), e.g. what
        :meth:`qp_grad` returns), new CUDA tensors {name: [N,k]} = dL/d of the references named in `parts` (default: all of
        REF_KEYS).  q, v, contact_mask and refs as in :meth:`problem_data`; a reference left out of `refs` is the handle's
        default and its gradient is the one at that default.  SE3 references are differentiated in their raw 12 or 24
        doubles (the rotation as its 9 column-major entries); the contact reference of a foot that is not in contact
        gets zeros.  See INTEGRATION.md, "Differentiating through the references"."""
        r = self._state_args("refs_grad", q, v, contact_mask, refs)
        n = q.shape[0]
        nx, neq, _ = self.problem_sizes()
        parts = REF_KEYS if parts is None else tuple(parts)
        if set(parts) - set(REF_KEYS):
            raise ValueError(f"refs_grad: parts {sorted(set(parts) - set(REF_KEYS))} are not references; choose from {REF_KEYS}")
        for name, t, lo in (("dg", dg, nx), ("dce0", dce0, neq)):
            if t is None:
                continue
            if not isinstance(t, torch.Tensor) or t.dtype is not torch.float64 or not t.is_cuda or t.get_device() != self._dev_index \
                    or not t.is_contiguous() or t.dim() != 2 or t.shape[0] != n or t.shape[1] < lo:
                raise TypeError(f"refs_grad: {name}: expected a contiguous torch.float64 tensor of shape ({n}, >= {lo}) on the "
                                f"engine's device")
        dims = dict(self._ref_dims)
        out = {k: torch.empty((n, dims[k]), dtype=torch.float64, device=self.device) for k in parts}
        ro = _capi.TsidbRefsOut(**{k: t.data_ptr() for k, t in out.items()})
        check(self.lib.tsidb_refs_grad(self.h, n, 0, q.data_ptr(), v.data_ptr(),
                                       contact_mask.data_ptr() if contact_mask is not None else None, C.byref(r),
                                       dg.shape[1] if dg is not None else nx, dce0.shape[1] if dce0 is not None else neq,
                                       dg.data_ptr() if dg is not None else None, dce0.data_ptr() if dce0 is not None else None,
                                       C.byref(ro), self._stream()), "tsidb_refs_grad")
        return out

    def state_grad(self, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor] = None,
                   refs: Optional[Dict[str, torch.Tensor]] = None, grads: Optional[Dict[str, torch.Tensor]] = None,
                   parts: Tuple[str, ...] = ("q", "v")) -> Dict[str, torch.Tensor]:
        """Adjoint of all of :meth:`problem_data` with respect to the state (tsidb_state_grad): from `grads`, dL/d of any
        of the export's parts H, g, CE, ce0, CI, ci0, TA, ta0 in the layout problem_data returns (strides from the shapes,
        at least problem_sizes(); an absent part counts as zero; a "status" entry, as :meth:`qp_grad` returns it, is
        ignored), new CUDA tensors {"q": [N,nq], "v": [N,nv]} for `parts`.  q, v, contact_mask and refs as in
        :meth:`problem_data`.  The gradient is with respect to the raw doubles of q (the free-flyer quaternion's four
        components, unnormalised); only the state-dependent entries inside each env's sizes are read, so padding and
        constant blocks may hold anything.  See INTEGRATION.md, "Differentiating with respect to the state"."""
        r = self._state_args("state_grad", q, v, contact_mask, refs)
        n = q.shape[0]
        parts = tuple(parts)
        if not parts or set(parts) - {"q", "v"}:
            raise ValueError(f"state_grad: parts must name q and/or v, got {parts}")
        floats = self.PROBLEM_PARTS + self.ACTUATION_PARTS
        grads = {k: t for k, t in (grads or {}).items() if k != "status"}
        if set(grads) - set(floats):
            raise ValueError(f"state_grad: unknown parts {sorted(set(grads) - set(floats))}; choose from {floats}")
        nx0, neq0, nin0 = self.problem_sizes()

        def stride(where, default):  # the first given part that has the axis; the shape check below catches the rest
            return next((grads[k].shape[d] for k, d in where if k in grads and grads[k].dim() > d), default)

        nx = stride((("H", 2), ("g", 1), ("CE", 2), ("CI", 2), ("TA", 2)), nx0)
        neq = stride((("ce0", 1), ("CE", 1)), neq0)
        nin = stride((("ci0", 1), ("CI", 1)), nin0)
        if nx < nx0 or neq < neq0 or nin < nin0:
            raise TypeError(f"state_grad: strides ({nx}, {neq}, {nin}) below problem_sizes() ({nx0}, {neq0}, {nin0})")
        shapes = {"H": (n, nx, nx), "g": (n, nx), "CE": (n, neq, nx), "ce0": (n, neq), "CI": (n, nin, nx), "ci0": (n, nin),
                  "TA": (n, self.na, nx), "ta0": (n, self.na)}
        self._qp_tensors("state_grad", grads, shapes)
        out = {k: torch.empty((n, self.nq if k == "q" else self.nv), dtype=torch.float64, device=self.device) for k in parts}
        po = _capi.TsidbProblemOut(**{k: t.data_ptr() for k, t in grads.items()})
        check(self.lib.tsidb_state_grad(self.h, n, 0, q.data_ptr(), v.data_ptr(),
                                        contact_mask.data_ptr() if contact_mask is not None else None, C.byref(r),
                                        nx, neq, nin, C.byref(po), out["q"].data_ptr() if "q" in out else None,
                                        out["v"].data_ptr() if "v" in out else None, self._stream()), "tsidb_state_grad")
        return out

    GAIN_NAMES = tuple(k for k, _ in _capi.GAIN_FIELDS)

    def gains(self) -> Dict[str, torch.Tensor]:
        """The handle's task gains and weights (tsidb_get_gains): {name: float64 tensor [k]} on the engine's device, k = 6,
        3 or na for the gains and 1 for each weight; names as in tsidb_conf (GAIN_NAMES)."""
        g = _capi.TsidbGains()
        check(self.lib.tsidb_get_gains(self.h, C.byref(g)), "tsidb_get_gains")
        flat = np.frombuffer(bytes(g), dtype=np.float64)
        out, c = {}, 0
        for (k, n), (_, kk) in zip(_capi.GAIN_FIELDS, self._gain_dims):
            out[k] = torch.tensor(flat[c:c + kk], dtype=torch.float64, device=self.device)
            c += n
        return out

    def set_gains(self, gains: Dict[str, object]) -> None:
        """Replaces some of the task gains and weights for every later call (tsidb_set_gains, tsid's setKp / setKd /
        updateTaskWeight): `gains` maps names of :meth:`gains` to values of its shapes (tensors or array-likes); an absent
        name keeps its value.  Synchronises the device.  Raises TsidbError, the handle unchanged, on a non-finite value,
        w_foot, w_com or w_posture <= 0, a w_force_reg that leaves the force block not positive definite, or a w_am that
        would switch the AM task on or off.  Values equal bit for bit to the current ones are a no-op: no library call, no
        device synchronisation, and the gains version that tick_layer's backward pass checks stays as it is."""
        unknown = set(gains) - set(self.GAIN_NAMES)
        if unknown:
            raise ValueError(f"set_gains: unknown names {sorted(unknown)}; choose from {self.GAIN_NAMES}")
        g = _capi.TsidbGains()
        check(self.lib.tsidb_get_gains(self.h, C.byref(g)), "tsidb_get_gains")
        current = bytes(g)
        dims = dict(self._gain_dims)
        for k, val in gains.items():
            if isinstance(val, torch.Tensor):
                val = val.detach().to("cpu", torch.float64).numpy()
            a = np.asarray(val, dtype=np.float64).reshape(-1)
            if a.shape != (dims[k],):
                raise ValueError(f"set_gains: {k}: expected {dims[k]} values, got {a.size}")
            if dims[k] == 1 and k.startswith("w_"):
                setattr(g, k, float(a[0]))
            else:
                field = getattr(g, k)
                for i, x in enumerate(a):
                    field[i] = float(x)
        if bytes(g) == current:
            return
        check(self.lib.tsidb_set_gains(self.h, C.byref(g)), "tsidb_set_gains")
        self._gains_version += 1

    def gains_grad(self, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor] = None,
                   refs: Optional[Dict[str, torch.Tensor]] = None, grads: Optional[Dict[str, torch.Tensor]] = None,
                   parts: Optional[Tuple[str, ...]] = None) -> Dict[str, torch.Tensor]:
        """Adjoint of :meth:`problem_data` with respect to the handle's current gains and weights (tsidb_gains_grad), per
        env: from `grads`, the dict :meth:`qp_grad` returns (H, g and ce0 are read, absent = zero; every other entry is
        ignored), new CUDA tensors {name: [N,k]} for the names in `parts` (default: all of GAIN_NAMES), shapes as
        :meth:`gains` with a leading env axis.  A gain every env shares has as gradient the sum over envs.  q, v,
        contact_mask and refs as in :meth:`problem_data`.  See INTEGRATION.md, "Differentiating with respect to the gains
        and weights"."""
        r = self._state_args("gains_grad", q, v, contact_mask, refs)
        n = q.shape[0]
        parts = self.GAIN_NAMES if parts is None else tuple(parts)
        if set(parts) - set(self.GAIN_NAMES):
            raise ValueError(f"gains_grad: unknown names {sorted(set(parts) - set(self.GAIN_NAMES))}")
        grads = {k: t for k, t in (grads or {}).items() if k in ("H", "g", "ce0")}
        nx0, neq0, _ = self.problem_sizes()
        nx = grads["g"].shape[-1] if "g" in grads else (grads["H"].shape[-1] if "H" in grads else nx0)
        neq = grads["ce0"].shape[-1] if "ce0" in grads else neq0
        if nx < nx0 or neq < neq0:
            raise TypeError(f"gains_grad: strides ({nx}, {neq}) below problem_sizes() ({nx0}, {neq0})")
        self._qp_tensors("gains_grad", grads, {"H": (n, nx, nx), "g": (n, nx), "ce0": (n, neq)})
        out = torch.empty((n, _capi.GAINS_LEN), dtype=torch.float64, device=self.device)
        ptr = {k: (t.data_ptr() if k in grads else None) for k, t in (("H", grads.get("H")), ("g", grads.get("g")),
                                                                      ("ce0", grads.get("ce0")))}
        check(self.lib.tsidb_gains_grad(self.h, n, 0, q.data_ptr(), v.data_ptr(),
                                        contact_mask.data_ptr() if contact_mask is not None else None, C.byref(r), nx, neq,
                                        ptr["H"], ptr["g"], ptr["ce0"], out.data_ptr(), self._stream()), "tsidb_gains_grad")
        res, c = {}, 0
        for (k, nfield), (_, kk) in zip(_capi.GAIN_FIELDS, self._gain_dims):
            if k in parts:
                res[k] = out[:, c:c + kk].contiguous()
            c += nfield
        return res

    def tick_layer(self, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor] = None,
                   refs: Optional[Dict[str, torch.Tensor]] = None,
                   gains: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """A tick as a differentiable function of its state and references: {tau [N,na], dv [N,nv], f [N,24], status,
        iters [N] int32}, with tau, dv and f carrying a grad_fn for q, v and every tensor of `refs` that requires grad
        (first order only).
        f holds the corner forces in the tick's fixed slots, LF 0..11 and RF 12..23, zero for a foot not in contact.
        The forward pass is :meth:`problem_data` (with TA, ta0) followed by :meth:`qp_solve`, not the fast tick: the
        backward pass (:meth:`qp_grad` for g and ce0, then :meth:`refs_grad`) must differentiate the working set its own
        forward pass found, and the two solves can end in different working sets at degenerate contact-corner ties.  That
        costs time: about 74 ms for the forward pass at 65536 walking envs against 3 ms for a tick.  An env whose solve or
        adjoint status is not 0 contributes zero.  When q or v requires grad, the backward pass asks :meth:`qp_grad` for
        every part and adds :meth:`state_grad` (q in its raw doubles, the quaternion unnormalised); otherwise it makes
        the same calls as for references alone.  contact_mask gets no gradient.
        `gains` maps names of :meth:`gains` to tensors of its shapes: the forward pass first applies them as
        :meth:`set_gains` does (which synchronises), and when any of them requires grad the backward pass also asks
        qp_grad for H and adds :meth:`gains_grad`, summed over the envs.  The backward pass raises if set_gains changed
        the gains after the forward pass (its gradients would be those of other gains); calls that pass the same values,
        such as the ticks of one closed loop, leave each other's backward passes valid."""
        self._state_args("tick_layer", q, v, contact_mask, refs)
        keys = tuple(k for k in REF_KEYS if refs and refs.get(k) is not None)
        gains = dict(gains or {})
        dims = dict(self._gain_dims)
        for k, t in gains.items():
            if k not in dims:
                raise ValueError(f"tick_layer: unknown gain {k!r}; choose from {self.GAIN_NAMES}")
            if not isinstance(t, torch.Tensor) or t.dtype is not torch.float64 or tuple(t.shape) != (dims[k],):
                raise TypeError(f"tick_layer: gains[{k!r}]: expected a torch.float64 tensor of shape ({dims[k]},)")
        gkeys = tuple(k for k in self.GAIN_NAMES if k in gains)
        outs = _TickLayer.apply(self, q, v, contact_mask, keys, gkeys, *(refs[k] for k in keys), *(gains[k] for k in gkeys))
        return dict(zip(("tau", "dv", "f", "status", "iters"), outs))

    def tick_jvp(self, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor] = None,
                 refs: Optional[Dict[str, torch.Tensor]] = None, tangents: Optional[Dict[str, torch.Tensor]] = None,
                 prob: Optional[Dict[str, torch.Tensor]] = None, sol: Optional[Dict[str, torch.Tensor]] = None
                 ) -> Dict[str, torch.Tensor]:
        """Forward-mode derivative of :meth:`tick_layer`'s forward pass (tsidb_tick_jvp): for D tangent directions,
        `tangents` maps "q", "v" and reference names to [N,D,k] (per env) or [D,k] (shared by every env) float64 tensors,
        all of one kind (an absent name: zero tangent).  Returns new CUDA tensors x [N,D,n_max] (the tangent of the solve's
        x), tau [N,D,na], dv [N,D,nv] and f [N,D,24] (in the tick's fixed LF/RF slots, as tick_layer maps x) and status
        [N] int32 (4 with zero tangents where qp_grad would refuse the env).  `prob` (problem_data with TA, ta0) and `sol`
        (qp_solve on it) are the forward pass; without them the call runs it.  q is differentiated in its raw doubles
        (the quaternion unnormalised), SE3 references in their raw 12 or 24 doubles.  See INTEGRATION.md, "Linearizing
        the controller"."""
        r = self._state_args("tick_jvp", q, v, contact_mask, refs)
        n = q.shape[0]
        tangents = dict(tangents or {})
        dims = dict(self._ref_dims, q=self.nq, v=self.nv)
        if not tangents or set(tangents) - set(dims):
            raise ValueError(f"tick_jvp: tangents must name some of {tuple(dims)}, got {sorted(tangents)}")
        ranks = {t.dim() if isinstance(t, torch.Tensor) else -1 for t in tangents.values()}
        if ranks - {2, 3} or len(ranks) != 1:
            raise TypeError("tick_jvp: tangents must all be [N,D,k] (per env) or all [D,k] (shared)")
        shared = ranks == {2}
        d = next(iter(tangents.values())).shape[0 if shared else 1]
        for k, t in tangents.items():
            want = (d, dims[k]) if shared else (n, d, dims[k])
            if t.dtype is not torch.float64 or not t.is_cuda or t.get_device() != self._dev_index or not t.is_contiguous() \
                    or tuple(t.shape) != want or d < 1:
                raise TypeError(f"tick_jvp: tangents[{k!r}]: expected a contiguous torch.float64 tensor of shape {want} "
                                f"on the engine's device")
        if (prob is None) != (sol is None):
            raise ValueError("tick_jvp: prob and sol go together")
        if prob is None:
            prob = self.problem_data(q, v, contact_mask, refs, parts=self.PROBLEM_PARTS + self.ACTUATION_PARTS)
            sol = self.qp_solve(prob)
        for k in ("CE", "CI", "TA"):
            if k not in prob:
                raise ValueError(f"tick_jvp: prob needs {k}")
        n_, nx, neq, nin = self._qp_problem("tick_jvp", prob)
        if n_ != n:
            raise TypeError(f"tick_jvp: prob has {n_} envs, q has {n}")
        need = ("x", "status", "active", "lambda", "lambda_eq")
        if set(need) - set(sol):
            raise ValueError(f"tick_jvp: sol needs {need}")
        sol = {k: sol[k] for k in need}
        self._qp_tensors("tick_jvp", sol, {"x": (n, nx), "status": (n,), "active": (n, nx), "lambda": (n, nx),
                                           "lambda_eq": (n, neq)})
        f64 = dict(dtype=torch.float64, device=self.device)
        out = {"x": torch.empty((n, d, nx), **f64), "tau": torch.empty((n, d, self.na), **f64),
               "status": torch.empty(n, dtype=torch.int32, device=self.device)}
        dr = _capi.TsidbRefs(**{k: t.data_ptr() for k, t in tangents.items() if k in REF_KEYS})
        jd = _capi.TsidbJvpDirs(q=tangents["q"].data_ptr() if "q" in tangents else None,
                                v=tangents["v"].data_ptr() if "v" in tangents else None, refs=dr)
        jo = _capi.TsidbJvpOut(x=out["x"].data_ptr(), tau=out["tau"].data_ptr())
        po = _capi.TsidbProblemOut(**{k: t.data_ptr() for k, t in prob.items()})
        so = _capi.TsidbQpOut(**{k: t.data_ptr() for k, t in sol.items()})
        check(self.lib.tsidb_tick_jvp(self.h, n, 0, q.data_ptr(), v.data_ptr(),
                                      contact_mask.data_ptr() if contact_mask is not None else None, C.byref(r), nx, neq, nin,
                                      C.byref(po), C.byref(so), d, int(shared), C.byref(jd), C.byref(jo),
                                      out["status"].data_ptr(), self._stream()), "tsidb_tick_jvp")
        out["dv"], out["f"] = _TickLayer.split_x(out["x"], contact_mask, self.nv)
        return out

    def tick_jacobian(self, q: torch.Tensor, v: torch.Tensor, contact_mask: Optional[torch.Tensor] = None,
                      refs: Optional[Dict[str, torch.Tensor]] = None, wrt: Tuple[str, ...] = ("q", "v")
                      ) -> Dict[str, torch.Tensor]:
        """The Jacobian of :meth:`tick_layer`'s forward pass (not of the fast tick: at degenerate contact-corner ties the
        two solves can end in different working sets) with respect to the raw doubles of the inputs named in `wrt`, in
        that order: {"tau": [N,na,K], "dv": [N,nv,K], "f": [N,24,K], "status": [N]}, K the total size of those inputs.
        One :meth:`tick_jvp` call with shared identity directions."""
        dims = dict(self._ref_dims, q=self.nq, v=self.nv)
        wrt = tuple(wrt)
        if not wrt or set(wrt) - set(dims) or len(set(wrt)) != len(wrt):
            raise ValueError(f"tick_jacobian: wrt must name distinct inputs among {tuple(dims)}, got {wrt}")
        K = sum(dims[k] for k in wrt)
        eye = torch.eye(K, dtype=torch.float64, device=self.device)
        tangents, c = {}, 0
        for k in wrt:
            tangents[k] = eye[:, c:c + dims[k]].contiguous()
            c += dims[k]
        o = self.tick_jvp(q, v, contact_mask, refs, tangents)
        return {"tau": o["tau"].transpose(1, 2).contiguous(), "dv": o["dv"].transpose(1, 2).contiguous(),
                "f": o["f"].transpose(1, 2).contiguous(), "status": o["status"]}

    def ci_row(self, block: int, side: int, i: int) -> int:
        return int(self.lib.tsidb_ci_row(self.h, block, side, i))

    def debug_terms(self, env: int, n_contacts: int) -> Dict[str, np.ndarray]:
        """M, nle, JF (LF, RF sole Jacobians, LOCAL), the dv block of the Hessian and the dv part of the gradient that the
        dynamics kernel produced for `env` in the last tick (tsidb_debug_terms; parity tests)."""
        nv = self.nv
        out = {"M": np.empty((nv, nv)), "nle": np.empty(nv), "JF": np.empty((2, 6, nv)), "H": np.empty((nv, nv)), "g": np.empty(nv)}
        check(self.lib.tsidb_debug_terms(self.h, env, n_contacts, *(out[k].ctypes.data for k in ("M", "nle", "JF", "H", "g"))),
              "tsidb_debug_terms")
        return out

    def launch_count(self) -> int:
        return int(self.lib.tsidb_launch_count(self.h))

    KERNEL_NAMES = ("class_sort", "dynamics", "eliminate", "j2", "activeset")

    def set_sched_hint(self, on: bool) -> None:
        """Longest-first order of the envs inside a contact class by the previous tick's iteration counts (tsidb.h)."""
        check(self.lib.tsidb_set_sched_hint(self.h, int(on)), "tsidb_set_sched_hint")

    def set_timing(self, on: bool) -> None:
        check(self.lib.tsidb_set_timing(self.h, int(on)), "tsidb_set_timing")

    def last_tick_ms(self) -> Dict[str, float]:
        """CUDA-event durations of the kernels of the last tick (needs set_timing(True))."""
        ms = (C.c_float * 5)()
        check(self.lib.tsidb_last_tick_ms(self.h, ms), "tsidb_last_tick_ms")
        return {k: float(ms[i]) for i, k in enumerate(self.KERNEL_NAMES)}


class _QpLayer(torch.autograd.Function):
    """forward: TsidEngine.qp_solve; backward: TsidEngine.qp_grad (the tensors of `keys` are the problem's float parts)."""

    @staticmethod
    def forward(ctx, engine, sizes, keys, *tensors):
        problem = dict(zip(keys, tensors), sizes=sizes)
        sol = engine.qp_solve(problem)
        ctx.engine, ctx.keys = engine, keys
        ctx.mark_non_differentiable(sol["status"], sol["iters"], sol["active"])
        ctx.save_for_backward(sizes, *tensors, sol["x"], sol["status"], sol["active"], sol["lambda"], sol["lambda_eq"])
        outs = (sol["x"], sol["lambda"], sol["lambda_eq"], sol["status"], sol["iters"], sol["active"])
        return outs + ((sol["tau"],) if "tau" in sol else ())

    @staticmethod
    @once_differentiable
    def backward(ctx, *grad_outs):
        saved = ctx.saved_tensors
        nk = len(ctx.keys)
        problem = dict(zip(ctx.keys, saved[1:1 + nk]), sizes=saved[0])
        sol = dict(zip(("x", "status", "active", "lambda", "lambda_eq"), saved[1 + nk:]))
        names = ("x", "lambda", "lambda_eq", None, None, None, "tau")
        grads = {k: g.contiguous() for k, g in zip(names, grad_outs) if k is not None and g is not None}
        parts = tuple(k for i, k in enumerate(ctx.keys) if ctx.needs_input_grad[3 + i])
        out = ctx.engine.qp_grad(problem, sol, grads, parts)
        return (None, None, None) + tuple(out.get(k) for k in ctx.keys)


class _TickLayer(torch.autograd.Function):
    """forward: TsidEngine.problem_data -> qp_solve; backward: qp_grad (g, ce0; every part when q or v needs a gradient)
    -> refs_grad and state_grad (the tensors of `keys` are the caller's reference tensors)."""

    SOL = ("x", "status", "active", "lambda", "lambda_eq")
    PROB = TsidEngine.PROBLEM_PARTS + TsidEngine.ACTUATION_PARTS + ("sizes",)

    @staticmethod
    def _feet(mask: Optional[torch.Tensor], n: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
        """[N,1] bools: LF in contact, RF in contact (no mask: double support)."""
        if mask is None:
            t = torch.ones((n, 1), dtype=torch.bool, device=device)
            return t, t
        m = mask.to(torch.int32).unsqueeze(1)
        return (m & 1) != 0, (m & 2) != 0

    @staticmethod
    def forward(ctx, engine, q, v, mask, keys, gkeys, *tensors):
        tensors, gtensors = tensors[:len(keys)], tensors[len(keys):]
        if gkeys:
            engine.set_gains(dict(zip(gkeys, gtensors)))
        ctx.gains_version, ctx.gkeys = engine._gains_version, gkeys
        refs = dict(zip(keys, tensors))
        prob = engine.problem_data(q, v, mask, refs, parts=engine.PROBLEM_PARTS + engine.ACTUATION_PARTS)
        sol = engine.qp_solve(prob)
        n, nv = q.shape[0], engine.nv
        x = sol["x"]
        lf, rf = _TickLayer._feet(mask, n, x.device)
        zero = torch.zeros((), dtype=x.dtype, device=x.device)
        s0, s1 = x[:, nv:nv + 12], x[:, nv + 12:nv + 24]  # force slot 0: LF if in contact, else RF; slot 1: RF
        f = torch.cat([torch.where(lf, s0, zero), torch.where(rf, torch.where(lf, s1, s0), zero)], dim=1)
        ctx.engine, ctx.keys = engine, keys
        ctx.mark_non_differentiable(sol["status"], sol["iters"])
        ctx.save_for_backward(q, v, mask, *(sol[k] for k in _TickLayer.SOL), *(prob[k] for k in _TickLayer.PROB), *tensors)
        ctx.save_for_forward(q, v, mask, *(sol[k] for k in _TickLayer.SOL), *(prob[k] for k in _TickLayer.PROB), *tensors)
        return sol["tau"], x[:, :nv].contiguous(), f, sol["status"], sol["iters"]

    @staticmethod
    def split_x(x: torch.Tensor, mask: Optional[torch.Tensor], nv: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """x [N,D,n_max] -> dv [N,D,nv], f [N,D,24] in the tick's fixed slots (LF 0..11, RF 12..23), as forward maps x."""
        n = x.shape[0]
        lf, rf = (t.unsqueeze(2) for t in _TickLayer._feet(mask, n, x.device))
        zero = torch.zeros((), dtype=x.dtype, device=x.device)
        s0, s1 = x[:, :, nv:nv + 12], x[:, :, nv + 12:nv + 24]
        f = torch.cat([torch.where(lf, s0, zero), torch.where(rf, torch.where(lf, s1, s0), zero)], dim=2)
        return x[:, :, :nv].contiguous(), f

    @staticmethod
    def jvp(ctx, _gengine, tq, tv, _gmask, _gkeys, _ggkeys, *trefs):
        """forward mode: tsidb_tick_jvp with one per-env direction, the inputs' tangents (None = zero)."""
        if any(t is not None for t in trefs[len(ctx.keys):]):
            raise NotImplementedError("tick_layer: forward mode in the gains and weights is not implemented "
                                      "(reverse mode is: tick_layer's backward pass, gains_grad)")
        trefs = trefs[:len(ctx.keys)]
        e, ns, npb = ctx.engine, len(_TickLayer.SOL), len(_TickLayer.PROB)
        q, v, mask, *rest = ctx.saved_tensors
        sol, prob, tensors = dict(zip(_TickLayer.SOL, rest[:ns])), dict(zip(_TickLayer.PROB, rest[ns:ns + npb])), rest[ns + npb:]
        tangents = {k: t for k, t in (("q", tq), ("v", tv)) if t is not None}
        tangents.update({k: t for k, t in zip(ctx.keys, trefs) if t is not None})
        if not tangents:
            return None, None, None, None, None
        tangents = {k: t.contiguous().unsqueeze(1) for k, t in tangents.items()}
        o = e.tick_jvp(q, v, mask, dict(zip(ctx.keys, tensors)), tangents, prob, sol)
        return o["tau"][:, 0], o["dv"][:, 0], o["f"][:, 0], None, None

    @staticmethod
    @once_differentiable
    def backward(ctx, gtau, gdv, gf, _gstatus, _giters):
        e, ns, npb = ctx.engine, len(_TickLayer.SOL), len(_TickLayer.PROB)
        if e._gains_version != ctx.gains_version:
            raise RuntimeError("tick_layer: set_gains ran after the forward pass; its gradients would be those of other "
                               "gains and weights")
        q, v, mask, *rest = ctx.saved_tensors
        sol, prob, tensors = dict(zip(_TickLayer.SOL, rest[:ns])), dict(zip(_TickLayer.PROB, rest[ns:ns + npb])), rest[ns + npb:]
        nk, none = len(ctx.keys), (None,) * (6 + len(ctx.keys) + len(ctx.gkeys))
        parts = tuple(k for i, k in enumerate(ctx.keys) if ctx.needs_input_grad[6 + i])
        gparts = tuple(k for i, k in enumerate(ctx.gkeys) if ctx.needs_input_grad[6 + nk + i])
        sparts = tuple(k for k, i in (("q", 1), ("v", 2)) if ctx.needs_input_grad[i])
        if not parts and not sparts and not gparts:
            return none
        n, nv = q.shape[0], e.nv
        grads = {}
        if gdv is not None or gf is not None:
            gx = torch.zeros_like(sol["x"])
            if gdv is not None:
                gx[:, :nv] = gdv
            if gf is not None:
                lf, rf = _TickLayer._feet(mask, n, gx.device)
                zero = torch.zeros((), dtype=gx.dtype, device=gx.device)
                gx[:, nv:nv + 12] = torch.where(lf, gf[:, :12], torch.where(rf, gf[:, 12:], zero))
                gx[:, nv + 12:nv + 24] = torch.where(lf & rf, gf[:, 12:], zero)
            grads["x"] = gx
        if gtau is not None:
            grads["tau"] = gtau.contiguous()
        if not grads:
            return none
        refs = dict(zip(ctx.keys, tensors[:nk]))
        qparts = e.PROBLEM_PARTS + e.ACTUATION_PARTS if sparts else (("H", "g", "ce0") if gparts else ("g", "ce0"))
        qg = e.qp_grad(prob, sol, grads, qparts)
        out = e.refs_grad(q, v, mask, refs, qg["g"], qg["ce0"], parts) if parts else {}
        st = e.state_grad(q, v, mask, refs, qg, sparts) if sparts else {}
        gg = {k: t.sum(0) for k, t in e.gains_grad(q, v, mask, refs, qg, gparts).items()} if gparts else {}
        return (None, st.get("q"), st.get("v"), None, None, None) + tuple(out.get(k) for k in ctx.keys) + \
            tuple(gg.get(k) for k in ctx.gkeys)


def fp64_peak_tflops(device: int = 0) -> float:
    lib = load_library()
    out = C.c_double(0.0)
    check(lib.tsidb_fp64_peak(device, C.byref(out)), "tsidb_fp64_peak")
    return float(out.value)
