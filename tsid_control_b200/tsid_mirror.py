"""Small stand-ins for the `tsid` / `pinocchio` objects the reference scripts touch, backed by the
batched CUDA engine.  They keep the reference's call shapes so that the tick of ref:main.py:119-127

    HQPData = controller.formulation.computeProblemData(t, q, v)
    sol     = controller.solver.solve(HQPData)
    tau     = controller.formulation.getActuatorForces(sol)
    dv      = controller.formulation.getAccelerations(sol)

runs unchanged for one robot (numpy in/out), while `controller.compute(q, v, t)` is the batched
entry over torch tensors.  Nothing here does arithmetic of the tick on the CPU.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np
import torch


class SE3:
    """Minimal pin.SE3: .translation, .rotation, act(point)."""

    def __init__(self, R: np.ndarray, p: np.ndarray):
        self.rotation = np.asarray(R, dtype=np.float64).reshape(3, 3)
        self.translation = np.asarray(p, dtype=np.float64).reshape(3)

    @staticmethod
    def from_vec12(v12: np.ndarray) -> "SE3":
        v12 = np.asarray(v12, dtype=np.float64)
        return SE3(v12[3:].reshape(3, 3).T, v12[:3])

    def to_vec12(self) -> np.ndarray:
        return np.concatenate([self.translation, self.rotation.T.ravel()])

    def act(self, p) -> np.ndarray:
        return self.rotation @ np.asarray(p, dtype=np.float64) + self.translation

    def __repr__(self) -> str:
        return f"  R =\n{self.rotation}\n  p = {self.translation}\n"


class TrajectorySample:
    """tsid.TrajectorySample: value / derivative / second_derivative.  Arrays may be [k] (one robot)
    or [N,k] torch tensors (batched)."""

    def __init__(self, pos, vel=None, acc=None):
        self.pos = pos
        nd = 6 if (pos.shape[-1] == 12) else pos.shape[-1]
        zeros = (lambda: torch.zeros(pos.shape[:-1] + (nd,), dtype=pos.dtype, device=pos.device)) if isinstance(pos, torch.Tensor) \
            else (lambda: np.zeros(pos.shape[:-1] + (nd,)))
        self.vel = vel if vel is not None else zeros()
        self.acc = acc if acc is not None else zeros()

    def value(self):
        return self.pos

    def derivative(self):
        return self.vel

    def second_derivative(self):
        return self.acc


class TrajectorySE3Constant:
    def __init__(self, name: str, M: SE3):
        self.name = name
        self.M = M

    def setReference(self, M: SE3) -> None:
        self.M = M

    def computeNext(self) -> TrajectorySample:
        return TrajectorySample(self.M.to_vec12())


class TrajectoryEuclidianConstant:
    def __init__(self, name: str, ref: np.ndarray):
        self.name = name
        self.ref = np.array(ref, dtype=np.float64)

    def setReference(self, ref) -> None:
        self.ref = np.array(ref, dtype=np.float64)

    def computeNext(self) -> TrajectorySample:
        return TrajectorySample(self.ref.copy())


class Task:
    """Named handle of a task; setReference writes into the controller's reference table."""

    def __init__(self, ctrl, name: str, key: str):
        self._ctrl, self.name, self._key = ctrl, name, key

    def setReference(self, sample) -> None:
        self._ctrl._set_task_reference(self._key, sample)


class Contact(Task):
    def __init__(self, ctrl, name: str, key: str, foot: int, T: np.ndarray):
        super().__init__(ctrl, name, key)
        self.foot = foot
        self.getForceGeneratorMatrix = T  # the reference reads it as an attribute (ref:ctrl/WalkController.py:262)

    def setReference(self, M) -> None:
        v12 = M.to_vec12() if isinstance(M, SE3) else M
        self._ctrl._set_task_reference(self._key, TrajectorySample(v12))


class HQPData:
    """What formulation.computeProblemData returns: the state, the sizes and, read on first access, the assembled QP of
    the single-robot view in the reference's variable and row order (SolverHQuadProgFast's input):
    min 1/2 x'Hx + g'x  s.t.  CE x + ce0 = 0,  CI x + ci0 >= 0, x = [dv; f of the contacts in insertion order].
    The matrices are formed on the device at the first access of any of them (TsidEngine.problem_data), with the
    contacts of the computeProblemData call and the task references current at that access."""

    PARTS = ("H", "g", "CE", "ce0", "CI", "ci0")

    def __init__(self, t, q, v, sizes, formulation=None, contact_order=(), ci_order=()):
        self.t, self.q, self.v, self.sizes = t, q, v, sizes
        self._formulation, self._contact_order, self._ci_order = formulation, list(contact_order), list(ci_order)
        self._problem = None

    def __getattr__(self, name):
        if name in HQPData.PARTS and self.__dict__.get("_formulation") is not None:
            if self._problem is None:
                self._problem = self._formulation._problem(self)
            return self._problem[name]
        raise AttributeError(name)

    def print_all(self) -> None:
        n, neq, nin = self.sizes
        print(f"HQPData: 2 levels, {n} variables, {neq} equality rows, {nin} inequality rows (level 0)")


class HQPOutput:
    """tsid HQPOutput for one robot (numpy) — .status .x .iterations .activeSet."""

    def __init__(self, status, x, iterations, activeSet, raw):
        self.status, self.x, self.iterations, self.activeSet, self._raw = status, x, iterations, activeSet, raw


class Data:
    def __init__(self):
        self.com = None
        self.foot = [None, None]


class RobotWrapperMirror:
    def __init__(self, ctrl):
        self._c = ctrl
        self.nv, self.na, self.nq = ctrl.engine.nv, ctrl.engine.na, ctrl.engine.nq

    def model(self):
        return self._c.model

    def framePosition(self, data: Data, frame_id: int) -> SE3:
        return SE3.from_vec12(data.foot[frame_id])

    def com(self, data: Data) -> np.ndarray:
        return np.array(data.com[:3])

    def com_vel(self, data: Data) -> np.ndarray:
        return np.array(data.com[3:6])


class ModelMirror:
    """What the reference reads from pinocchio's Model (ref:main.py:70-77, ref:ctrl/WalkController.py:72,119,167,179)."""

    def __init__(self, compiled, frame_names):
        self.compiled = compiled
        self.nq, self.nv, self.njoints = compiled.nq, compiled.nv, compiled.nb + 1
        self.names = ["universe", "root_joint"] + list(compiled.joint_names)
        self.idx_qs = [0, 0] + [7 + i for i in range(compiled.na)]
        self.effortLimit = np.concatenate([np.zeros(6), compiled.effort])
        self.velocityLimit = np.concatenate([np.zeros(6), compiled.velocity])
        self.referenceConfigurations = {k: v.copy() for k, v in compiled.q_ref.items()}
        self._frames = list(frame_names)

    def getJointId(self, name: str) -> int:
        return self.names.index(name)

    def getFrameId(self, name: str) -> int:
        return self._frames.index(name)

    def existFrame(self, name: str) -> bool:
        return name in self._frames


class FormulationMirror:
    """InverseDynamicsFormulationAccForce stand-in for ONE robot view of the batched controller."""

    def __init__(self, ctrl):
        self._c = ctrl
        self._data = Data()
        self._pending: Optional[HQPData] = None

    # sizes as the reference's solver.resize(nVar, nEq, nIn) reads them (ref:ctrl/WalkController.py:187)
    @property
    def nVar(self) -> int:
        return self._c.engine.nv + 12 * len(self._c._contact_order)

    @property
    def nEq(self) -> int:
        return 6 + 6 * len(self._c._contact_order)

    @property
    def nIn(self) -> int:
        e = self._c.engine
        return 17 * len(self._c._contact_order) + (e.na if e.cc.use_torque_bounds else 0) + (e.nv if e.cc.use_joint_bounds else 0)

    def computeProblemData(self, t, q, v) -> HQPData:
        c = self._c
        qd = torch.as_tensor(np.asarray(q, dtype=np.float64).reshape(1, -1), device=c.engine.device)
        vd = torch.as_tensor(np.asarray(v, dtype=np.float64).reshape(1, -1), device=c.engine.device)
        com, lf, rf = c.engine.kinematics(qd, vd)
        self._data.com = com[0].cpu().numpy()
        self._data.foot = [lf[0].cpu().numpy(), rf[0].cpu().numpy()]
        self._pending = HQPData(t, qd, vd, (self.nVar, self.nEq, self.nIn), self, c._contact_order, c._ci_order)
        return self._pending

    def _problem(self, hqp: HQPData) -> Dict[str, np.ndarray]:
        """The exported QP of env 0 (compact order: contacts LF first, CI blocks [LF, RF, actuation, joint bounds]),
        permuted into the order of hqp's contacts and level-0 blocks."""
        c = self._c
        e = c.engine
        mask = sum(1 << f for f in hqp._contact_order)
        refs = {k: t[0:1].contiguous() for k, t in c.refs.items()}
        out = e.problem_data(hqp.q, hqp.v, torch.tensor([mask], dtype=torch.uint8, device=e.device), refs)
        P = {k: out[k][0].cpu().numpy() for k in HQPData.PARTS}
        nv, feet = e.nv, sorted(hqp._contact_order)
        var = list(range(nv))
        eq = list(range(6))
        for f in hqp._contact_order:
            k = feet.index(f)
            var += range(nv + 12 * k, nv + 12 * k + 12)
            eq += range(6 + 6 * k, 12 + 6 * k)
        rows = {0: 17, 1: 17, 2: e.na, 3: e.nv}
        off, start = 0, {}
        for blk in feet + [b for b in (2, 3) if b in hqp._ci_order]:
            start[blk] = off
            off += 2 * rows[blk]
        ci: List[int] = []
        for blk in hqp._ci_order:
            ci += range(start[blk], start[blk] + 2 * rows[blk])
        ix = np.ix_
        return {"H": P["H"][ix(var, var)], "g": P["g"][var], "CE": P["CE"][ix(eq, var)], "ce0": P["ce0"][eq],
                "CI": P["CI"][ix(ci, var)], "ci0": P["ci0"][ci]}

    def data(self) -> Data:
        return self._data

    def getActuatorForces(self, sol: HQPOutput) -> np.ndarray:
        return sol._raw["tau"].copy()

    def getAccelerations(self, sol: HQPOutput) -> np.ndarray:
        return sol._raw["ddq"].copy()

    def getContactForce(self, name: str, sol: HQPOutput) -> np.ndarray:
        foot = self._c._contact_foot(name)
        return sol._raw["f"][12 * foot:12 * foot + 12].copy()

    def removeRigidContact(self, name: str, transition_time: float = 0.0) -> bool:
        return self._c._remove_contact_by_name(name)

    def addRigidContact(self, contact: Contact, w_forceRef: float, w_motion: float = 1.0, level: int = 0) -> bool:
        return self._c._add_contact_by_name(contact.name)


class SolverMirror:
    def __init__(self, ctrl, name: str = "qp solver"):
        self._c, self.name = ctrl, name

    def resize(self, n: int, neq: int, nin: int) -> None:
        pass

    def solve(self, hqp: HQPData) -> HQPOutput:
        c = self._c
        out = c._tick(hqp.q, hqp.v, env_slice=slice(0, 1), aux=True)
        raw = {k: getattr(out, k)[0].cpu().numpy() for k in ("tau", "ddq", "f")}
        status = int(out.status[0].item())
        words = out.active_set[:, 0].cpu().numpy().astype(np.uint64)
        bits = [64 * w + b for w in range(3) for b in range(64) if (int(words[w]) >> b) & 1]
        x = np.concatenate([raw["ddq"]] + [raw["f"][12 * f:12 * f + 12] for f in c._contact_order])
        return HQPOutput(status, x, int(out.iters[0].item()), np.array(c._bits_to_reference_rows(bits)), raw)
