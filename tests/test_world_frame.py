"""Where the robot stands: the tick and its derivatives away from the world origin.

Batched users place env i at its own grid offset, hundreds of metres out, and walking envs drift.  Under a translation of
the base and of every reference position by `off`, exact arithmetic leaves tau, dv, f, the status, the working sets, the
whole QP export and every gradient and tangent unchanged and moves the CoM and sole placements by exactly `off`.  The
kernels take their spatial algebra relative to each env's base position, so this holds to rounding at any distance; taken
at the world origin, the rounding of M, h and J grew with the square of the distance (DESIGN.md, reference point).

On the host emulator: the translation sweep of the tick (against the unshifted run and the 80-bit oracle at the shifted
inputs), of the export and of refs_grad, state_grad, gains_grad and tick_jvp (against the unshifted run); the sign of
the base quaternion; the heading of the whole scene against the 80-bit oracle.  On the GPU: the sweep through both tick
paths and the derivative kernels, and a 65536-env batch on a 256 x 256 grid with random headings against the oracle."""
import os

import numpy as np
import pytest

from common import TOL, assert_parity, bits_to_rows, canonical_active, compare_outputs, rel_err, setup, words_to_bits
from emu_gains_grad import EmuGainsGrad
from emu_py import Emu
from emu_qp import EmuProblemTA, emu_qp_solve
from emu_refs_grad import REF_KEYS, EmuRefsGrad
from emu_state_grad import EmuStateGrad
from emu_tick_jvp import EmuTickJvp
from test_gains_grad import _weights as _gains_weights
from test_refs_grad import TIGHT, _controller, _dev, live  # noqa: F401  (the fixture closes the engines)
from test_refs_grad import _weights as _refs_weights
from test_state_grad import _strides
from test_state_grad import _weights as _state_weights
from tsid_control_b200 import synth

DISTANCES = (0.0, 1.0, 10.0, 100.0, 1000.0, 10000.0)
STEP = {"v1": (0.3, 0.2, 0.2, 0.5), "v0": (0.1, 0.1275, 0.05, 0.7)}
POSITIONS = ("com", "foot_lf", "foot_rf", "contact_lf", "contact_rf")  # references whose first three entries are a point
QP_PARTS = ("H", "g", "CE", "ce0", "CI", "ci0", "TA", "ta0")
BIG = 1e9  # the export's +-1e10 bounds of the joint-bound rows
# Bars between runs whose inputs differ by their rounding (a translated batch against the batch at d = 0).  robot/v1: the
# parity bar.  The legacy conf (fMin = 0, cond(H) ~ 1e8) amplifies the last bits of its data: fp64 is only good to
# 1e-8 .. 1e-7 on its QP (assert_parity grants the oracle's own distance to the exact answer, 2e-7), so two fp64 runs of
# the same problem rounded differently are held to 1e-7, and tick_jvp's tangents, which solve with the same factors, to
# ten times their bar against the emulator.
SAME = {"v1": TOL, "v0": 1e-7}
JVP_SAME = {"v1": 1e-9, "v0": 1e-8}


def offset(d):
    """The translation of the sweep at distance scale d: (d, -0.7 d, 0)."""
    return np.array([d, -0.7 * d, 0.0])


def translated(q, refs, off):
    """The same batch with the base position and every reference position moved by `off` ([3] or per env [N,3])."""
    q = q.copy()
    q[:, :3] += off
    refs = {k: a.copy() for k, a in refs.items()}
    for k in POSITIONS:
        refs[k][:, :3] += off
    return q, refs


def _rz(psi):
    c, s = np.cos(psi), np.sin(psi)
    R = np.zeros(np.shape(psi) + (3, 3))
    R[..., 0, 0], R[..., 0, 1], R[..., 1, 0], R[..., 1, 1], R[..., 2, 2] = c, -s, s, c, 1.0
    return R


def yawed(q, refs, psi):
    """The whole scene turned about the world's vertical axis by psi (scalar or per env [N]).  The base position and
    orientation turn; v (the base twist in the base frame) and the joints do not.  Of the references (oracle/tsid_oracle.c:
    the CoM task's pos, vel, acc; an SE3 task's placement, and its velocity and acceleration, which the law maps with
    R_foot^T) everything is a world vector or a world orientation except the posture."""
    n = q.shape[0]
    psi = np.broadcast_to(np.asarray(psi, np.float64), (n,))
    R = _rz(psi)
    rot = lambda x: np.einsum("nij,nj->ni", R, x)  # noqa: E731
    q = q.copy()
    q[:, :3] = rot(q[:, :3])
    qz = np.stack([np.zeros(n), np.zeros(n), np.sin(psi / 2), np.cos(psi / 2)], axis=1)
    q[:, 3:7] = synth.quat_mul(qz, q[:, 3:7])
    out = {k: a.copy() for k, a in refs.items()}
    for k in ("com",):
        for o in (0, 3, 6):
            out[k][:, o:o + 3] = rot(refs[k][:, o:o + 3])
    for k in ("foot_lf", "foot_rf", "contact_lf", "contact_rf"):
        a = refs[k]
        out[k][:, :3] = rot(a[:, :3])
        Rr = a[:, 3:12].reshape(n, 3, 3).transpose(0, 2, 1)  # column-major
        out[k][:, 3:12] = (R @ Rr).transpose(0, 2, 1).reshape(n, 9)
        for o in range(12, a.shape[1], 3):
            out[k][:, o:o + 3] = rot(a[:, o:o + 3])
    return q, out


def _batch(kind, n, seed, overrides=()):
    """n walking envs, the contact masks cycling through double support, LF, RF and flight."""
    s = setup(kind, overrides=tuple(overrides))
    q, v = synth.random_states(s["q0"], n, seed)
    _, refs = synth.walking_batch(s["refs"], n, seed, *STEP[kind], float(s["refs"]["com"][2]))
    mask = np.array([3, 1, 2, 0] * ((n + 3) // 4), np.uint8)[:n]
    return s, q, v, mask, refs


def _canon(na, nv, words):
    return canonical_active(bits_to_rows(na, nv, words_to_bits(words)))


def assert_same_tick(a, b, na, nv, what, bar=TOL):
    """Two tick outputs of the same problem (b the reference): status equal, tau, dv and the contact wrenches within `bar`
    (the parity bar by default), corner forces within the force bar, working sets equal after canonicalising degenerate
    corners."""
    assert np.array_equal(a["status"], b["status"]), what
    ok = b["status"] == 0
    err = {k: rel_err(a[k][ok], b[k][ok]) for k in ("tau", "ddq", "wrench")}
    assert all(e <= bar for e in err.values()), (what, err)
    assert rel_err(a["f"][ok], b["f"][ok]) <= 1e-4, what
    for i in np.where(ok)[0]:
        assert _canon(na, nv, a["active_set"][:, i]) == _canon(na, nv, b["active_set"][:, i]), (what, int(i))
    return err


def _emu_tick(emu, q, v, mask, refs):
    out = emu.tick(q, v, mask, refs)
    out["active_set"], out["lam"], out["lam_row"] = out["active"], out["lambda"], out["lambda_row"]
    return out


def assert_aux_moved(a, b, off, what):
    """a: the aux outputs (or kinematics) at the translated input, b: at the original one.  The CoM and the soles move by
    `off`, their orientations, the CoM velocity and acceleration do not move, all up to the rounding of the world
    coordinates themselves: 1e-15 (1 + |off|), a few units in the last place of the offset."""
    off = np.broadcast_to(off, a["com"][:, :3].shape)
    bar = 1e-15 * (1.0 + np.abs(off).max(axis=1, keepdims=True))
    shift = {"com": np.concatenate([off, np.zeros_like(off), np.zeros_like(off)], axis=1),
             "foot_lf": np.concatenate([off, np.zeros((len(off), 9))], axis=1)}
    shift["foot_rf"] = shift["foot_lf"]
    for k, sh in shift.items():
        err = np.abs(a[k] - sh - b[k])
        assert (err <= bar).all(), (what, k, float(err.max()))


# ------------------------------------------------------------------ CPU: the kernel header on the host emulator
@pytest.mark.parametrize("kind,overrides", [("v1", ()), ("v0", ()), ("v1", TIGHT)])
def test_emulated_tick_is_translation_invariant(kind, overrides):
    """32 walking envs (every contact mask) translated by (d, -0.7 d, 0), d up to 10 km: the tick against the unshifted
    tick (SAME) and against the oracle at the translated inputs (assert_parity: 1e-8 against the 80-bit build), the aux
    CoM and soles moved by the offset.  The tight conf puts actuation and joint-velocity rows in the working sets."""
    n = 32
    s, q, v, mask, refs = _batch(kind, n, 5, overrides)
    na, nv = s["oracle"].na, s["oracle"].nv
    emu = Emu(s["cm"], s["cc"], s["refs"])
    base = _emu_tick(emu, q, v, mask, refs)
    assert (base["status"] == 0).sum() >= n - 2
    print(f"\n{kind}{' tight' if overrides else ''}: d, tau/dv/wrench vs d=0, tau/dv/wrench vs the 80-bit oracle")
    for d in DISTANCES:
        off = offset(d)
        qd, rd = translated(q, refs, off)
        out = _emu_tick(emu, qd, v, mask, rd)
        same = assert_same_tick(out, base, na, nv, d, SAME[kind])
        assert_aux_moved(out, base, off, d)
        res, _ = compare_outputs(kind, qd, v, mask, rd, out, overrides=tuple(overrides))
        print(f"d {d:7.0f} m  " + " ".join(f"{same[k]:.1e}" for k in ("tau", "ddq", "wrench")) + "  " +
              " ".join(f"{res[k + '_truth']:.1e}" for k in ("tau", "ddq", "wrench")))
        assert_parity(res, kind)


def _export(s, q, v, mask, refs):
    return EmuProblemTA(s["cm"], s["cc"]).problem_ta(q, v, mask, refs)


def _export_err(a, b):
    """Per part, the worst env's max|a-b| / (1e-2 + max|b|) (test_problem_data's metric) over each env's own sizes; the
    sizes equal and the +-1e10 bounds exactly equal."""
    assert np.array_equal(a["sizes"], b["sizes"])
    worst = {}
    for i, (n, neq, nin) in enumerate(b["sizes"]):
        na = b["TA"].shape[1]
        lead = {"H": (n, n), "g": (n,), "CE": (neq, n), "ce0": (neq,), "CI": (nin, n), "ci0": (nin,), "TA": (na, n), "ta0": (na,)}
        for k, shp in lead.items():
            x, y = (m[k][i][tuple(slice(0, e) for e in shp)] for m in (a, b))
            if k == "ci0":
                big = np.abs(y) >= BIG
                assert np.array_equal(x[big], y[big])
                x, y = x[~big], y[~big]
            e = float(np.max(np.abs(x - y)) / (1e-2 + np.max(np.abs(y)))) if y.size else 0.0
            worst[k] = max(worst.get(k, 0.0), e)
    return worst


def _grad_err(a, b):
    """The worst env's max |a - b| over the parts, relative to the env's gradient norm in b."""
    norm = np.sqrt(sum((b[k].reshape(len(b[k]), -1) ** 2).sum(1) for k in b)) + 1e-300
    return float(max((np.abs(a[k] - b[k]).reshape(len(b[k]), -1).max(1) / norm).max() for k in b))


@pytest.mark.parametrize("kind", ["v1", "v0"])
def test_emulated_export_and_derivatives_are_translation_invariant(kind):
    """8 walking envs (two per contact mask) translated by (d, -0.7 d, 0), d up to 10 km, against the unshifted run: the
    export with TA, ta0 within 1e-10 (test_problem_data's metric and bar), refs_grad and state_grad within 1e-11 and
    gains_grad within 1e-10 of each env's gradient norm, tick_jvp's x' and tau' within JVP_SAME of each env's tangent
    norm (the bars at which the GPU kernels are held to the emulator; for the legacy conf's tangents see SAME)."""
    n = 8
    s, q, v, mask, refs = _batch(kind, n, 7)
    nv = s["oracle"].nv
    rg, sg = EmuRefsGrad(s["cm"], s["cc"], s["refs"]), EmuStateGrad(s["cm"], s["cc"], s["refs"])
    gg, jv = EmuGainsGrad(s["cm"], s["cc"], s["refs"]), EmuTickJvp(s["cm"], s["cc"], s["refs"])
    dg, dce0 = _refs_weights(n, nv, mask, 8)
    W = _state_weights(s["cc"], nv, mask, 9)
    dH, dg2, dce02 = _gains_weights(n, nv, mask, 10)
    rng = np.random.default_rng(11)
    dims = {"q": jv.nq, "v": jv.nv, "com": 9, "foot_lf": 24, "foot_rf": 24, "contact_lf": 12, "contact_rf": 12, "posture": jv.na}
    dirs = {k: rng.standard_normal((n, 2, m)) for k, m in dims.items()}

    def run(qq, rr):
        prob = _export(s, qq, v, mask, rr)
        sol = emu_qp_solve(prob, s["cc"].max_iter)
        return {"prob": prob,
                "refs": rg.refs_grad(qq, v, mask, rr, dg, dce0),
                "state": sg.state_grad(qq, v, mask, rr, W, _strides(s["cc"], nv)),
                "gains": {"g": gg.gains_grad(qq, v, mask, rr, dH, dg2, dce02)},
                "jvp": {k: o for k, o in jv.tick_jvp(qq, v, mask, rr, prob, sol, dirs).items() if k != "status"},
                "sol": sol}

    base = run(q, refs)
    assert (base["sol"]["status"] == 0).all()
    bars = {"refs": 1e-11, "state": 1e-11, "gains": 1e-10, "jvp": JVP_SAME[kind]}
    print(f"\n{kind}: d, export (worst part), refs_grad, state_grad, gains_grad, tick_jvp")
    for d in DISTANCES[1:]:
        out = run(*translated(q, refs, offset(d)))
        assert np.array_equal(out["sol"]["status"], base["sol"]["status"])
        ex = _export_err(out["prob"], base["prob"])
        errs = {k: _grad_err(out[k], base[k]) for k in bars}
        print(f"d {d:7.0f} m  {max(ex.values()):.1e}  " + " ".join(f"{errs[k]:.1e}" for k in bars))
        assert all(e < 1e-10 for e in ex.values()), (d, ex)
        assert all(errs[k] < bars[k] for k in bars), (d, errs)


@pytest.mark.parametrize("kind", ["v1", "v0"])
def test_emulated_quaternion_sign(kind):
    """q and q with the base quaternion negated are the same placement, and the kernels' rotation matrix is quadratic in
    the quaternion: the tick (tau, dv, f, status, iterations, working sets, aux), the export, refs_grad and gains_grad
    are bit-identical, state_grad's quaternion components flip their sign bit for bit and its other components do not
    move, and tick_jvp along a direction whose quaternion part is negated gives the same tangents."""
    n = 8
    s, q, v, mask, refs = _batch(kind, n, 13)
    nv = s["oracle"].nv
    qn = q.copy()
    qn[:, 3:7] = -qn[:, 3:7]
    emu = Emu(s["cm"], s["cc"], s["refs"])
    a, b = emu.tick(q, v, mask, refs), emu.tick(qn, v, mask, refs)
    for k in ("tau", "ddq", "f", "status", "iters", "active", "com", "foot_lf", "foot_rf", "wrench", "lambda", "lambda_row"):
        assert np.array_equal(a[k], b[k]), k
    pa, pb = _export(s, q, v, mask, refs), _export(s, qn, v, mask, refs)
    for k in QP_PARTS + ("sizes",):
        assert np.array_equal(pa[k], pb[k], equal_nan=True), k
    dg, dce0 = _refs_weights(n, nv, mask, 14)
    rg = EmuRefsGrad(s["cm"], s["cc"], s["refs"])
    ra, rb = rg.refs_grad(q, v, mask, refs, dg, dce0), rg.refs_grad(qn, v, mask, refs, dg, dce0)
    for k in REF_KEYS:
        assert np.array_equal(ra[k], rb[k]), k
    dH, dg2, dce02 = _gains_weights(n, nv, mask, 15)
    gg = EmuGainsGrad(s["cm"], s["cc"], s["refs"])
    assert np.array_equal(gg.gains_grad(q, v, mask, refs, dH, dg2, dce02), gg.gains_grad(qn, v, mask, refs, dH, dg2, dce02))
    W = _state_weights(s["cc"], nv, mask, 16)
    sg = EmuStateGrad(s["cm"], s["cc"], s["refs"])
    ga, gb = sg.state_grad(q, v, mask, refs, W, _strides(s["cc"], nv)), sg.state_grad(qn, v, mask, refs, W, _strides(s["cc"], nv))
    assert np.array_equal(ga["v"], gb["v"])
    assert np.array_equal(ga["q"][:, :3], gb["q"][:, :3]) and np.array_equal(ga["q"][:, 7:], gb["q"][:, 7:])
    assert np.array_equal(ga["q"][:, 3:7], -gb["q"][:, 3:7]) and np.abs(ga["q"][:, 3:7]).max() > 0
    sol = emu_qp_solve(pa, s["cc"].max_iter)
    jv = EmuTickJvp(s["cm"], s["cc"], s["refs"])
    rng = np.random.default_rng(17)
    dirs = {"q": rng.standard_normal((n, 2, jv.nq)), "v": rng.standard_normal((n, 2, jv.nv)),
            "com": rng.standard_normal((n, 2, 9))}
    dn = dict(dirs, q=dirs["q"].copy())
    dn["q"][:, :, 3:7] *= -1.0
    ja, jb = jv.tick_jvp(q, v, mask, refs, pa, sol, dirs), jv.tick_jvp(qn, v, mask, refs, pa, sol, dn)
    for k in ("x", "tau", "status"):
        assert np.array_equal(ja[k], jb[k], equal_nan=True), k


@pytest.mark.parametrize("psi", [np.pi / 2, np.pi, -2.5])
@pytest.mark.parametrize("kind", ["v1", "v0"])
def test_emulated_heading_against_the_oracle(kind, psi):
    """The whole scene yawed about the vertical axis, at the origin and translated by (1000, -700, 0) m: the CoM gains are
    per axis, so yaw is no invariance of the controller; the tick is held to the oracle at the yawed inputs with the
    parity rules (assert_parity)."""
    n = 64
    s, q, v, mask, refs = _batch(kind, n, 19)
    emu = Emu(s["cm"], s["cc"], s["refs"])
    for d in (0.0, 1000.0):
        qy, ry = translated(*yawed(q, refs, psi), offset(d))
        out = _emu_tick(emu, qy, v, mask, ry)
        res, _ = compare_outputs(kind, qy, v, mask, ry, out)
        print(f"\n{kind} yaw {psi:+.3f} at {d:.0f} m: vs 80-bit tau {res['tau_truth']:.1e} dv {res['ddq_truth']:.1e} "
              f"wrench {res['wrench_truth']:.1e}")
        assert_parity(res, kind)


# ------------------------------------------------------------------ GPU
def _gpu_tick(ctrl, q, v, mask, refs):
    from test_gpu_parity import _run

    return _run(ctrl, q, v, mask, refs)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("v1", 97), ("v1", 4100), ("v0", 97), ("v0", 4100)])
def test_tick_is_translation_invariant(kind, n, live):
    """The translation sweep through the single-launch kernel (97 envs) and the batched pipeline with its class sort
    (4100 envs: ragged, several persistent trips): every env against the GPU at d = 0 (SAME), the aux outputs and
    tsidb_kinematics (every env, equal to the tick's aux outputs) moved by the offset; 24 envs against the emulator at the
    translated inputs (parity bars)."""
    import torch

    s, q, v, mask, refs = _batch(kind, n, 23)
    na, nv = s["oracle"].na, s["oracle"].nv
    ctrl = _controller(kind, n)
    emu = Emu(s["cm"], s["cc"], s["refs"])
    idx = np.linspace(0, n - 1, 24).astype(int)
    def kinematics(qq):
        # in reversed env order: the call shares its output buffers with the tick's aux outputs of the same size, and an
        # env it did not write must not pass for one it did
        dev = lambda a: torch.as_tensor(a[::-1].copy(), device=ctrl.device)  # noqa: E731
        r = ctrl.engine.kinematics(dev(qq), dev(v))
        return dict(zip(("com", "foot_lf", "foot_rf"), (t.cpu().numpy()[::-1] for t in r)))

    base = _gpu_tick(ctrl, q, v, mask, refs)
    assert (base["status"] == 0).mean() > 0.9
    kin0 = kinematics(q)
    for d in DISTANCES:
        off = offset(d)
        qd, rd = translated(q, refs, off)
        out = _gpu_tick(ctrl, qd, v, mask, rd)
        same = assert_same_tick(out, base, na, nv, d, SAME[kind])
        aux = {"com": out["com"], "foot_lf": out["foot_lf"], "foot_rf": out["foot_rf"]}
        assert_aux_moved(aux, {"com": base["com"], "foot_lf": base["foot_lf"], "foot_rf": base["foot_rf"]}, off, d)
        kin = kinematics(qd)
        for k in aux:  # every env's kinematics equal the tick's own (one K1, another kernel)
            assert (np.abs(kin[k] - aux[k]) <= 1e-13 * (1.0 + np.abs(aux[k]))).all(), (d, k)
        assert_aux_moved(kin, kin0, off, d)
        ref = _emu_tick(emu, qd[idx], v[idx], mask[idx], {k: a[idx] for k, a in rd.items()})
        sub = {k: (a[:, idx] if k == "active_set" else a[idx]) for k, a in out.items() if a is not None and k in
               ("tau", "ddq", "f", "wrench", "status", "active_set")}
        emu_err = assert_same_tick(sub, ref, na, nv, d)
        print(f"\n{kind} n={n} at {d:.0f} m: vs d=0 " + " ".join(f"{same[k]:.1e}" for k in same) +
              "; vs emulator " + " ".join(f"{emu_err[k]:.1e}" for k in emu_err))


def _np(d):
    return {k: t.cpu().numpy() for k, t in d.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["v1", "v0"])
def test_export_and_derivatives_are_translation_invariant(kind, live):
    """The translation sweep through problem_data, refs_grad, state_grad, gains_grad and tick_jvp: 512 envs (every
    contact mask) against the GPU at d = 0 on every env and against the emulator at the translated inputs on 16 envs, at
    the bars the kernels' own GPU tests hold them to the emulator (export 1e-10 of test_problem_data's metric, refs_grad
    and state_grad 1e-11, gains_grad 1e-10 of each env's gradient norm, tick_jvp 1e-9 of each env's tangent norm; against
    d = 0 the legacy conf's tangents within JVP_SAME)."""
    from tsid_control_b200._capi import GAIN_FIELDS

    from test_gains_grad import COL

    n = 512
    s, q, v, mask, refs = _batch(kind, n, 29)
    nv = s["oracle"].nv
    e = _controller(kind, n).engine
    na = e.na
    dg, dce0 = _refs_weights(n, nv, mask, 30)
    W = _state_weights(s["cc"], nv, mask, 31)
    dH, dg2, dce02 = _gains_weights(n, nv, mask, 32)
    rng = np.random.default_rng(33)
    dims = {"q": e.nq, "v": e.nv, "com": 9, "foot_lf": 24, "foot_rf": 24, "contact_lf": 12, "contact_rf": 12, "posture": na}
    dirs = {k: rng.standard_normal((n, 1, m)) for k, m in dims.items()}
    used = [c for k, nf in GAIN_FIELDS for c in range(COL[k], COL[k] + (na if k in ("kp_posture", "kd_posture") else nf))]
    idx = np.linspace(0, n - 1, 16).astype(int)
    emus = (EmuRefsGrad(s["cm"], s["cc"], s["refs"]), EmuStateGrad(s["cm"], s["cc"], s["refs"]),
            EmuGainsGrad(s["cm"], s["cc"], s["refs"]), EmuTickJvp(s["cm"], s["cc"], s["refs"]))

    def gpu(qq, rr):
        qd, vd, md, rd, dgd, dcd, dHd, dg2d, dc2d = _dev(e, qq, v, mask, rr, dg, dce0, dH, dg2, dce02)
        prob = e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
        sol = e.qp_solve(prob)
        gains = e.gains_grad(qd, vd, md, rd, {"H": dHd, "g": dg2d, "ce0": dc2d})
        out = {"prob": _np(prob), "sol": _np(sol), "refs": _np(e.refs_grad(qd, vd, md, rd, dgd, dcd)),
               "state": _np(e.state_grad(qd, vd, md, rd, _dev(e, W)[0])),
               "gains": {"g": np.concatenate([gains[k].cpu().numpy() for k, _ in GAIN_FIELDS if k in gains], axis=1)},
               "jvp": {k: t.cpu().numpy() for k, t in e.tick_jvp(qd, vd, md, rd, _dev(e, dirs)[0], prob, sol).items()
                       if k != "status"}}
        return out

    def emulated(qq, rr, g):
        r = {k: a[idx] for k, a in rr.items()}
        rg, sg, gg, jv = emus
        P = {k: a[idx] for k, a in g["prob"].items()}
        S = {k: a[idx] for k, a in g["sol"].items()}
        return {"refs": rg.refs_grad(qq[idx], v[idx], mask[idx], r, dg[idx], dce0[idx]),
                "state": sg.state_grad(qq[idx], v[idx], mask[idx], r, {k: a[idx] for k, a in W.items()},
                                       tuple(W[k].shape[1] for k in ("H", "CE", "CI"))),
                "gains": {"g": gg.gains_grad(qq[idx], v[idx], mask[idx], r, dH[idx], dg2[idx], dce02[idx])[:, used]},
                "jvp": {k: o for k, o in jv.tick_jvp(qq[idx], v[idx], mask[idx], r, P, S, {k: a[idx] for k, a in dirs.items()})
                        .items() if k != "status"},
                "prob": _export(s, qq[idx], v[idx], mask[idx], r)}

    bars = {"refs": 1e-11, "state": 1e-11, "gains": 1e-10, "jvp": 1e-9}
    same = dict(bars, jvp=JVP_SAME[kind])
    base = gpu(q, refs)
    ok = (base["sol"]["status"] == 0)
    assert ok.mean() > 0.9
    for d in DISTANCES:
        qq, rr = translated(q, refs, offset(d))
        out = gpu(qq, rr)
        assert np.array_equal(out["sol"]["status"], base["sol"]["status"])
        ex = _export_err(out["prob"], base["prob"])
        errs = {k: _grad_err({kk: a[ok] for kk, a in out[k].items()}, {kk: a[ok] for kk, a in base[k].items()})
                for k in bars}
        emu = emulated(qq, rr, out)
        ex_e = _export_err({k: a[idx] for k, a in out["prob"].items()}, emu["prob"])
        errs_e = {k: _grad_err({kk: a[idx] for kk, a in out[k].items()}, emu[k]) for k in bars}
        print(f"\n{kind} at {d:.0f} m: vs d=0 export {max(ex.values()):.1e} " + " ".join(f"{k} {errs[k]:.1e}" for k in bars) +
              f"; vs emulator export {max(ex_e.values()):.1e} " + " ".join(f"{k} {errs_e[k]:.1e}" for k in bars))
        assert all(x < 1e-10 for x in ex.values()) and all(x < 1e-10 for x in ex_e.values()), (d, ex, ex_e)
        assert all(errs[k] < same[k] and errs_e[k] < bars[k] for k in bars), (d, errs, errs_e)


@pytest.mark.gpu
def test_grid_batch65536_with_random_headings_every_env_against_the_oracle(live):
    """65536 walking envs (the bench's inputs, seed 0) on a 256 x 256 grid at 2.5 m spacing centred on the origin (up to
    453 m out), each env's scene first turned about the vertical axis by its own random heading: tau, dv and f of every
    env against the oracle at those inputs with the parity rules (assert_parity), as for the same batch at the origin."""
    n = 65536
    s = setup("v1")
    q, v = synth.random_states(s["q0"], n, 0)
    mask, refs = synth.walking_batch(s["refs"], n, 0, *STEP["v1"], float(s["refs"]["com"][2]))
    psi = np.random.default_rng(37).uniform(-np.pi, np.pi, n)
    ix, iy = np.divmod(np.arange(n), 256)
    grid = np.stack([2.5 * (ix - 127.5), 2.5 * (iy - 127.5), np.zeros(n)], axis=1)
    qg, rg = translated(*yawed(q, refs, psi), grid)
    ctrl = _controller("v1", n)
    out = _gpu_tick(ctrl, qg, v, mask, rg)
    res, _ = compare_outputs("v1", qg, v, mask, rg, out, threads=max(8, os.cpu_count() or 8))
    print("\ngrid 65536: " + " ".join(f"{k}={x:.3g}" for k, x in res.items() if isinstance(x, (int, float))))
    assert_parity(res, "v1")
    assert res["n_optimal"] == n
