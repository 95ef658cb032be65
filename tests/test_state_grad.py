"""Differentiating with respect to the state (tsidb_state_grad / TsidEngine.state_grad / TsidEngine.tick_layer): the
adjoint of the whole QP export in q and v against central differences of the 80-bit oracle's dump of the same problem,
part by part, with layouts, defaults and an exact contact on the host emulator; on the GPU the kernel against the
emulator and the oracle, the autograd layer against gradcheck and differences through the GPU forward, a fit that
recovers a state, a two-tick closed loop, and the absence of side effects."""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from common import force_generator, setup
from emu_refs_grad import REF_KEYS
from emu_state_grad import PARTS, EmuStateGrad
from test_problem_data import canonical_orders
from tsid_control_b200 import synth

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tsid_control_b200", "csrc")
STEP = {"v1": (0.3, 0.2, 0.2, 0.5), "v0": (0.1, 0.1275, 0.05, 0.7)}
BIG = 1e10  # the export's clip of the joint-bound rows: such entries are constant


def _inputs(kind, n, seed, overrides=()):
    s = setup(kind, overrides=tuple(overrides))
    q, v = synth.random_states(s["q0"], n, seed)
    mask, refs = synth.walking_batch(s["refs"], n, seed, *STEP[kind], float(s["refs"]["com"][2]))
    return s, q, v, mask, refs


def _strides(cc, nv):
    na = nv - 6
    return nv + 24, 18, 2 * (34 + (na if cc.use_torque_bounds else 0) + (nv if cc.use_joint_bounds else 0))


def _sizes(cc, nv, m):
    nc = (int(m) & 1) + ((int(m) >> 1) & 1)
    na = nv - 6
    return nv + 12 * nc, 6 + 6 * nc, 2 * (17 * nc + (na if cc.use_torque_bounds else 0) + (nv if cc.use_joint_bounds else 0))


def _weights(cc, nv, masks, seed):
    """Random dL/d of every entry the export writes inside each env's (n, neq, nin); NaN everywhere else."""
    rng = np.random.default_rng(seed)
    nx, neqx, ninx = _strides(cc, nv)
    N, na = len(masks), nv - 6
    W = {"H": np.full((N, nx, nx), np.nan), "g": np.full((N, nx), np.nan), "CE": np.full((N, neqx, nx), np.nan),
         "ce0": np.full((N, neqx), np.nan), "CI": np.full((N, ninx, nx), np.nan), "ci0": np.full((N, ninx), np.nan),
         "TA": np.full((N, na, nx), np.nan), "ta0": np.full((N, na), np.nan)}
    for i, m in enumerate(masks):
        n, neq, nin = _sizes(cc, nv, m)
        W["H"][i, :n, :n] = rng.standard_normal((n, n))
        W["g"][i, :n] = rng.standard_normal(n)
        W["CE"][i, :neq, :n] = rng.standard_normal((neq, n))
        W["ce0"][i, :neq] = rng.standard_normal(neq)
        W["CI"][i, :nin, :n] = rng.standard_normal((nin, n))
        W["ci0"][i, :nin] = rng.standard_normal(nin)
        W["TA"][i, :, :n] = rng.standard_normal((na, n))
        W["ta0"][i] = rng.standard_normal(na)
    return W


def _unread_nan(W, cc, nv, masks):
    """A copy of W with NaN in every block inside an env's (n, neq, nin) that does not depend on the state, which the
    adjoint documents as unread: the force rows and columns of H, the force columns of g, the force columns of the contact
    rows of CE, the contact-force and joint-bound rows of CI, the contact-force rows and the base joint-bound rows of ci0."""
    W = {k: a.copy() for k, a in W.items()}
    na = nv - 6
    for i, m in enumerate(masks):
        n, neq, _ = _sizes(cc, nv, m)
        nc = (n - nv) // 12
        jb = 34 * nc + (2 * na if cc.use_torque_bounds else 0)
        W["H"][i, :n, nv:n] = np.nan
        W["H"][i, nv:n, :n] = np.nan
        W["g"][i, nv:n] = np.nan
        W["CE"][i, 6:neq, nv:n] = np.nan
        W["CI"][i, :34 * nc] = np.nan
        W["ci0"][i, :34 * nc] = np.nan
        if cc.use_joint_bounds:
            W["CI"][i, jb:jb + 2 * nv] = np.nan
            W["ci0"][i, jb:jb + 6] = np.nan
            W["ci0"][i, jb + nv:jb + nv + 6] = np.nan
    return W


class OracleStateLoss:
    """L_part(q, v) = <W_part, part> of one env from the 80-bit oracle's dump of its problem, in the export's order; TA and
    ta0 are built from the dump's M, nle and JF (TA = [M_a | -J_c,a^T], ta0 = h_a).  Entries clipped to +-1e10 are
    constant and left out."""

    def __init__(self, kind, overrides, refs, mask, W):
        s = setup(kind, "liboracle_ld.so", overrides=tuple(overrides))
        self.orc, self.T = s["oracle"], force_generator(s["cc"])
        self.refs, self.mask, self.W = refs, int(mask), W
        self.nv = self.orc.nv
        self.orders = canonical_orders(self.orc, self.mask)

    def parts(self, q, v):
        d = self.orc.tick(q, v, self.mask, self.refs, dump=True, orders=self.orders)["dump"]
        nv, na, n = self.nv, self.nv - 6, d["n"]
        feet = [f for f in (0, 1) if (self.mask >> f) & 1]
        TA = np.zeros((na, n))
        TA[:, :nv] = d["M"][6:, :nv]
        for s_, f in enumerate(feet):
            TA[:, nv + 12 * s_:nv + 12 * s_ + 12] = -(self.T.T @ d["JF"][f][:, 6:]).T
        d = dict(d, TA=TA, ta0=d["nle"][6:])
        out = {}
        for k in PARTS:
            b = np.asarray(d[k], np.float64)
            w = self.W[k][tuple(slice(0, m) for m in b.shape)]
            keep = np.abs(b) < BIG
            out[k] = float(np.sum(np.where(keep, w * b, 0.0)))
        return out

    def gradient(self, q, v, h=1e-5):
        """Central differences of every part's loss with respect to every raw component of q (quaternion included) and
        of v -> {part: (dq, dv)}."""
        nq, nv = len(q), len(v)
        fd = {k: (np.zeros(nq), np.zeros(nv)) for k in PARTS}
        for which, x, cnt in ((0, q, nq), (1, v, nv)):
            for j in range(cnt):
                xp, xm = x.copy(), x.copy()
                xp[j] += h
                xm[j] -= h
                lp = self.parts(xp, v) if which == 0 else self.parts(q, xp)
                lm = self.parts(xm, v) if which == 0 else self.parts(q, xm)
                for k in PARTS:
                    fd[k][which][j] = (lp[k] - lm[k]) / (2 * h)
        return fd


def _tangent(gq, q):
    """gq with its quaternion block projected onto the tangent space of the unit sphere at q's quaternion.  The tick and
    the oracle compute the same functions of a unit quaternion but extend them differently off the sphere (world-frame
    against joint-frame recursions), so their derivatives agree along the three rotation directions and not along the
    radial one; that one is checked against the emulated export itself (test_emulated_quaternion_radial_direction)."""
    u = q[3:7] / np.linalg.norm(q[3:7])
    out = np.array(gq, dtype=np.float64)
    out[3:7] -= u * float(u @ out[3:7])
    return out


def _rel_err(gq, gv, fq, fv, q):
    """max |adjoint - differences| / norm of the adjoint, q's quaternion block in the tangent directions."""
    norm = np.sqrt(float((gq ** 2).sum() + (gv ** 2).sum()))
    return max(float(np.abs(_tangent(gq, q) - _tangent(fq, q)).max()), float(np.abs(gv - fv).max())) / norm


# ------------------------------------------------------------------ CPU: the kernel bodies on the host emulator
@pytest.mark.parametrize("kind", ["v1", "v0"])
@pytest.mark.parametrize("maskval", [3, 1, 2, 0])
def test_emulated_state_grad_matches_oracle_differences(kind, maskval):
    """Every raw component of q (the quaternion in its three rotation directions, see _tangent) and of v, two walking
    envs per contact mask: the emulated adjoint of all eight parts together, and of each part alone (the others NULL),
    against central differences (h = 1e-5) of the 80-bit oracle's dump, with NaN everywhere outside the entries the
    export writes.  Measured: at most ~3e-9 of the gradient's norm (the differences' own truncation and rounding); the
    bar is 1e-8."""
    n = 2
    s, q, v, _, refs = _inputs(kind, n, 171 + maskval)
    mask = np.full(n, maskval, np.uint8)
    emu = EmuStateGrad(s["cm"], s["cc"], s["refs"])
    st = _strides(s["cc"], emu.nv)
    W = _weights(s["cc"], emu.nv, mask, 172)
    G = emu.state_grad(q, v, mask, refs, W, st)
    alone = {k: emu.state_grad(q, v, mask, refs, {k: W[k]}, st) for k in PARTS}
    worst, worst_part = 0.0, 0.0
    for i in range(n):
        r = {k: a[i].copy() for k, a in refs.items()}
        fd = OracleStateLoss(kind, (), r, maskval, {k: a[i] for k, a in W.items()}).gradient(q[i], v[i])
        fq, fv = sum(fd[k][0] for k in PARTS), sum(fd[k][1] for k in PARTS)
        worst = max(worst, _rel_err(G["q"][i], G["v"][i], fq, fv, q[i]))
        norm = np.sqrt(float((G["q"][i] ** 2).sum() + (G["v"][i] ** 2).sum()))
        for k in PARTS:
            e = max(float(np.abs(_tangent(alone[k]["q"][i], q[i]) - _tangent(fd[k][0], q[i])).max()),
                    float(np.abs(alone[k]["v"][i] - fd[k][1]).max())) / norm
            worst_part = max(worst_part, e)
    print(f"\nemulated state_grad vs 80-bit central differences ({kind}, mask {maskval}): all parts {worst:.1e}, "
          f"single parts {worst_part:.1e} of the norm")
    assert worst < 1e-8 and worst_part < 1e-8


@pytest.mark.parametrize("kind", ["v1", "v0"])
def test_emulated_unread_blocks_may_hold_nan(kind):
    """Every contact mask: NaN in every block the adjoint documents as unread (constant blocks inside the env's sizes,
    _unread_nan) gives the same gradient, bit for bit, as random weights there."""
    n = 4
    s, q, v, _, refs = _inputs(kind, n, 161)
    mask = np.array([3, 1, 2, 0], np.uint8)
    emu = EmuStateGrad(s["cm"], s["cc"], s["refs"])
    st = _strides(s["cc"], emu.nv)
    W = _weights(s["cc"], emu.nv, mask, 162)
    a = emu.state_grad(q, v, mask, refs, W, st)
    b = emu.state_grad(q, v, mask, refs, _unread_nan(W, s["cc"], emu.nv, mask), st)
    for k in ("q", "v"):
        assert np.isfinite(b[k]).all() and np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("kind,maskval", [("v1", 3), ("v0", 1)])
def test_emulated_quaternion_radial_direction(kind, maskval):
    """The gradient is taken in the raw doubles of q: along the quaternion itself (the direction the oracle's
    differences leave out, see _tangent) the adjoint of all eight parts matches central differences (h = 1e-6) of the
    emulated export, which runs the tick's own quat -> R formula."""
    import ctypes as C

    from emu_problem import EmuProblem
    from emu_py import TickArgs
    from tsid_control_b200._capi import TsidbProblemOut

    n = 2
    s, q, v, _, refs = _inputs(kind, n, 181)
    mask = np.full(n, maskval, np.uint8)
    emu = EmuStateGrad(s["cm"], s["cc"], s["refs"])
    st = _strides(s["cc"], emu.nv)
    W = _weights(s["cc"], emu.nv, mask, 182)
    G = emu.state_grad(q, v, mask, refs, W, st)
    ep = EmuProblem(s["cm"], s["cc"])

    def loss(qq):
        """The emulated export of all eight parts (EmuProblem's call with TA and ta0 added) against W."""
        out = {k: np.full(a.shape, np.nan) for k, a in W.items()}
        out["sizes"] = np.full((n, 3), -1, np.int32)
        keep = [np.ascontiguousarray(qq), np.ascontiguousarray(v), np.ascontiguousarray(mask)]
        arrs = {k: np.ascontiguousarray(refs[k], dtype=np.float64) for k in REF_KEYS}
        a = TickArgs()
        a.n_envs, a.layout, a.slot = n, 0, 0
        a.q, a.v, a.mask = (x.ctypes.data for x in keep)
        a.r_com, a.r_posture = arrs["com"].ctypes.data, arrs["posture"].ctypes.data
        a.r_foot[0], a.r_foot[1] = arrs["foot_lf"].ctypes.data, arrs["foot_rf"].ctypes.data
        a.r_contact[0], a.r_contact[1] = arrs["contact_lf"].ctypes.data, arrs["contact_rf"].ctypes.data
        po = TsidbProblemOut(**{k: x.ctypes.data for k, x in out.items()})
        assert ep.lib.emu_problem(C.byref(a), C.byref(po)) == 0
        tot = np.zeros(n)
        for k in PARTS:
            body = np.where(np.isnan(W[k]) | (np.abs(out[k]) >= BIG), 0.0, W[k] * out[k])
            tot += body.reshape(n, -1).sum(axis=1)
        return tot

    d = np.zeros_like(q)
    d[:, 3:7] = q[:, 3:7]
    h = 1e-6
    fd = (loss(q + h * d) - loss(q - h * d)) / (2 * h)
    ad = (G["q"] * d).sum(axis=1)
    norm = np.sqrt((G["q"] ** 2).sum(axis=1) + (G["v"] ** 2).sum(axis=1))
    err = float((np.abs(fd - ad) / norm).max())
    print(f"\nradial quaternion direction ({kind}): adjoint vs emulated differences {err:.1e} of the norm")
    assert err < 1e-7


def test_emulated_layouts_defaults_and_exact_contact():
    """Layout 1 gives the transpose of layout 0 bit for bit; references left out give the gradient at the defaults;
    NULL parts count as zero; a contact reference equal to the sole placement the kernel computes (theta = 0 exactly)
    gives a finite gradient equal to its interior limit and to the oracle's differences."""
    n = 4
    s, q, v, _, refs = _inputs("v1", n, 191)
    mask = np.array([3, 1, 2, 0], np.uint8)
    emu = EmuStateGrad(s["cm"], s["cc"], s["refs"])
    st = _strides(s["cc"], emu.nv)
    W = _weights(s["cc"], emu.nv, mask, 192)
    g0 = emu.state_grad(q, v, mask, refs, W, st)
    g1 = emu.state_grad(q, v, mask, refs, W, st, layout=1)
    for k in ("q", "v"):
        assert np.array_equal(g0[k], g1[k]), k
        assert np.isfinite(g0[k]).all()
    tiled = {k: np.tile(s["refs"][k], (n, 1)) for k in REF_KEYS}
    a = emu.state_grad(q, v, mask, {}, W, st)
    b = emu.state_grad(q, v, mask, tiled, W, st)
    for k in ("q", "v"):
        assert np.array_equal(a[k], b[k]), k
    z = emu.state_grad(q, v, mask, refs, {}, st)
    assert not z["q"].any() and not z["v"].any()
    only_q = emu.state_grad(q, v, mask, refs, W, st, parts=("q",))
    assert set(only_q) == {"q"} and np.array_equal(only_q["q"], g0["q"])

    # exact contact: the LF contact reference placed on the sole as the kernel's own K1 computes it (the emulated
    # kinematics), on an env where E = Rf^T R_ref then has trace >= 3 in the kernel's arithmetic, so log6 takes theta = 0
    # exactly; then moved by 1e-9 in rotation
    from emu_py import Emu

    m = 3
    feet = Emu(s["cm"], s["cc"], s["refs"]).tick(q, v, np.full(n, m, np.uint8), refs, kin_only=True)["foot_lf"]

    def trace_e(pl):
        Rf = pl[3:12].reshape(3, 3).T  # row-major, as the kernel keeps it
        Rr = pl[3:12].reshape(3, 3).T
        e = [Rf[0, c] * Rr[0, c] + Rf[1, c] * Rr[1, c] + Rf[2, c] * Rr[2, c] for c in range(3)]
        return (e[0] + e[1]) + e[2]

    exact = [j for j in range(n) if trace_e(feet[j]) >= 3.0]
    assert exact, [trace_e(f) - 3.0 for f in feet]
    i = exact[0]
    placed = [feet[i]]
    r = {k: x[i:i + 1].copy() for k, x in refs.items()}
    r["contact_lf"][0] = placed[0]
    Wi = _weights(s["cc"], emu.nv, [m], 193)
    mi = np.array([m], np.uint8)
    G = emu.state_grad(q[i:i + 1], v[i:i + 1], mi, r, Wi, st)
    assert np.isfinite(G["q"]).all() and np.isfinite(G["v"]).all()
    w = np.array([0.3, -0.2, 0.5]) * 1e-9
    K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    R = placed[0][3:12].reshape(3, 3).T @ (np.eye(3) + K)
    r1 = {k: x.copy() for k, x in r.items()}
    r1["contact_lf"][0][3:12] = R.T.ravel()
    G1 = emu.state_grad(q[i:i + 1], v[i:i + 1], mi, r1, Wi, st)
    norm = np.sqrt(float((G["q"] ** 2).sum() + (G["v"] ** 2).sum()))
    lim = max(float(np.abs(G[k] - G1[k]).max()) for k in ("q", "v")) / norm
    print(f"\nexact contact against the gradient at 1e-9: {lim:.1e} of the norm")
    assert lim < 1e-7
    fd = OracleStateLoss("v1", (), {k: x[0] for k, x in r.items()}, m, {k: a[0] for k, a in Wi.items()}).gradient(q[i], v[i])
    fq, fv = sum(fd[k][0] for k in PARTS), sum(fd[k][1] for k in PARTS)
    err = _rel_err(G["q"][0], G["v"][0], fq, fv, q[i])
    print(f"exact contact vs 80-bit central differences: {err:.1e} of the norm")
    assert err < 1e-8


def _ptxas_lines(text, name):
    m = re.search(r"Compiling entry function '(_Z\d+" + name + r"[^']*)'.*?\n(.*?)\n(.*?Used (\d+) registers[^\n]*)", text, re.S)
    spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", m.group(2) + m.group(3))
    return int(m.group(4)), int(spill.group(1)), int(spill.group(2))


def test_state_grad_kernel_spills_within_the_dynamics_kernel():
    """nvcc -Xptxas -v for sm_100a: the adjoint kernel spills no more than the dynamics kernel (both NV instantiations)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                            "-o", os.path.join(tmp, "k.cubin"), os.path.join(SRC, "tsidb.cu")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    for nv in (24, 26):
        dyn = _ptxas_lines(r.stderr, f"tsidb_dynamics_kernelILi{nv}E")
        new = _ptxas_lines(r.stderr, f"tsidb_state_grad_kernelILi{nv}E")
        print(f"\nnv {nv}: dynamics kernel {dyn}, state_grad kernel {new} (registers, spill stores, spill loads)")
        assert new[1] <= dyn[1] and new[2] <= dyn[2]


# ------------------------------------------------------------------ GPU
from test_refs_grad import TIGHT, _controller, _dev, _margin, live  # noqa: E402,F401  (the fixture closes the engines)


def _dev_weights(e, W):
    return {k: t for k, t in zip(W, _dev(e, *W.values()))}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,overrides", [("v1", ()), ("v0", ()), ("v1", TIGHT)])
def test_state_grad_matches_emulator_and_oracle(kind, overrides, live):
    """2048-env walking batches (every contact mask, some envs in flight), NaN outside the written entries: state_grad on
    the GPU against the emulator on 64 envs (rounding: the GPU contracts to FMA) and on 6 of them against central
    differences of the 80-bit oracle (the quaternion in its rotation directions, see _tangent)."""
    import torch

    n = 2048
    s, q, v, mask, refs = _inputs(kind, n, 201, overrides)
    mask[::97] = 0
    e = _controller(kind, n, overrides).engine
    W = _weights(s["cc"], e.nv, mask, 202)
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    out = {k: t.cpu().numpy() for k, t in e.state_grad(qd, vd, md, rd, _dev_weights(e, W)).items()}
    torch.cuda.synchronize()
    assert np.isfinite(out["q"]).all() and np.isfinite(out["v"]).all()
    emu = EmuStateGrad(s["cm"], s["cc"], s["refs"])
    idx = np.linspace(0, n - 1, 64).astype(int)
    ref = emu.state_grad(q[idx], v[idx], mask[idx], {k: a[idx] for k, a in refs.items()}, {k: a[idx] for k, a in W.items()},
                         _strides(s["cc"], e.nv))
    norm = np.sqrt((ref["q"] ** 2).sum(axis=1) + (ref["v"] ** 2).sum(axis=1))
    err = max(float((np.abs(out[k][idx] - ref[k]).max(axis=1) / norm).max()) for k in ("q", "v"))
    worst = 0.0
    for i in idx[::11]:
        r = {k: a[i].copy() for k, a in refs.items()}
        fd = OracleStateLoss(kind, overrides, r, mask[i], {k: a[i] for k, a in W.items()}).gradient(q[i], v[i])
        fq, fv = sum(fd[k][0] for k in PARTS), sum(fd[k][1] for k in PARTS)
        worst = max(worst, _rel_err(out["q"][i], out["v"][i], fq, fv, q[i]))
    print(f"\nstate_grad {kind}{' tight' if overrides else ''}: GPU vs emulator {err:.1e}, vs 80-bit differences (6 envs) "
          f"{worst:.1e} of the gradient's norm")
    assert err < 1e-11 and worst < 1e-8


@pytest.mark.gpu
def test_tick_layer_state_gradcheck_and_refs_only_unchanged(live):
    """On envs with a complementarity margin gradcheck of tick_layer passes with respect to q and to v; with only
    references requiring grad the backward pass returns exactly what qp_grad (g, ce0) followed by refs_grad returns."""
    import torch

    n = 1024
    s, q, v, mask, refs = _inputs("v1", n, 211, TIGHT)
    mask[::97] = 0
    e = _controller("v1", n, TIGHT).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    prob = e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
    sol = e.qp_solve(prob)
    picked = _margin(e, prob, sol, 3)
    assert len(picked) == 3, picked
    idx = torch.as_tensor(picked, device=e.device)
    sub_r = {k: t[idx].contiguous() for k, t in rd.items()}
    q0, v0, m0 = qd[idx].contiguous(), vd[idx].contiguous(), md[idx].contiguous()

    def fq(t):
        o = e.tick_layer(t, v0, m0, sub_r)
        return o["tau"], o["dv"], o["f"]

    def fv(t):
        o = e.tick_layer(q0, t, m0, sub_r)
        return o["tau"], o["dv"], o["f"]

    assert torch.autograd.gradcheck(fq, (q0.clone().requires_grad_(True),), eps=1e-6, atol=1e-5, rtol=1e-4)
    assert torch.autograd.gradcheck(fv, (v0.clone().requires_grad_(True),), eps=1e-6, atol=1e-5, rtol=1e-4)

    rng = np.random.default_rng(212)
    wt = {k: torch.as_tensor(rng.standard_normal((n, d)), device=e.device) for k, d in (("tau", e.na), ("dv", e.nv))}
    base = {k: t.clone().requires_grad_(True) for k, t in rd.items()}
    o = e.tick_layer(qd, vd, md, base)
    loss = sum((o[k] * wt[k]).sum(dim=1) for k in wt)
    got = torch.autograd.grad(loss.sum(), [base[k] for k in REF_KEYS])
    gx = torch.zeros_like(sol["x"])
    gx[:, :e.nv] = wt["dv"]
    qg = e.qp_grad(prob, sol, {"x": gx, "tau": wt["tau"]}, ("g", "ce0"))
    want = e.refs_grad(qd, vd, md, rd, qg["g"], qg["ce0"])
    for g, k in zip(got, REF_KEYS):
        assert torch.equal(g, want[k]), k


def _integrate(q, v, dv, dt):
    """Explicit step in torch, differentiable: v' = v + dt dv; joints and base position by v', the quaternion by the
    first-order update quat + dt/2 quat (x) (w, 0) with w the base's local angular velocity."""
    import torch

    v1 = v + dt * dv
    x, y, z, w = q[:, 3], q[:, 4], q[:, 5], q[:, 6]
    a, b, c = v1[:, 3], v1[:, 4], v1[:, 5]
    dquat = 0.5 * torch.stack([w * a + y * c - z * b, w * b + z * a - x * c, w * c + x * b - y * a, -(x * a + y * b + z * c)], 1)
    q1 = torch.cat([q[:, :3] + dt * v1[:, :3], q[:, 3:7] + dt * dquat, q[:, 7:] + dt * v1[:, 6:]], dim=1)
    return q1, v1


@pytest.mark.gpu
def test_two_tick_closed_loop_matches_differences(live):
    """Two ticks with a torch integration between them: the gradient of a loss on the second tick with respect to the
    first state (autograd through tick_layer, the integration and tick_layer again) matches central differences through
    the GPU forward along random directions in q and v, on the envs whose working sets stay the same at +-h in both
    ticks (measured: 479 of 1024; median relative error 8e-9, 99th percentile 4e-5)."""
    import torch

    n = 1024
    s, q, v, mask, refs = _inputs("v1", n, 221)
    e = _controller("v1", n).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    dt = 0.002
    rng = np.random.default_rng(222)
    wt = {k: torch.as_tensor(rng.standard_normal(s_), device=e.device) for k, s_ in (("tau", (n, e.na)), ("dv", (n, e.nv)),
                                                                                        ("f", (n, 24)))}

    def run(q0, v0):
        o1 = e.tick_layer(q0, v0, md, rd)
        q1, v1 = _integrate(q0, v0, o1["dv"], dt)
        o2 = e.tick_layer(q1.contiguous(), v1.contiguous(), md, rd)
        loss = sum((o2[k] * wt[k]).sum(dim=1) for k in wt)
        return loss, (o1, o2, q1.detach(), v1.detach())

    q0, v0 = qd.clone().requires_grad_(True), vd.clone().requires_grad_(True)
    loss, (o1, o2, q1, v1) = run(q0, v0)
    gq, gv = torch.autograd.grad(loss.sum(), [q0, v0])
    dq = torch.as_tensor(rng.standard_normal((n, e.nq)), device=e.device)
    dvv = torch.as_tensor(rng.standard_normal((n, e.nv)), device=e.device)
    ad = (gq * dq).sum(dim=1) + (gv * dvv).sum(dim=1)
    h = 1e-6

    def act(qq, vv):
        return e.qp_solve(e.problem_data(qq, vv, md, rd, parts=e.PROBLEM_PARTS))

    with torch.no_grad():
        lp, (p1, p2, pq1, pv1) = run(qd + h * dq, vd + h * dvv)
        lm, (m1, m2, mq1, mv1) = run(qd - h * dq, vd - h * dvv)
        a1, a2 = act(qd, vd)["active"], act(q1, v1)["active"]
        same = (o1["status"] == 0) & (o2["status"] == 0)
        for (qq, vv, q2, v2) in ((qd + h * dq, vd + h * dvv, pq1, pv1), (qd - h * dq, vd - h * dvv, mq1, mv1)):
            r1, r2 = act(qq, vv), act(q2.contiguous(), v2.contiguous())
            same &= (r1["active"] == a1).all(dim=1) & (r2["active"] == a2).all(dim=1) & (r1["status"] == 0) & (r2["status"] == 0)
    fd = (lp - lm) / (2 * h)
    kept = int(same.sum())
    rel = ((fd - ad).abs() / (1e-2 + ad.abs()))[same].cpu().numpy()
    print(f"\ntwo-tick loop: {kept}/{n} envs keep their working sets; relative error median {np.median(rel):.1e}, "
          f"99th percentile {np.quantile(rel, 0.99):.1e}, max {rel.max():.1e}")
    assert kept >= 0.3 * n
    assert np.median(rel) < 1e-6 and np.quantile(rel, 0.99) < 1e-2


@pytest.mark.gpu
def test_tick_layer_fit_recovers_state(live):
    """torch.optim (L-BFGS) recovers a perturbed state, every raw component of q (1e-5) and of v (1e-4), from the tau, dv
    and f it produced, on 8 envs whose working set is the same at the true and at the perturbed state, one optimisation
    per env.  On the envs whose working set stays fixed during the fit, the loss falls by more than four orders of
    magnitude and the recovered state is within 10 residual / sigma_min of the true one, sigma_min the smallest singular
    value of d(tau, dv, f) / d(q, v) by central differences through the forward: some directions of the state barely
    show in tau, dv and f (sigma_min reaches 5e-9), and such a direction is recovered only that far."""
    import torch

    n = 256
    s, q, v, mask, refs = _inputs("v1", n, 231)
    e = _controller("v1", n).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    nq, nv = e.nq, e.nv
    gen = torch.Generator(device=e.device).manual_seed(232)
    x0 = torch.cat([1e-5 * torch.randn((n, nq), generator=gen, dtype=torch.float64, device=e.device),
                    1e-4 * torch.randn((n, nv), generator=gen, dtype=torch.float64, device=e.device)], dim=1)
    active = lambda qq, vv, mm, rr: e.qp_solve(e.problem_data(qq, vv, mm, rr, parts=e.PROBLEM_PARTS))["active"]  # noqa: E731
    keep = (active(qd, vd, md, rd) == active(qd + x0[:, :nq], vd + x0[:, nq:], md, rd)).all(dim=1)
    picked = torch.nonzero(keep).flatten()[:8].tolist()
    assert len(picked) == 8
    l0s, l1s, errs, bounds, smins, fixed = [], [], [], [], [], []
    for j in picked:
        qj, vj, mj = qd[j:j + 1].contiguous(), vd[j:j + 1].contiguous(), md[j:j + 1].contiguous()
        rj = {k: t[j:j + 1].contiguous() for k, t in rd.items()}

        def outputs(x, k=1, qj=qj, vj=vj, mj=mj, rj=rj):
            rep = {kk: t.repeat(k, 1) for kk, t in rj.items()}
            o = e.tick_layer((qj.repeat(k, 1) + x[:, :nq]).contiguous(), (vj.repeat(k, 1) + x[:, nq:]).contiguous(),
                             mj.repeat(k), rep)
            return torch.cat([o["tau"], o["dv"], o["f"]], dim=1)

        with torch.no_grad():
            y0 = outputs(torch.zeros((1, nq + nv), dtype=torch.float64, device=e.device))
        x = x0[j:j + 1].clone().requires_grad_(True)
        opt = torch.optim.LBFGS([x], lr=1.0, max_iter=200, history_size=100, tolerance_grad=1e-20,
                                tolerance_change=1e-30, line_search_fn="strong_wolfe")

        def closure(x=x, opt=opt, outputs=outputs, y0=y0):
            opt.zero_grad()
            lo = ((outputs(x) - y0) ** 2).sum()
            lo.backward()
            return lo

        with torch.no_grad():
            l0s.append(float(((outputs(x) - y0) ** 2).sum()))
        for _ in range(3):
            opt.step(closure)
        with torch.no_grad():
            xs = x.detach()
            res = float((outputs(xs) - y0).norm())
            l1s.append(res ** 2)
            h, m = 1e-6, nq + nv
            eye = torch.eye(m, dtype=torch.float64, device=e.device)
            Y = outputs(xs.repeat(2 * m, 1) + h * torch.cat([eye, -eye]), 2 * m)
            smin = float(torch.linalg.svdvals(((Y[:m] - Y[m:]) / (2 * h)).T)[-1])
            fixed.append(bool((active(qj + xs[:, :nq], vj + xs[:, nq:], mj, rj) == active(qj, vj, mj, rj)).all()))
        errs.append(float(xs.norm()))
        smins.append(smin)
        bounds.append(10 * res / smin + 1e-8)
    print(f"\nfit of the state (q and v, {nq + nv} raw components) on {len(picked)} envs: loss {sum(l0s):.2e} -> "
          f"{sum(l1s):.2e}; {sum(fixed)} keep their working set; state error median {np.median(errs):.1e}, max "
          f"{max(errs):.1e} (initial {float(x0[picked].norm(dim=1).median()):.1e}); smallest sigma_min {min(smins):.1e}")
    l0f = sum(x for x, fx in zip(l0s, fixed) if fx)
    l1f = sum(x for x, fx in zip(l1s, fixed) if fx)
    print(f"on the envs that keep their working set: loss {l0f:.2e} -> {l1f:.2e}")
    assert sum(fixed) >= 4
    assert l1f < 1e-4 * l0f
    assert all(err <= bd for err, bd, fx in zip(errs, bounds, fixed) if fx)


@pytest.mark.gpu
def test_state_grad_has_no_side_effects_and_checks_arguments(live):
    """A tick after state_grad is bit-identical to one without it; state_grad on a side stream concurrent with a tick
    gives the same result as alone; bad arguments are refused."""
    import ctypes as C

    import torch

    from tsid_control_b200 import _capi

    n = 2048
    s, q, v, mask, refs = _inputs("v1", n, 241)
    keys = ("tau", "ddq", "f", "status", "iters", "active_set")
    runs = []
    for with_grad in (False, True):
        e = _controller("v1", n).engine
        qd, vd, md, rd = _dev(e, q, v, mask, refs)
        W = _dev_weights(e, _weights(s["cc"], e.nv, mask, 242))
        outs = []
        for _ in range(2):
            if with_grad:
                alone = e.state_grad(qd, vd, md, rd, W)
            t = e.compute(qd, vd, md, rd)
            torch.cuda.synchronize()
            outs.append({k: getattr(t, k).cpu().numpy().copy() for k in keys})
        runs.append(outs)
    for a, b in zip(*runs):
        for k in keys:
            assert np.array_equal(a[k], b[k]), k
    side = torch.cuda.Stream(device=e.device)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        conc = e.state_grad(qd, vd, md, rd, W)
    e.compute(qd, vd, md, rd)
    torch.cuda.synchronize()
    for k in ("q", "v"):
        assert torch.equal(conc[k], alone[k]), k

    lib = e.lib
    nx, neq, nin = e.problem_sizes()
    po = _capi.TsidbProblemOut(g=W["g"].data_ptr())
    dq = torch.empty((n, e.nq), dtype=torch.float64, device=e.device)
    args = lambda nn=n, lay=0, x=nx, eq=neq, i=nin, qp=qd.data_ptr(), vp=vd.data_ptr(), o=dq.data_ptr(): (  # noqa: E731
        e.h, nn, lay, qp, vp, None, None, x, eq, i, C.byref(po), o, None, e._stream())
    assert lib.tsidb_state_grad(*args()) == 0
    assert lib.tsidb_state_grad(*args(nn=n + 1)) < 0 and b"max_envs" in lib.tsidb_last_error()
    assert lib.tsidb_state_grad(*args(nn=0)) < 0
    assert lib.tsidb_state_grad(*args(lay=2)) < 0 and b"layout" in lib.tsidb_last_error()
    assert lib.tsidb_state_grad(*args(x=nx - 1)) < 0 and b"n_max" in lib.tsidb_last_error()
    assert lib.tsidb_state_grad(*args(eq=neq - 1)) < 0
    assert lib.tsidb_state_grad(*args(i=nin - 1)) < 0
    assert lib.tsidb_state_grad(*args(qp=None)) < 0 and b"null" in lib.tsidb_last_error()
    assert lib.tsidb_state_grad(*args(vp=None)) < 0 and b"null" in lib.tsidb_last_error()
    assert lib.tsidb_state_grad(*args(o=None)) < 0 and b"NULL" in lib.tsidb_last_error()
    torch.cuda.synchronize()
    with pytest.raises(TypeError, match="strides"):
        e.state_grad(qd, vd, md, rd, {"g": W["g"][:, :40].contiguous()})
    with pytest.raises(ValueError, match="parts"):
        e.state_grad(qd, vd, md, rd, W, parts=("tau",))
    with pytest.raises(ValueError, match="unknown"):
        e.state_grad(qd, vd, md, rd, {"x": W["g"]})
