"""Linearizing the controller (tsidb_tick_jvp / TsidEngine.tick_jvp / tick_jacobian / forward mode of tick_layer): on the
host emulator, with shared memory NaN-poisoned before every env, the forward derivative against the already verified
adjoints (dot-product identity) and against central differences of the 80-bit oracle's export solved by the oracle's
eiquadprog, with its conventions (layouts, shared directions, NULL parts, unread blocks, enlarged problems, refused
envs); on the GPU the kernel against the emulator and the GPU adjoints, the Jacobian against reverse-mode rows,
forward-mode autograd, differences through the GPU forward, and the absence of side effects."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import force_generator, setup
from emu_py import Emu
from emu_qp import EmuProblemTA, emu_qp_solve
from emu_qp_grad import emu_qp_grad
from emu_refs_grad import REF_KEYS, EmuRefsGrad
from emu_state_grad import EmuStateGrad
from emu_tick_jvp import EmuTickJvp
from oracle_qp import oracle_qp_solve
from test_problem_data import canonical_orders
from test_state_grad import _ptxas_lines
from tsid_control_b200 import synth

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tsid_control_b200", "csrc")
STEP = {"v1": (0.3, 0.2, 0.2, 0.5), "v0": (0.1, 0.1275, 0.05, 0.7)}
QP_PARTS = ("H", "g", "CE", "ce0", "CI", "ci0", "TA", "ta0")


def _inputs(kind, n, seed, overrides=()):
    s = setup(kind, overrides=tuple(overrides))
    q, v = synth.random_states(s["q0"], n, seed)
    mask, refs = synth.walking_batch(s["refs"], n, seed, *STEP[kind], float(s["refs"]["com"][2]))
    return s, q, v, mask, refs


def _dims(nq, nv, na):
    return {"q": nq, "v": nv, "com": 9, "foot_lf": 24, "foot_rf": 24, "contact_lf": 12, "contact_rf": 12, "posture": na}


def _forward(s, q, v, mask, refs):
    """The emulated export with TA, ta0 and the emulated solve on it."""
    prob = EmuProblemTA(s["cm"], s["cc"]).problem_ta(q, v, mask, refs)
    return prob, emu_qp_solve(prob, s["cc"].max_iter)


def _adjoint(s, q, v, mask, refs, prob, sol, ux, ut):
    """J^T u through the emulated qp_grad, state_grad and refs_grad -> {input: [N,k]}."""
    qg = emu_qp_grad(prob, sol, {"x": ux, "tau": ut})
    st = (prob["H"].shape[1], prob["CE"].shape[1], prob["CI"].shape[1])
    sg = EmuStateGrad(s["cm"], s["cc"], s["refs"]).state_grad(q, v, mask, refs, {k: qg[k] for k in QP_PARTS}, st)
    rg = EmuRefsGrad(s["cm"], s["cc"], s["refs"]).refs_grad(q, v, mask, refs, qg["g"], qg["ce0"])
    return dict(rg, q=sg["q"], v=sg["v"])


# ------------------------------------------------------------------ CPU: the kernel body on the host emulator
@pytest.mark.parametrize("kind", ["v1", "v0"])
@pytest.mark.parametrize("maskval", [3, 1, 2, 0])
def test_emulated_dot_product_identity(kind, maskval):
    """<u, J d> from the emulated JVP equals <J^T u, d> from the emulated qp_grad, state_grad and refs_grad within 1e-10
    of |u| |J d| + |J^T u| |d| (the norms of the directions in all inputs together: a reference without effect, such as a
    foot task in double support, has |J d| at rounding level): random per-env directions in q, v and every reference,
    alone and all together, and random cotangents on (x, tau)."""
    n = 2
    s, q, v, _, refs = _inputs(kind, n, 301 + maskval)
    mask = np.full(n, maskval, np.uint8)
    prob, sol = _forward(s, q, v, mask, refs)
    assert (sol["status"] == 0).all()
    J = EmuTickJvp(s["cm"], s["cc"], s["refs"])
    dims = _dims(J.nq, J.nv, J.na)
    rng = np.random.default_rng(302)
    nm = prob["H"].shape[1]
    ux = rng.standard_normal((n, nm)) * (np.arange(nm)[None, :] < prob["sizes"][:, :1])
    ut = rng.standard_normal((n, J.na))
    adj = _adjoint(s, q, v, mask, refs, prob, sol, ux, ut)
    dirs = {k: rng.standard_normal((n, 1, d)) for k, d in dims.items()}
    worst, scale = 0.0, None
    for group in [tuple(dims), ("q",), ("v",)] + [(k,) for k in REF_KEYS]:
        o = J.tick_jvp(q, v, mask, refs, prob, sol, {k: dirs[k] for k in group})
        assert (o["status"] == 0).all()
        if scale is None:
            jd = np.sqrt((o["x"][:, 0] ** 2).sum(1) + (o["tau"][:, 0] ** 2).sum(1))
            ju = np.sqrt(sum((adj[k] ** 2).sum(1) for k in dims))
            dn = np.sqrt(sum((dirs[k][:, 0] ** 2).sum(1) for k in dims))
            scale = np.sqrt((ux ** 2).sum(1) + (ut ** 2).sum(1)) * jd + ju * dn
        for i in range(n):
            lhs = float(ux[i] @ o["x"][i, 0] + ut[i] @ o["tau"][i, 0])
            rhs = sum(float(adj[k][i] @ dirs[k][i, 0]) for k in group)
            worst = max(worst, abs(lhs - rhs) / scale[i])
    print(f"\ndot-product identity ({kind}, mask {maskval}): {worst:.1e}")
    assert worst < 1e-10


class OracleForward:
    """(x, tau) of one env: the 80-bit oracle's dump of the export, solved by the oracle's eiquadprog; tau = TA x + ta0
    with TA built from the dump's M and JF."""

    def __init__(self, kind, mask, max_iter):
        s = setup(kind, "liboracle_ld.so")
        self.orc, self.T, self.mask, self.max_iter = s["oracle"], force_generator(s["cc"]), int(mask), max_iter
        self.orders = canonical_orders(self.orc, self.mask)

    def __call__(self, q, v, refs):
        d = self.orc.tick(q, v, self.mask, refs, dump=True, orders=self.orders)["dump"]
        nv, n = self.orc.nv, d["n"]
        r = oracle_qp_solve(d["H"], d["g"], d["CE"], d["ce0"], d["CI"], d["ci0"], self.max_iter)
        TA = np.zeros((nv - 6, n))
        TA[:, :nv] = d["M"][6:, :nv]
        for s_, f in enumerate(f for f in (0, 1) if (self.mask >> f) & 1):
            TA[:, nv + 12 * s_:nv + 12 * s_ + 12] = -(self.T.T @ d["JF"][f][:, 6:]).T
        x = r["x"][:n]
        return x, TA @ x + d["nle"][6:], sorted(int(a) for a in r["active"] if a >= 0), r["status"]


def _rot_dir(rng, quat):
    """A random direction of the quaternion in the tangent space of the unit sphere (a rotation direction)."""
    u = quat / np.linalg.norm(quat)
    d = rng.standard_normal(4)
    return d - u * float(u @ d)


@pytest.mark.parametrize("kind,maskval", [("v1", 3), ("v1", 1), ("v0", 2), ("v0", 3)])
def test_emulated_jvp_matches_oracle_differences(kind, maskval):
    """On envs whose oracle working set is the same at 0 and +-eps (eps = 1e-6), x' and tau' of the emulated JVP match
    central differences of the oracle's export solved by its eiquadprog, along raw v directions, q directions with the
    quaternion in its rotation directions (off the unit sphere the tick and the oracle extend the functions differently,
    see test_state_grad._tangent), reference directions with the LF contact reference on the sole (log6 at theta = 0)
    and at a generic angle: at most 1e-6 of max(|(x', tau')|, 1) (the floor for directions without effect, such as
    the contact reference of a foot not in contact).  A direction whose differences at eps and 10 eps disagree by more
    than that bar (the oracle's solve in double rounds too coarsely there) is left out and counted."""
    n, eps = 3, 1e-6
    s, q, v, _, refs = _inputs(kind, n, 311 + maskval)
    mask = np.full(n, maskval, np.uint8)
    feet = Emu(s["cm"], s["cc"], s["refs"]).tick(q, v, mask, refs, kin_only=True)["foot_lf"]
    refs["contact_lf"][0] = feet[0]  # env 0: theta = 0 at the LF contact
    prob, sol = _forward(s, q, v, mask, refs)
    J = EmuTickJvp(s["cm"], s["cc"], s["refs"])
    orc = OracleForward(kind, maskval, s["cc"].max_iter)
    rng = np.random.default_rng(312)
    dims = _dims(J.nq, J.nv, J.na)
    checked, noisy, worst = 0, 0, 0.0
    for i in range(n):
        r0 = {k: a[i].copy() for k, a in refs.items()}
        x0, _, act0, st0 = orc(q[i], v[i], r0)
        emu_act = sorted(int(a) for a in sol["active"][i] if a >= 0)
        if st0 != 0 or act0 != emu_act:
            continue
        for group in (("q",), ("v",), ("contact_lf", "foot_rf"), ("com", "posture", "foot_lf", "contact_rf")):
            d = {k: rng.standard_normal(dims[k]) for k in group}
            if "q" in d:
                d["q"][3:7] = _rot_dir(rng, q[i, 3:7])
            o = J.tick_jvp(q[i:i + 1], v[i:i + 1], mask[i:i + 1], {k: a[i:i + 1] for k, a in refs.items()},
                           {k: a[i:i + 1] for k, a in prob.items()}, {k: a[i:i + 1] for k, a in sol.items()},
                           {k: a[None, None] for k, a in d.items()})
            fds = []
            for h in (eps, 10 * eps):
                res = []
                for sgn in (1.0, -1.0):
                    qq = q[i] + sgn * h * d.get("q", 0.0)
                    vv = v[i] + sgn * h * d.get("v", 0.0)
                    rr = {k: a + sgn * h * d[k] if k in d else a for k, a in r0.items()}
                    res.append(orc(qq, vv, rr))
                if any(r[2] != act0 or r[3] != 0 for r in res):
                    break
                fds.append(((res[0][0] - res[1][0]) / (2 * h), (res[0][1] - res[1][1]) / (2 * h)))
            if len(fds) < 2:
                continue
            nx = len(x0)
            jx, jt = o["x"][0, 0, :nx], o["tau"][0, 0]
            norm = max(np.sqrt(float((jx ** 2).sum() + (jt ** 2).sum())), 1.0)
            (fx, ft), (gx, gt) = fds
            if max(float(np.abs(fx - gx).max()), float(np.abs(ft - gt).max())) > 1e-6 * norm:
                noisy += 1  # the oracle's own differences do not resolve this direction to the bar
                continue
            worst = max(worst, max(float(np.abs(jx - fx).max()), float(np.abs(jt - ft).max())) / norm)
            checked += 1
    print(f"\nemulated JVP vs 80-bit oracle differences ({kind}, mask {maskval}, eps {eps}): {checked} direction groups, "
          f"worst {worst:.1e} of the norm; {noisy} groups left out, where the differences at eps and 10 eps disagree")
    assert checked >= 4 and worst < 1e-6


def test_emulated_conventions():
    """Layout 1 equals layout 0, shared directions equal per-env ones, a Jacobian in the references alone (no tangent
    K1 pass) equals the reference columns of one in (q, v, references), NULL parts behave as zero, and NaN in every block
    the call does not read (g, ce0, ci0, the padding, the CI rows outside the working set) changes nothing: bit for bit."""
    n = 4
    s, q, v, _, refs = _inputs("v1", n, 321)
    mask = np.array([3, 1, 2, 0], np.uint8)
    prob, sol = _forward(s, q, v, mask, refs)
    J = EmuTickJvp(s["cm"], s["cc"], s["refs"])
    dims = _dims(J.nq, J.nv, J.na)
    K = sum(dims.values())
    eye = np.eye(K)
    shared, c = {}, 0
    for k, d in dims.items():
        shared[k] = eye[:, c:c + d].copy()
        c += d
    a = J.tick_jvp(q, v, mask, refs, prob, sol, shared, shared=True)
    per_env = {k: np.broadcast_to(x, (n,) + x.shape).copy() for k, x in shared.items()}
    b = J.tick_jvp(q, v, mask, refs, prob, sol, per_env)
    c1 = J.tick_jvp(q, v, mask, refs, prob, sol, shared, shared=True, layout=1)
    nq_nv = dims["q"] + dims["v"]
    only = J.tick_jvp(q, v, mask, refs, prob, sol, {k: shared[k][nq_nv:] for k in REF_KEYS}, shared=True)
    nulls = J.tick_jvp(q, v, mask, refs, prob, sol, {"q": shared["q"][:5], "v": np.zeros((5, dims["v"]))}, shared=True)
    garbage = {k: x.copy() for k, x in prob.items()}
    for i in range(n):
        nx, neq, nin = prob["sizes"][i]
        act = set(int(r) for r in sol["active"][i] if r >= 0)
        for k in ("g", "ce0", "ci0"):
            garbage[k][i] = np.nan
        garbage["H"][i, nx:], garbage["H"][i, :, nx:] = np.nan, np.nan
        garbage["CE"][i, neq:], garbage["CE"][i, :, nx:] = np.nan, np.nan
        garbage["CI"][i, [r for r in range(garbage["CI"].shape[1]) if r not in act]] = np.nan
        garbage["CI"][i, :, nx:], garbage["TA"][i, :, nx:] = np.nan, np.nan
    g = J.tick_jvp(q, v, mask, refs, garbage, sol, shared, shared=True)
    for k in ("x", "tau"):
        assert np.isfinite(a[k]).all()
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], c1[k]) and np.array_equal(a[k], g[k]), k
        assert np.array_equal(only[k], a[k][:, nq_nv:]), k
        assert np.array_equal(nulls[k], a[k][:, :5]), k


def test_emulated_enlarged_problem():
    """An appended constant inequality row and a slack variable (cost 1/2 s^2, the row x_0 + s >= -10): the tangents on
    the export's variables match central differences of the emulated export, enlarged the same way and solved by the
    emulated solve (double precision: eps = 1e-5, bar 1e-5 of the norm), along random q, v and reference directions."""
    n, eps = 2, 1e-5
    s, q, v, _, refs = _inputs("v1", n, 331)
    mask = np.array([3, 1], np.uint8)
    ep = EmuProblemTA(s["cm"], s["cc"])
    J = EmuTickJvp(s["cm"], s["cc"], s["refs"])
    dims = _dims(J.nq, J.nv, J.na)

    def enlarged(qq, vv, rr):
        p = ep.problem_ta(qq, vv, mask, rr)
        N, nm = p["g"].shape
        nin = p["CI"].shape[1]
        e = {"H": np.zeros((N, nm + 1, nm + 1)), "g": np.zeros((N, nm + 1)), "CE": np.zeros((N, 18, nm + 1)),
             "ce0": p["ce0"].copy(), "CI": np.zeros((N, nin + 1, nm + 1)), "ci0": np.zeros((N, nin + 1)),
             "TA": np.zeros((N, J.na, nm + 1)), "ta0": p["ta0"].copy(), "sizes": p["sizes"].copy()}
        for i in range(N):
            nx, neq, ni = p["sizes"][i]
            e["H"][i, :nx, :nx] = p["H"][i, :nx, :nx]
            e["H"][i, nx, nx] = 1.0
            e["g"][i, :nx] = p["g"][i, :nx]
            e["CE"][i, :neq, :nx] = p["CE"][i, :neq, :nx]
            e["CI"][i, :ni, :nx] = p["CI"][i, :ni, :nx]
            e["ci0"][i, :ni] = p["ci0"][i, :ni]
            e["CI"][i, ni, 0], e["CI"][i, ni, nx], e["ci0"][i, ni] = 1.0, 1.0, 10.0
            e["TA"][i, :, :nx] = p["TA"][i, :, :nx]
            e["sizes"][i] = (nx + 1, neq, ni + 1)
        return e

    prob = enlarged(q, v, refs)
    sol = emu_qp_solve(prob, s["cc"].max_iter)
    assert (sol["status"] == 0).all()
    rng = np.random.default_rng(332)
    d = {k: rng.standard_normal((n, 1, dims[k])) for k in ("q", "v", "com", "foot_lf", "contact_rf")}
    o = J.tick_jvp(q, v, mask, refs, prob, sol, d)
    assert (o["status"] == 0).all()
    sp = emu_qp_solve(enlarged(q + eps * d["q"][:, 0], v + eps * d["v"][:, 0],
                               {k: a + eps * d[k][:, 0] if k in d else a for k, a in refs.items()}), s["cc"].max_iter)
    sm = emu_qp_solve(enlarged(q - eps * d["q"][:, 0], v - eps * d["v"][:, 0],
                               {k: a - eps * d[k][:, 0] if k in d else a for k, a in refs.items()}), s["cc"].max_iter)
    worst = 0.0
    for i in range(n):
        same = [sorted(a[i][a[i] >= 0]) for a in (sol["active"], sp["active"], sm["active"])]
        assert same[0] == same[1] == same[2]
        nx = prob["sizes"][i][0]
        fx = (sp["x"][i, :nx] - sm["x"][i, :nx]) / (2 * eps)
        ft = (sp["tau"][i] - sm["tau"][i]) / (2 * eps)
        norm = np.sqrt(float((o["x"][i, 0] ** 2).sum() + (o["tau"][i, 0] ** 2).sum()))
        worst = max(worst, max(float(np.abs(o["x"][i, 0, :nx] - fx).max()), float(np.abs(o["tau"][i, 0] - ft).max())) / norm)
    print(f"\nenlarged problem: emulated JVP vs emulated differences {worst:.1e} of the norm")
    assert worst < 1e-5


def test_emulated_refused_envs_get_zeros():
    """A non-OPTIMAL solve, a corrupt working set (a duplicate row) and dependent working-set rows (an equality row copied
    into a CI row that joins the working set) give status 4 and all-zero tangents; the other envs are unchanged."""
    n = 4
    s, q, v, _, refs = _inputs("v1", n, 341)
    mask = np.array([3, 3, 1, 2], np.uint8)
    prob, sol = _forward(s, q, v, mask, refs)
    J = EmuTickJvp(s["cm"], s["cc"], s["refs"])
    d = {"q": np.random.default_rng(342).standard_normal((2, J.nq))}
    base = J.tick_jvp(q, v, mask, refs, prob, sol, d, shared=True)
    sol2 = {k: a.copy() for k, a in sol.items()}
    prob2 = {k: a.copy() for k, a in prob.items()}
    sol2["status"][0] = 3
    w = int((sol["active"][1] >= 0).sum())
    assert w >= 1
    sol2["active"][1, w] = sol["active"][1, 0]  # duplicate row
    w3 = int((sol["active"][3] >= 0).sum())
    free = [r for r in range(prob["sizes"][3][2]) if r not in set(sol["active"][3][:w3])][0]
    prob2["CI"][3, free] = prob["CE"][3, 0]
    sol2["active"][3, w3], sol2["lambda"][3, w3] = free, 0.0  # a dependent row
    o = J.tick_jvp(q, v, mask, refs, prob2, sol2, d, shared=True)
    assert list(o["status"]) == [4, 4, 0, 4]
    for k in ("x", "tau"):
        assert (o[k][[0, 1, 3]] == 0).all() and np.array_equal(o[k][2], base[k][2])


def test_tick_jvp_kernel_spills_within_the_dynamics_kernel():
    """nvcc -Xptxas -v for sm_100a: the JVP kernel and each of its non-inlined parts (setup, tangent K1, per-direction
    solve) spill no more than the dynamics kernel (both NV instantiations)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-cubin",
                            "-o", os.path.join(tmp, "k.cubin"), os.path.join(SRC, "tsidb.cu")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    import re
    for nv in (24, 26):
        dyn = _ptxas_lines(r.stderr, f"tsidb_dynamics_kernelILi{nv}E")
        new = _ptxas_lines(r.stderr, f"tsidb_tick_jvp_kernelILi{nv}E")
        assert new[1] <= dyn[1] and new[2] <= dyn[2], (dyn, new)
        for fn in ("tick_jvp_setup", "tick_jvp_k1", "tick_jvp_dir"):
            m = re.search(r"Function properties for _Z\d+" + fn + r"ILi" + str(nv) + r"E[^\n]*\n\s*(\d+) bytes stack frame, "
                          r"(\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
            assert m, fn
            assert int(m.group(2)) <= dyn[1] and int(m.group(3)) <= dyn[2], (fn, m.groups())
        print(f"\nnv {nv}: dynamics kernel {dyn}, tick_jvp kernel {new} (registers, spill stores, spill loads)")


# ------------------------------------------------------------------ GPU
from test_refs_grad import TIGHT, _controller, _dev, _margin, live  # noqa: E402,F401  (the fixture closes the engines)


def _dev_np(e, d):
    import torch
    return {k: torch.as_tensor(np.ascontiguousarray(a), device=e.device) for k, a in d.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,overrides", [("v1", ()), ("v0", ()), ("v1", TIGHT)])
def test_tick_jvp_matches_emulator_and_adjoints(kind, overrides, live):
    """2048-env walking batches (every contact mask, some envs in flight), one random per-env direction in q, v and
    every reference: the GPU JVP against the emulator on 32 envs, and the dot-product identity against the GPU's qp_grad,
    state_grad and refs_grad on every env (the CPU bar, 1e-10; for the tight conf the worst env's cond(KKT) is reported).
    The GPU contracts to FMA and the emulator does not, and the KKT solve amplifies that rounding by its conditioning:
    measured 1e-10 (v1), 1.8e-10 (v0) and 5.5e-10 (tight) relative per env against the emulator; the bar is 1e-9."""
    import torch

    n = 2048
    s, q, v, mask, refs = _inputs(kind, n, 401, overrides)
    mask[::97] = 0
    e = _controller(kind, n, overrides).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    prob = e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
    sol = e.qp_solve(prob)
    dims = _dims(e.nq, e.nv, e.na)
    rng = np.random.default_rng(402)
    dirs = {k: rng.standard_normal((n, 1, d)) for k, d in dims.items()}
    o = e.tick_jvp(qd, vd, md, rd, _dev_np(e, dirs), prob, sol)
    O = {k: t.cpu().numpy() for k, t in o.items()}
    P = {k: t.cpu().numpy() for k, t in prob.items()}
    S = {k: t.cpu().numpy() for k, t in sol.items()}
    ok = (O["status"] == 0) & (S["status"] == 0)
    assert ok.mean() > 0.9 and np.isfinite(O["x"]).all() and np.isfinite(O["tau"]).all()
    idx = np.linspace(0, n - 1, 32).astype(int)
    J = EmuTickJvp(s["cm"], s["cc"], s["refs"])
    ref = J.tick_jvp(q[idx], v[idx], mask[idx], {k: a[idx] for k, a in refs.items()}, {k: a[idx] for k, a in P.items()},
                     {k: a[idx] for k, a in S.items()}, {k: a[idx] for k, a in dirs.items()})
    assert np.array_equal(ref["status"], O["status"][idx])
    norm = np.sqrt((ref["x"] ** 2).sum(axis=(1, 2)) + (ref["tau"] ** 2).sum(axis=(1, 2))) + 1e-300
    err = max(float((np.abs(O[k][idx] - ref[k]).max(axis=(1, 2)) / norm).max()) for k in ("x", "tau"))
    nm = P["H"].shape[1]
    ux = rng.standard_normal((n, nm)) * (np.arange(nm)[None, :] < P["sizes"][:, :1])
    ut = rng.standard_normal((n, e.na))
    qg = e.qp_grad(prob, sol, _dev_np(e, {"x": ux, "tau": ut}))
    g = {k: t for k, t in qg.items() if k != "status"}
    sg = e.state_grad(qd, vd, md, rd, g)
    rg = e.refs_grad(qd, vd, md, rd, qg["g"], qg["ce0"])
    adj = {k: t.cpu().numpy() for k, t in dict(rg, q=sg["q"], v=sg["v"]).items()}
    ok &= qg["status"].cpu().numpy() == 0
    lhs = (ux * O["x"][:, 0]).sum(1) + (ut * O["tau"][:, 0]).sum(1)
    rhs = sum((adj[k] * dirs[k][:, 0]).sum(1) for k in dims)
    jd = np.sqrt((O["x"][:, 0] ** 2).sum(1) + (O["tau"][:, 0] ** 2).sum(1))
    ju = np.sqrt(sum((adj[k] ** 2).sum(1) for k in dims))
    dn = np.sqrt(sum((dirs[k][:, 0] ** 2).sum(1) for k in dims))
    un = np.sqrt((ux ** 2).sum(1) + (ut ** 2).sum(1))
    rel = np.abs(lhs - rhs) / (un * jd + ju * dn)
    worst = int(np.argmax(np.where(ok, rel, 0.0)))
    print(f"\ntick_jvp {kind}{' tight' if overrides else ''}: GPU vs emulator {err:.1e}; dot-product identity worst "
          f"{rel[ok].max():.1e} (env {worst}), median {np.median(rel[ok]):.1e}")
    if overrides:
        i = worst
        nx, neq, _ = P["sizes"][i]
        w = int((S["active"][i] >= 0).sum())
        G = np.vstack([P["CE"][i, :neq, :nx], P["CI"][i, S["active"][i, :w], :nx]])
        K = np.block([[P["H"][i, :nx, :nx], G.T], [G, np.zeros((G.shape[0], G.shape[0]))]])
        print(f"tight conf: env {i} cond(KKT) {np.linalg.cond(K):.1e}")
    assert err < 1e-9 and rel[ok].max() < 1e-10
    torch.cuda.synchronize()


def _reverse_rows(e, q, v, m, r):
    """The Jacobian of tau, dv, f with respect to (q, v) from unit cotangents through tick_layer's backward, one row at a
    time -> [N, rows, nq + nv]."""
    import torch

    qq, vv = q.clone().requires_grad_(True), v.clone().requires_grad_(True)
    o = e.tick_layer(qq, vv, m, r)
    rows = []
    for name in ("tau", "dv", "f"):
        for j in range(o[name].shape[1]):
            gq, gv = torch.autograd.grad(o[name][:, j].sum(), (qq, vv), retain_graph=True, allow_unused=True)
            rows.append(torch.cat([gq if gq is not None else torch.zeros_like(q), gv if gv is not None else torch.zeros_like(v)], 1))
    return torch.stack(rows, 1)


@pytest.mark.gpu
def test_tick_jacobian_equals_reverse_rows(live):
    """tick_jacobian in (q, v) on a 64-env batch equals the stack of reverse-mode rows (unit cotangents through
    tick_layer's backward) to 1e-9 relative per column."""
    import torch

    n = 64
    s, q, v, mask, refs = _inputs("v1", n, 411)
    e = _controller("v1", n).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    Jf = e.tick_jacobian(qd, vd, md, rd)
    fwd = torch.cat([Jf["tau"], Jf["dv"], Jf["f"]], 1)
    rev = _reverse_rows(e, qd, vd, md, rd)
    ok = Jf["status"] == 0
    col = torch.linalg.vector_norm(fwd, dim=1) + 1e-300
    err = ((fwd - rev).abs().amax(dim=1) / col)[ok]
    print(f"\ntick_jacobian vs reverse rows: {int(ok.sum())} envs, worst {float(err.max()):.1e} relative per column")
    assert ok.float().mean() > 0.9 and float(err.max()) < 1e-9


@pytest.mark.gpu
def test_forward_ad_and_gradcheck(live):
    """forward_ad dual tensors on q, v and every reference give tick_jvp's tangents bit for bit; gradcheck with
    check_forward_ad passes with respect to q, v and each reference on envs with a complementarity margin."""
    import torch
    import torch.autograd.forward_ad as fwAD

    n = 1024
    s, q, v, mask, refs = _inputs("v1", n, 211, TIGHT)
    mask[::97] = 0  # as in test_state_grad: the envs with a complementarity margin are among these
    e = _controller("v1", n, TIGHT).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    rng = np.random.default_rng(422)
    dims = _dims(e.nq, e.nv, e.na)
    tan = _dev_np(e, {k: rng.standard_normal((n, d)) for k, d in dims.items()})
    with fwAD.dual_level():
        qq, vv = fwAD.make_dual(qd, tan["q"]), fwAD.make_dual(vd, tan["v"])
        rr = {k: fwAD.make_dual(rd[k], tan[k]) for k in REF_KEYS}
        o = e.tick_layer(qq, vv, md, rr)
        got = {k: fwAD.unpack_dual(o[k]).tangent for k in ("tau", "dv", "f")}
    want = e.tick_jvp(qd, vd, md, rd, {k: t.unsqueeze(1).contiguous() for k, t in tan.items()})
    for k in ("tau", "dv", "f"):
        assert torch.equal(got[k], want[k][:, 0]), k
    prob = e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
    sol = e.qp_solve(prob)
    picked = _margin(e, prob, sol, 2)
    assert len(picked) == 2, picked
    idx = torch.as_tensor(picked, device=e.device)
    q0, v0, m0 = qd[idx].contiguous(), vd[idx].contiguous(), md[idx].contiguous()
    r0 = {k: t[idx].contiguous() for k, t in rd.items()}
    for name in ("q", "v") + REF_KEYS:
        def f(t, name=name):
            args = {"q": q0, "v": v0}
            rr = dict(r0)
            if name in args:
                args[name] = t
            else:
                rr[name] = t
            out = e.tick_layer(args["q"], args["v"], m0, rr)
            return out["tau"], out["dv"], out["f"]
        x0 = {"q": q0, "v": v0}.get(name, r0.get(name))
        assert torch.autograd.gradcheck(f, (x0.clone().requires_grad_(True),), eps=1e-6, atol=1e-5, rtol=1e-4,
                                        check_forward_ad=True, check_backward_ad=False, check_undefined_grad=False), name


@pytest.mark.gpu
def test_jvp_matches_gpu_differences(live):
    """Central differences (h = 1e-6) through the GPU forward (problem_data + qp_solve) along random directions in q,
    v and the references agree with tick_jvp on the envs whose working set stays fixed at +-h; the share of such envs
    and the median and max relative error are reported."""
    import torch

    n, h = 1024, 1e-6
    s, q, v, mask, refs = _inputs("v1", n, 431)
    e = _controller("v1", n).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    rng = np.random.default_rng(432)
    dims = _dims(e.nq, e.nv, e.na)
    tan = _dev_np(e, {k: rng.standard_normal((n, d)) for k, d in dims.items()})
    o = e.tick_jvp(qd, vd, md, rd, {k: t.unsqueeze(1).contiguous() for k, t in tan.items()})

    def fwd(sg):
        r = {k: rd[k] + sg * h * tan[k] for k in REF_KEYS}
        p = e.problem_data(qd + sg * h * tan["q"], vd + sg * h * tan["v"], md, r, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
        return e.qp_solve(p)

    s0, sp, sm = fwd(0.0), fwd(1.0), fwd(-1.0)
    same = (s0["status"] == 0) & (sp["status"] == 0) & (sm["status"] == 0) & (o["status"] == 0) & \
        (torch.sort(s0["active"], 1)[0] == torch.sort(sp["active"], 1)[0]).all(1) & \
        (torch.sort(s0["active"], 1)[0] == torch.sort(sm["active"], 1)[0]).all(1)
    fx = (sp["x"] - sm["x"]) / (2 * h)
    ft = (sp["tau"] - sm["tau"]) / (2 * h)
    jx, jt = o["x"][:, 0], o["tau"][:, 0]
    norm = torch.sqrt((jx ** 2).sum(1) + (jt ** 2).sum(1))
    rel = torch.maximum((jx - fx).abs().amax(1), (jt - ft).abs().amax(1)) / norm
    rel = rel[same].cpu().numpy()
    print(f"\nJVP vs GPU central differences: {same.float().mean().item():.0%} of envs keep their working set; relative "
          f"error median {np.median(rel):.1e}, max {rel.max():.1e}")
    assert same.float().mean().item() > 0.5 and np.median(rel) < 1e-6 and rel.max() < 1e-3


@pytest.mark.gpu
def test_tick_jvp_has_no_side_effects_and_checks_arguments(live):
    """A tick after the call is bit-identical to one without it, a call on a side stream gives the same result, repeated
    calls are bit-identical, and bad arguments are refused."""
    import torch

    from tsid_control_b200._capi import TsidbError

    n = 512
    s, q, v, mask, refs = _inputs("v1", n, 441)
    e = _controller("v1", n).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    keys = ("tau", "ddq", "f", "status")
    t0 = e.compute(qd, vd, md, rd)
    t0 = {k: getattr(t0, k).clone() for k in keys}
    rng = np.random.default_rng(442)
    tan = _dev_np(e, {"q": rng.standard_normal((3, e.nq)), "contact_lf": rng.standard_normal((3, 12))})
    a = e.tick_jvp(qd, vd, md, rd, tan)
    t1 = e.compute(qd, vd, md, rd)
    for k in keys:
        assert torch.equal(t0[k], getattr(t1, k)), k
    b = e.tick_jvp(qd, vd, md, rd, tan)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        c = e.tick_jvp(qd, vd, md, rd, tan)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for k in ("x", "tau", "dv", "f", "status"):
        assert torch.equal(a[k], b[k]) and torch.equal(a[k], c[k]), k
    with pytest.raises(ValueError):
        e.tick_jvp(qd, vd, md, rd, {})
    with pytest.raises(ValueError):
        e.tick_jvp(qd, vd, md, rd, {"bogus": tan["q"]})
    with pytest.raises(TypeError):
        e.tick_jvp(qd, vd, md, rd, {"q": tan["q"], "v": torch.zeros((n, 3, e.nv), dtype=torch.float64, device=e.device)})
    with pytest.raises(TypeError):
        e.tick_jvp(qd, vd, md, rd, {"q": tan["q"][:, :5].contiguous()})
    with pytest.raises(ValueError):
        e.tick_jacobian(qd, vd, md, rd, wrt=("q", "q"))
    import ctypes as C

    from tsid_control_b200 import _capi
    jd, jo = _capi.TsidbJvpDirs(), _capi.TsidbJvpOut()
    st = torch.empty(n, dtype=torch.int32, device=e.device)
    po, so = _capi.TsidbProblemOut(), _capi.TsidbQpOut()
    rc = e.lib.tsidb_tick_jvp(e.h, n, 0, qd.data_ptr(), vd.data_ptr(), None, None, 50, 18, 160, C.byref(po), C.byref(so), 1,
                              0, C.byref(jd), C.byref(jo), st.data_ptr(), None)
    assert rc == -1 and b"both NULL" in e.lib.tsidb_last_error()
    with pytest.raises(TsidbError):
        _capi.check(rc, "tsidb_tick_jvp")
