"""Differentiating through the task references (tsidb_refs_grad / TsidEngine.refs_grad / TsidEngine.tick_layer): the
adjoint of the map references -> (g, ce0) against central differences of the 80-bit oracle's dump of the same problem,
the SE3 logarithm's branches, layouts, defaults and NULL parts on the host emulator, and on the GPU the kernel against
the emulator and the oracle, the autograd layer against gradcheck and finite differences through the GPU forward, a fit
that recovers references, and the absence of side effects on the tick."""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from common import make_conf, setup
from emu_refs_grad import REF_KEYS, EmuRefsGrad
from test_problem_data import canonical_orders
from tsid_control_b200 import synth

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tsid_control_b200", "csrc")
STEP = {"v1": (0.3, 0.2, 0.2, 0.5), "v0": (0.1, 0.1275, 0.05, 0.7)}


def _inputs(kind, n, seed, overrides=()):
    s = setup(kind, overrides=tuple(overrides))
    q, v = synth.random_states(s["q0"], n, seed)
    mask, refs = synth.walking_batch(s["refs"], n, seed, *STEP[kind], float(s["refs"]["com"][2]))
    return s, q, v, mask, refs


def _weights(n, nv, masks, seed):
    """Random dL/dg [N,nv+24] and dL/dce0 [N,18] with NaN in every entry the adjoint must not read."""
    rng = np.random.default_rng(seed)
    dg = np.full((n, nv + 24), np.nan)
    dg[:, :nv] = rng.standard_normal((n, nv))
    dce0 = np.full((n, 18), np.nan)
    for i, m in enumerate(masks):
        nc = (int(m) & 1) + ((int(m) >> 1) & 1)
        dce0[i, 6:6 + 6 * nc] = rng.standard_normal(6 * nc)
    return dg, dce0


class OracleLoss:
    """L(refs) = dg . g[:nv] + dce0 . ce0[6:6+6nc] of one env from the 80-bit oracle's dump of its problem."""

    def __init__(self, kind, overrides, q, v, mask, dg, dce0):
        self.orc = setup(kind, "liboracle_ld.so", overrides=tuple(overrides))["oracle"]
        self.q, self.v, self.mask = q, v, int(mask)
        self.nv = self.orc.nv
        nc = (self.mask & 1) + ((self.mask >> 1) & 1)
        self.dg, self.dce0, self.rows = dg[:self.nv], dce0[6:6 + 6 * nc], slice(6, 6 + 6 * nc)
        self.orders = canonical_orders(self.orc, self.mask)

    def __call__(self, refs):
        d = self.orc.tick(self.q, self.v, self.mask, refs, dump=True, orders=self.orders)["dump"]
        return float(self.dg @ d["g"][:self.nv] + self.dce0 @ d["ce0"][self.rows])

    def gradient(self, refs, h=1e-5):
        """Central differences with respect to every component of every reference."""
        out = {}
        for k in REF_KEYS:
            fd = np.zeros(len(refs[k]))
            for j in range(len(fd)):
                rp = {kk: a.copy() for kk, a in refs.items()}
                rm = {kk: a.copy() for kk, a in refs.items()}
                rp[k][j] += h
                rm[k][j] -= h
                fd[j] = (self(rp) - self(rm)) / (2 * h)
            out[k] = fd
        return out


def _rel_err(grad, fd):
    """max |adjoint - differences| over all components / norm of the adjoint."""
    norm = np.sqrt(sum(float((grad[k] ** 2).sum()) for k in REF_KEYS))
    return max(float(np.abs(grad[k] - fd[k]).max()) for k in REF_KEYS) / norm


# ------------------------------------------------------------------ CPU: the kernel bodies on the host emulator
@pytest.mark.parametrize("kind", ["v1", "v0"])
@pytest.mark.parametrize("maskval", [3, 1, 2, 0])
def test_emulated_refs_grad_matches_oracle_differences(kind, maskval):
    """Every component of every reference, two walking envs per contact mask: the emulated adjoint against central
    differences (h = 1e-5) of the 80-bit oracle's g and ce0, with NaN in all padding of dg and dce0.  Measured: ~1e-11 of
    the gradient's norm (the differences' own rounding, eps |L| / h); the bar is 1e-8."""
    n = 2
    s, q, v, _, refs = _inputs(kind, n, 71 + maskval)
    mask = np.full(n, maskval, np.uint8)
    emu = EmuRefsGrad(s["cm"], s["cc"], s["refs"])
    dg, dce0 = _weights(n, emu.nv, mask, 72)
    G = emu.refs_grad(q, v, mask, refs, dg, dce0)
    worst = 0.0
    for i in range(n):
        r = {k: a[i].copy() for k, a in refs.items()}
        fd = OracleLoss(kind, (), q[i], v[i], maskval, dg[i], dce0[i]).gradient(r)
        worst = max(worst, _rel_err({k: G[k][i] for k in REF_KEYS}, fd))
        if not maskval & 1:
            assert not G["contact_lf"][i].any()
        if not maskval & 2:
            assert not G["contact_rf"][i].any()
    print(f"\nemulated refs_grad vs 80-bit central differences ({kind}, mask {maskval}): {worst:.1e} of the norm")
    assert worst < 1e-8


def _rodrigues(w):
    th = np.linalg.norm(w)
    K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    if th == 0.0:
        return np.eye(3)
    return np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * K @ K


@pytest.mark.parametrize("angle", [0.0, 1e-6, 1e-4, 0.7, np.pi - 5e-3])
def test_se3_log_branches(angle):
    """References of the LF contact and the RF foot task whose error rotation E = Rf^T R_ref has angle 0, 1e-6, 1e-4
    (small-angle branch), 0.7 (generic) and pi - 5e-3 (near pi, every sqrt argument ~2 w_k^2 bounded away from 0): the
    adjoint agrees with central differences of the 80-bit oracle along rotations R exp(e w^) and along positions; at 0
    it is finite and equals the limit from inside (the gradient at angle 1e-9)."""
    kind, maskval = "v1", 3
    s, q, v, _, refs = _inputs(kind, 1, 81)
    emu = EmuRefsGrad(s["cm"], s["cc"], s["refs"])
    orc = s["oracle"]
    placed = orc.tick(q[0], v[0], maskval, {k: a[0] for k, a in refs.items()})["foot"]
    axis = np.array([0.6, -0.5, 0.62]) / np.linalg.norm([0.6, -0.5, 0.62])

    def refs_at(th):
        r = {k: a[0].copy() for k, a in refs.items()}
        for key, f in (("contact_lf", 0), ("foot_rf", 1)):
            Rf = placed[f][3:12].reshape(3, 3).T  # (p, R column-major)
            R = Rf @ _rodrigues(th * axis)
            r[key][:3] = placed[f][:3] + np.array([0.01, -0.02, 0.015])
            r[key][3:12] = R.T.ravel()
        return r

    r = refs_at(angle)
    dg, dce0 = _weights(1, emu.nv, [maskval], 82)
    G = emu.refs_grad(q, v, np.array([maskval], np.uint8), {k: a[None] for k, a in r.items()}, dg, dce0)
    assert all(np.isfinite(G[k]).all() for k in REF_KEYS)
    L = OracleLoss(kind, (), q[0], v[0], maskval, dg[0], dce0[0])
    rng = np.random.default_rng(83)
    norm = np.sqrt(sum(float((G[k] ** 2).sum()) for k in REF_KEYS))
    worst, eps = 0.0, 1e-6
    for key in ("contact_lf", "foot_rf"):
        R = r[key][3:12].reshape(3, 3).T
        for _ in range(3):
            w = rng.standard_normal(3)
            Rp, Rm = R @ _rodrigues(eps * w), R @ _rodrigues(-eps * w)
            rp = {k: a.copy() for k, a in r.items()}
            rm = {k: a.copy() for k, a in r.items()}
            rp[key][3:12], rm[key][3:12] = Rp.T.ravel(), Rm.T.ravel()
            fd = (L(rp) - L(rm)) / (2 * eps)
            K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
            ad = float(G[key][0][3:12] @ (R @ K).T.ravel())
            worst = max(worst, abs(fd - ad) / norm)
            d = rng.standard_normal(3)
            rp, rm = {k: a.copy() for k, a in r.items()}, {k: a.copy() for k, a in r.items()}
            rp[key][:3] += eps * d
            rm[key][:3] -= eps * d
            worst = max(worst, abs((L(rp) - L(rm)) / (2 * eps) - float(G[key][0][:3] @ d)) / norm)
    print(f"\nangle {angle:.3g}: adjoint vs 80-bit directional differences {worst:.1e} of the norm")
    assert worst < 1e-7
    if angle == 0.0:
        G1 = emu.refs_grad(q, v, np.array([maskval], np.uint8), {k: a[None] for k, a in refs_at(1e-9).items()}, dg, dce0)
        lim = max(float(np.abs(G[k] - G1[k]).max()) for k in REF_KEYS) / norm
        print(f"angle 0 against the gradient at 1e-9: {lim:.1e} of the norm")
        assert lim < 1e-8


def test_emulated_layouts_defaults_and_null_parts():
    """Layout 1 gives the transpose of layout 0 bit for bit; references left out give the gradient at the defaults; a
    NULL dg or dce0 counts as zero; a part that is not requested is not written (its NaN stays)."""
    n = 4
    s, q, v, mask, refs = _inputs("v1", n, 91)
    mask = np.array([3, 1, 2, 0], np.uint8)
    emu = EmuRefsGrad(s["cm"], s["cc"], s["refs"])
    dg, dce0 = _weights(n, emu.nv, mask, 92)
    g0 = emu.refs_grad(q, v, mask, refs, dg, dce0)
    g1 = emu.refs_grad(q, v, mask, refs, dg, dce0, layout=1)
    for k in REF_KEYS:
        assert np.array_equal(g0[k], g1[k]), k
    tiled = {k: np.tile(s["refs"][k], (n, 1)) for k in REF_KEYS}
    a = emu.refs_grad(q, v, mask, {}, dg, dce0)
    b = emu.refs_grad(q, v, mask, tiled, dg, dce0)
    for k in REF_KEYS:
        assert np.array_equal(a[k], b[k]), k
    zg = np.where(np.isnan(dg), np.nan, 0.0)
    zc = np.where(np.isnan(dce0), np.nan, 0.0)
    for args in ((None, dce0), (dg, None)):
        x = emu.refs_grad(q, v, mask, refs, *args)
        y = emu.refs_grad(q, v, mask, refs, zg if args[0] is None else dg, zc if args[1] is None else dce0)
        for k in REF_KEYS:
            assert np.array_equal(x[k], y[k]), k
    part = emu.refs_grad(q, v, mask, refs, dg, dce0, parts=("com", "contact_rf"))
    assert set(part) == {"com", "contact_rf"}
    for k in part:
        assert np.array_equal(part[k], g0[k])
    assert np.isfinite(g0["posture"]).all()


def _ptxas_lines(text, name):
    m = re.search(r"Compiling entry function '(_Z\d+" + name + r"[^']*)'.*?\n(.*?)\n(.*?Used (\d+) registers[^\n]*)", text, re.S)
    spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", m.group(2) + m.group(3))
    return int(m.group(4)), int(spill.group(1)), int(spill.group(2))


def test_refs_grad_kernel_spills_within_the_dynamics_kernel():
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
        new = _ptxas_lines(r.stderr, f"tsidb_refs_grad_kernelILi{nv}E")
        print(f"\nnv {nv}: dynamics kernel {dyn}, refs_grad kernel {new} (registers, spill stores, spill loads)")
        assert new[1] <= dyn[1] and new[2] <= dyn[2]
        assert new[0] <= 168


# ------------------------------------------------------------------ GPU
_LIVE = []


@pytest.fixture
def live():
    yield _LIVE
    while _LIVE:
        _LIVE.pop().engine.close()


def _controller(kind, n, overrides=()):
    conf = make_conf(kind, overrides)
    conf.max_envs = n
    if kind == "v1":
        from tsid_control_b200.ctrl.WalkController import WalkController

        c = WalkController(conf, n_envs=n)
    else:
        from tsid_control_b200.legacy.biped import Biped

        c = Biped(conf, n_envs=n)
    _LIVE.append(c)
    return c


def _dev(e, *arrays):
    import torch

    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=e.device)  # noqa: E731
    return [({k: t(x) for k, x in a.items()} if isinstance(a, dict) else t(a)) for a in arrays]


TIGHT = (("tau_max_scaling", 0.08), ("v_max_scaling", 0.1))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,overrides", [("v1", ()), ("v0", ()), ("v1", TIGHT)])
def test_refs_grad_matches_emulator_and_oracle(kind, overrides, live):
    """2048-env walking batches (every contact mask, some envs in flight): refs_grad on the GPU against the emulator on
    every env (rounding: the GPU contracts to FMA), and on 64 envs against central differences of the 80-bit oracle."""
    import torch

    n = 2048
    s, q, v, mask, refs = _inputs(kind, n, 101, overrides)
    mask[::97] = 0
    e = _controller(kind, n, overrides).engine
    dg, dce0 = _weights(n, e.nv, mask, 102)
    qd, vd, md, rd, dgd, dcd = _dev(e, q, v, mask, refs, dg, dce0)
    out = {k: t.cpu().numpy() for k, t in e.refs_grad(qd, vd, md, rd, dgd, dcd).items()}
    torch.cuda.synchronize()
    emu = EmuRefsGrad(s["cm"], s["cc"], s["refs"])
    ref = emu.refs_grad(q, v, mask, refs, dg, dce0)
    norm = np.sqrt(sum((ref[k] ** 2).sum(axis=1) for k in REF_KEYS))
    err = max(float((np.abs(out[k] - ref[k]).max(axis=1) / norm).max()) for k in REF_KEYS)
    worst = 0.0
    for i in np.linspace(0, n - 1, 64).astype(int):
        r = {k: a[i].copy() for k, a in refs.items()}
        fd = OracleLoss(kind, overrides, q[i], v[i], mask[i], dg[i], dce0[i]).gradient(r)
        worst = max(worst, _rel_err({k: out[k][i] for k in REF_KEYS}, fd))
    print(f"\nrefs_grad {kind}{' tight' if overrides else ''}: GPU vs emulator {err:.1e}, vs 80-bit differences (64 envs) "
          f"{worst:.1e} of the gradient's norm")
    assert err < 1e-11 and worst < 1e-8


def _margin(e, prob, sol, count, margin=1e-3):
    """Envs whose solution has a strict-complementarity margin (multipliers of the working set and slacks of the other
    rows bounded away from zero), so that small reference perturbations keep the working set."""
    P = {k: t.cpu().numpy() for k, t in prob.items()}
    S = {k: t.cpu().numpy() for k, t in sol.items()}
    picked = []
    for i in np.where(S["status"] == 0)[0]:
        n_, neq, nin = (int(x) for x in P["sizes"][i])
        w = int((S["active"][i] >= 0).sum())
        lam = S["lambda"][i][:w]
        slack = np.delete(P["CI"][i][:nin, :n_] @ S["x"][i][:n_] + P["ci0"][i][:nin], S["active"][i][:w])
        ci0 = P["ci0"][i][:nin]
        if lam.min(initial=1.0) > margin * max(1.0, np.abs(lam).max(initial=0.0)) and \
                slack.min(initial=1.0) > margin * (1 + np.abs(ci0[np.abs(ci0) < 1e9]).max(initial=0.0)):
            picked.append(int(i))
    return picked[:count]


@pytest.mark.gpu
def test_tick_layer_forward_gradcheck_and_differences(live):
    """tick_layer's forward equals problem_data + qp_solve bit for bit; on envs with a complementarity margin gradcheck
    passes with respect to each reference tensor, and central differences of tau, dv and f through the GPU forward agree
    with the backward along random reference directions on the envs whose working set is the same at +-h."""
    import torch

    n = 1024
    s, q, v, mask, refs = _inputs("v1", n, 92, TIGHT)
    mask[::97] = 0  # envs in flight: with tight limits some have a complementarity margin
    e = _controller("v1", n, TIGHT).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    out = e.tick_layer(qd, vd, md, rd)
    prob = e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
    sol = e.qp_solve(prob)
    assert torch.equal(out["tau"], sol["tau"]) and torch.equal(out["dv"], sol["x"][:, :e.nv])
    assert torch.equal(out["status"], sol["status"]) and torch.equal(out["iters"], sol["iters"])
    x = sol["x"]
    for i in range(n):
        m = int(mask[i])
        slots = [f for f in (0, 1) if (m >> f) & 1]
        want = torch.zeros(24, dtype=torch.float64, device=e.device)
        for s_, f in enumerate(slots):
            want[12 * f:12 * f + 12] = x[i, e.nv + 12 * s_:e.nv + 12 * s_ + 12]
        assert torch.equal(out["f"][i], want)

    picked = _margin(e, prob, sol, 3)
    assert len(picked) == 3, picked
    idx = torch.as_tensor(picked, device=e.device)
    sub = (qd[idx].contiguous(), vd[idx].contiguous(), md[idx].contiguous())
    for key in REF_KEYS:
        base = {k: t[idx].clone() for k, t in rd.items()}

        def fn(t, key=key, base=base):
            r = dict(base)
            r[key] = t
            o = e.tick_layer(*sub, r)
            return o["tau"], o["dv"], o["f"]

        t0 = base[key].clone().requires_grad_(True)
        assert torch.autograd.gradcheck(fn, (t0,), eps=1e-6, atol=1e-5, rtol=1e-4), key

    # directional differences on the whole batch
    rng = np.random.default_rng(112)
    h = 1e-6
    errs, kept = [], 0
    base = {k: t.clone().requires_grad_(True) for k, t in rd.items()}
    o = e.tick_layer(qd, vd, md, base)
    wt = {k: torch.as_tensor(rng.standard_normal(tuple(o[k].shape)), device=e.device) for k in ("tau", "dv", "f")}
    loss = sum((o[k] * wt[k]).sum(dim=1) for k in wt)
    dirs = {k: torch.as_tensor(rng.standard_normal(tuple(t.shape)), device=e.device) for k, t in rd.items()}
    per_env = torch.autograd.grad(loss.sum(), [base[k] for k in REF_KEYS])
    ad = sum((g * dirs[k]).sum(dim=1) for g, k in zip(per_env, REF_KEYS))
    with torch.no_grad():
        lp = e.tick_layer(qd, vd, md, {k: rd[k] + h * dirs[k] for k in rd})
        lm = e.tick_layer(qd, vd, md, {k: rd[k] - h * dirs[k] for k in rd})
        act = [e.qp_solve(e.problem_data(qd, vd, md, {k: rd[k] + sg * h * dirs[k] for k in rd},
                                         parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS))["active"] for sg in (1, -1)]
    fd = sum(((lp[k] - lm[k]) * wt[k]).sum(dim=1) for k in wt) / (2 * h)
    same = (act[0] == sol["active"]).all(dim=1) & (act[1] == sol["active"]).all(dim=1) & (sol["status"] == 0) & \
        (lp["status"] == 0) & (lm["status"] == 0)
    kept = int(same.sum())
    rel = ((fd - ad).abs() / (1e-2 + ad.abs()))[same].cpu().numpy()
    print(f"\ntick_layer directional differences: {kept}/{n} envs keep their working set; relative error median "
          f"{np.median(rel):.1e}, 99th percentile {np.quantile(rel, 0.99):.1e}, max {rel.max():.1e}")
    assert kept >= 0.5 * n
    assert np.median(rel) < 1e-6 and np.quantile(rel, 0.99) < 1e-2


@pytest.mark.gpu
def test_tick_layer_fit_recovers_references(live):
    """torch.optim (L-BFGS) recovers a perturbed CoM position reference and a swing-foot position reference (right foot
    swinging: a foot in contact pins its own acceleration, so its task reference does not show in dv) from the dv they
    produced, on the envs whose working set is the same at the true and at the perturbed reference: the loss falls by
    orders of magnitude, and on the envs whose working set stays fixed the recovered reference matches to within
    10 residual / sigma_min of d dv / d ref (on some envs a CoM direction barely shows in dv: sigma_min reaches 1e-8), with
    a median error below 1e-5."""
    import torch

    n = 256
    s, q, v, mask, refs = _inputs("v1", n, 121)
    e = _controller("v1", n).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    active = lambda r, sub: e.qp_solve(e.problem_data(*sub, r, parts=e.PROBLEM_PARTS))["active"]  # noqa: E731
    gen = torch.Generator(device=e.device).manual_seed(122)
    for key in ("com", "foot_rf"):
        d0 = 2e-3 * torch.randn((n, 3), generator=gen, dtype=torch.float64, device=e.device)
        moved = dict(rd)
        moved[key] = torch.cat([rd[key][:, :3] + d0, rd[key][:, 3:]], dim=1)
        keep = (active(rd, (qd, vd, md)) == active(moved, (qd, vd, md))).all(dim=1)
        if key == "foot_rf":
            keep &= md == 1
        idx = torch.nonzero(keep).flatten()
        sub = (qd[idx].contiguous(), vd[idx].contiguous(), md[idx].contiguous())
        rs = {k: t[idx].contiguous() for k, t in rd.items()}
        target = e.tick_layer(*sub, rs)["dv"].clone()
        tact = active(rs, sub)
        delta = d0[idx].clone().requires_grad_(True)
        opt = torch.optim.LBFGS([delta], lr=1.0, max_iter=100, history_size=100, tolerance_grad=1e-20,
                                tolerance_change=1e-30, line_search_fn="strong_wolfe")

        def refs_of(dl):
            r = dict(rs)
            r[key] = torch.cat([rs[key][:, :3] + dl, rs[key][:, 3:]], dim=1)
            return r

        def loss_fn():
            return ((e.tick_layer(*sub, refs_of(delta))["dv"] - target) ** 2).sum()

        def closure():
            opt.zero_grad()
            lo = loss_fn()
            lo.backward()
            return lo

        with torch.no_grad():
            l0 = float(loss_fn())
        for _ in range(6):
            opt.step(closure)
        with torch.no_grad():
            dl = delta.detach()
            l1 = float(loss_fn())
            fixed = (active(refs_of(dl), sub) == tact).all(dim=1)
            # per env: residual and the smallest singular value of d dv / d ref (central differences through the forward):
            # a reference that barely shows in dv is recovered only to residual / sigma_min
            res = (e.tick_layer(*sub, refs_of(dl))["dv"] - target).norm(dim=1)
            h = 1e-6
            eye = torch.eye(3, dtype=torch.float64, device=e.device)
            J = torch.stack([(e.tick_layer(*sub, refs_of(dl + h * eye[k]))["dv"] - e.tick_layer(*sub, refs_of(dl - h * eye[k]))["dv"])
                             / (2 * h) for k in range(3)], dim=2)
            smin = torch.linalg.svdvals(J)[:, -1]
        err = dl.norm(dim=1)
        bound = 10 * res / smin + 1e-8
        good = fixed & (err < 1e-6)
        print(f"\nfit of {key}[:3]: {len(idx)} envs, loss {l0:.2e} -> {l1:.2e}; {int(fixed.sum())} keep their working set, "
              f"{int(good.sum())} of them recovered to 1e-6 (median error {float(err[fixed].median()):.1e}); the others within "
              f"residual / sigma_min (smallest sigma_min {float(smin[fixed].min()):.1e})")
        assert l1 < 1e-6 * l0
        assert int(fixed.sum()) >= 16 and bool((err <= bound)[fixed].all())
        assert float(err[fixed].median()) < 1e-5


@pytest.mark.gpu
def test_refs_grad_has_no_side_effects_and_checks_arguments(live):
    """A tick after refs_grad is bit-identical to one without it; refs_grad on a side stream concurrent with a tick gives
    the same result as alone; bad arguments are refused."""
    import ctypes as C

    import torch

    from tsid_control_b200 import _capi

    n = 2048
    s, q, v, mask, refs = _inputs("v1", n, 131)
    keys = ("tau", "ddq", "f", "status", "iters", "active_set")
    runs = []
    for with_grad in (False, True):
        e = _controller("v1", n).engine
        qd, vd, md, rd = _dev(e, q, v, mask, refs)
        dg, dce0 = _dev(e, *_weights(n, e.nv, mask, 132))
        outs = []
        for _ in range(2):
            if with_grad:
                alone = e.refs_grad(qd, vd, md, rd, dg, dce0)
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
        conc = e.refs_grad(qd, vd, md, rd, dg, dce0)
    e.compute(qd, vd, md, rd)
    torch.cuda.synchronize()
    for k in REF_KEYS:
        assert torch.equal(conc[k], alone[k]), k

    lib = e.lib
    ro = _capi.TsidbRefsOut(com=conc["com"].data_ptr())
    args = lambda nn=n, lay=0, nx=50, neq=18, qp=qd.data_ptr(), out=C.byref(ro): (  # noqa: E731
        e.h, nn, lay, qp, vd.data_ptr(), None, None, nx, neq, dg.data_ptr(), None, out, e._stream())
    assert lib.tsidb_refs_grad(*args()) == 0
    assert lib.tsidb_refs_grad(*args(nn=n + 1)) < 0 and b"max_envs" in lib.tsidb_last_error()
    assert lib.tsidb_refs_grad(*args(nn=0)) < 0
    assert lib.tsidb_refs_grad(*args(lay=2)) < 0 and b"layout" in lib.tsidb_last_error()
    assert lib.tsidb_refs_grad(*args(nx=49)) < 0 and b"n_max" in lib.tsidb_last_error()
    assert lib.tsidb_refs_grad(*args(neq=17)) < 0
    assert lib.tsidb_refs_grad(*args(qp=None)) < 0 and b"null" in lib.tsidb_last_error()
    assert lib.tsidb_refs_grad(*args(out=None)) < 0
    torch.cuda.synchronize()
    with pytest.raises(TypeError, match="dg"):
        e.refs_grad(qd, vd, md, rd, dg[:, :40].contiguous())
    with pytest.raises(ValueError, match="parts"):
        e.refs_grad(qd, vd, md, rd, dg, parts=("H",))
    with pytest.raises(ValueError, match="unknown references"):
        e.refs_grad(qd, vd, md, {"cop": rd["com"]}, dg)
