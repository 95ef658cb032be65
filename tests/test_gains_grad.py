"""Differentiating with respect to the task gains and weights (tsidb_set_gains / tsidb_gains_grad / TsidEngine.gains,
set_gains, gains_grad and tick_layer's gains): the adjoint of the export in the gains against central differences of the
80-bit oracle rebuilt with perturbed confs, its unread entries and exact zeros, layouts and the nvcc spill bound on the
host emulator; on the GPU the kernel against the emulator, set_gains against a fresh handle, the autograd layer against
gradcheck and differences through the GPU forward, and a fit that recovers gains."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from common import setup
from emu_gains_grad import EmuGainsGrad
from oracle_py import Oracle
from test_problem_data import canonical_orders
from tsid_control_b200 import synth
from tsid_control_b200._capi import GAIN_FIELDS, GAINS_LEN, TsidbConf

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tsid_control_b200", "csrc")
STEP = {"v1": (0.3, 0.2, 0.2, 0.5), "v0": (0.1, 0.1275, 0.05, 0.7)}
TIGHT = (("tau_max_scaling", 0.08), ("v_max_scaling", 0.1))
# column of each tsidb_gains field in the gradient
COL = {}
_c = 0
for _k, _n in GAIN_FIELDS:
    COL[_k] = _c
    _c += _n


def _inputs(kind, n, seed, overrides=()):
    s = setup(kind, overrides=tuple(overrides))
    q, v = synth.random_states(s["q0"], n, seed)
    mask, refs = synth.walking_batch(s["refs"], n, seed, *STEP[kind], float(s["refs"]["com"][2]))
    return s, q, v, mask, refs


def _weights(n, nv, masks, seed):
    """Random dL/dH, dL/dg, dL/dce0 on every entry the adjoint reads (H's dv block and the force blocks of the feet in
    contact, g[:nv], the contact rows of ce0); NaN everywhere else."""
    rng = np.random.default_rng(seed)
    nx = nv + 24
    dH, dg, dce0 = np.full((n, nx, nx), np.nan), np.full((n, nx), np.nan), np.full((n, 18), np.nan)
    for i, m in enumerate(masks):
        nc = (int(m) & 1) + ((int(m) >> 1) & 1)
        dH[i, :nv, :nv] = rng.standard_normal((nv, nv))
        for s_ in range(nc):
            b = slice(nv + 12 * s_, nv + 12 * s_ + 12)
            dH[i, b, b] = rng.standard_normal((12, 12))
        dg[i, :nv] = rng.standard_normal(nv)
        dce0[i, 6:6 + 6 * nc] = rng.standard_normal(6 * nc)
    return dH, dg, dce0


def _conf_with(cc, k, j, val):
    c = TsidbConf.from_buffer_copy(cc)
    f = getattr(c, k)
    if isinstance(f, float):
        setattr(c, k, val)
    else:
        f[j] = val
    return c


def _conf_get(cc, k, j):
    f = getattr(cc, k)
    return f if isinstance(f, float) else f[j]


class OracleGainsLoss:
    """L(conf) = <dH, H> + dg . g + dce0 . ce0 of one env from the 80-bit oracle's dump of its problem (export order); the
    NaN entries of the weights are left out."""

    def __init__(self, s, q, v, mask, refs, dH, dg, dce0):
        self.cm, self.cc = s["cm"], s["cc"]
        self.q, self.v, self.mask, self.refs = q, v, int(mask), refs
        self.W = (dH, dg, dce0)
        self.orders = canonical_orders(Oracle(self.cm, self.cc, "liboracle_ld.so"), self.mask)

    def __call__(self, cc):
        d = Oracle(self.cm, cc, "liboracle_ld.so").tick(self.q, self.v, self.mask, self.refs, dump=True,
                                                        orders=self.orders)["dump"]
        n, neq = d["n"], d["neq"]
        tot = 0.0
        for w, b in zip(self.W, (d["H"], d["g"], d["ce0"])):
            ww = w[tuple(slice(0, m) for m in b.shape)]
            tot += float(np.sum(np.where(np.isnan(ww), 0.0, ww) * b))
        return tot

    def gradient(self, skip=()):
        """Central differences in every tsidb_gains entry, in gradient column order; entries in `skip` (names) and
        posture entries past na are left at zero.  H, g and ce0 are affine in each entry, so the step only trades the
        dump's double rounding (eps |L| / h): relative steps 1e-3 |p| (w_force_reg is 1e-5; at 1e-5 |p| its difference
        carries 3e-5 of rounding)."""
        na = self.cm.nb - 1
        fd = np.zeros(GAINS_LEN)
        for k, n in GAIN_FIELDS:
            if k in skip:
                continue
            for j in range(n):
                if k in ("kp_posture", "kd_posture") and j >= na:
                    continue
                p = _conf_get(self.cc, k, j)
                h = 1e-3 * abs(p) if p != 0.0 else 1e-3
                fd[COL[k] + j] = (self(_conf_with(self.cc, k, j, p + h)) - self(_conf_with(self.cc, k, j, p - h))) / (2 * h)
        return fd


def _zero_cols(kind, na, mask):
    """Columns the export does not use: posture past na, the AM task when off, the contact gains and w_force_reg in
    flight."""
    cols = list(range(COL["kp_posture"] + na, COL["kp_posture"] + 23)) + list(range(COL["kd_posture"] + na, COL["kd_posture"] + 23))
    if kind == "v1":
        cols += [COL["kp_am"] + k for k in range(3)] + [COL["w_am"]]
    if mask == 0:
        cols += list(range(COL["kp_contact"], COL["kp_contact"] + 12)) + [COL["w_force_reg"]]
    return cols


# ------------------------------------------------------------------ CPU: the kernel body on the host emulator
@pytest.mark.parametrize("kind", ["v1", "v0"])
@pytest.mark.parametrize("maskval", [3, 1, 2, 0])
def test_emulated_gains_grad_matches_oracle_differences(kind, maskval):
    """Every tsidb_gains entry, two walking envs per contact mask (v0 has the AM task on): the emulated adjoint against
    central differences of L = <dH, H> + dg . g + dce0 . ce0 from the 80-bit oracle rebuilt with a perturbed conf, with NaN
    in every unread entry.  Bar: 1e-8 of the gradient's norm; the exact zeros are exact."""
    n = 2
    s, q, v, _, refs = _inputs(kind, n, 171 + maskval)
    mask = np.full(n, maskval, np.uint8)
    emu = EmuGainsGrad(s["cm"], s["cc"], s["refs"])
    dH, dg, dce0 = _weights(n, emu.nv, mask, 172)
    G = emu.gains_grad(q, v, mask, refs, dH, dg, dce0)
    assert np.isfinite(G).all()
    worst = 0.0
    skip = ("kp_am", "w_am") if kind == "v1" else ()
    for i in range(n):
        r = {k: a[i].copy() for k, a in refs.items()}
        fd = OracleGainsLoss(s, q[i], v[i], maskval, r, dH[i], dg[i], dce0[i]).gradient(skip)
        worst = max(worst, float(np.abs(G[i] - fd).max()) / float(np.linalg.norm(G[i])))
        assert not G[i][_zero_cols(kind, emu.na, maskval)].any()
    print(f"\nemulated gains_grad vs 80-bit central differences ({kind}, mask {maskval}): {worst:.1e} of the norm")
    assert worst < 1e-8


@pytest.mark.parametrize("kind", ["v1", "v0"])
def test_emulated_unread_entries_nulls_and_layouts(kind):
    """NaN or any other value in every unread entry gives the same gradient bit for bit; a NULL part counts as zero;
    layout 1 gives the transpose of layout 0 bit for bit; the contact gains of a foot not in contact get nothing from it
    (one foot in contact: the shared column equals the gradient with that foot's rows alone)."""
    n = 4
    s, q, v, _, refs = _inputs(kind, n, 181)
    mask = np.array([3, 1, 2, 0], np.uint8)
    emu = EmuGainsGrad(s["cm"], s["cc"], s["refs"])
    dH, dg, dce0 = _weights(n, emu.nv, mask, 182)
    g0 = emu.gains_grad(q, v, mask, refs, dH, dg, dce0)
    rng = np.random.default_rng(183)
    fill = lambda a: np.where(np.isnan(a), rng.standard_normal(a.shape), a)  # noqa: E731
    assert np.array_equal(g0, emu.gains_grad(q, v, mask, refs, fill(dH), fill(dg), fill(dce0)))
    assert np.array_equal(g0, emu.gains_grad(q, v, mask, refs, dH, dg, dce0, layout=1))
    zero = lambda a: np.where(np.isnan(a), np.nan, 0.0)  # noqa: E731
    for which in range(3):
        parts = [dH, dg, dce0]
        x = emu.gains_grad(q, v, mask, refs, *[None if k == which else p for k, p in enumerate(parts)])
        y = emu.gains_grad(q, v, mask, refs, *[zero(p) if k == which else p for k, p in enumerate(parts)])
        assert np.array_equal(x, y), which
    for i, m in enumerate(mask):
        assert not g0[i][_zero_cols(kind, emu.na, int(m))].any()
    # with one foot in contact, the other foot's rows of dce0 are not read even when they hold numbers
    d2 = dce0.copy()
    d2[1, 12:18] = 1e3
    d2[2, 12:18] = 1e3
    assert np.array_equal(g0, emu.gains_grad(q, v, mask, refs, dH, dg, d2))


def _ptxas_lines(text, name):
    m = re.search(r"Compiling entry function '(_Z\d+" + name + r"[^']*)'.*?\n(.*?)\n(.*?Used (\d+) registers[^\n]*)", text, re.S)
    spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", m.group(2) + m.group(3))
    return int(m.group(4)), int(spill.group(1)), int(spill.group(2))


def test_gains_grad_kernel_spills_within_the_dynamics_kernel():
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
        new = _ptxas_lines(r.stderr, f"tsidb_gains_grad_kernelILi{nv}E")
        print(f"\nnv {nv}: dynamics kernel {dyn}, gains_grad kernel {new} (registers, spill stores, spill loads)")
        assert new[1] <= dyn[1] and new[2] <= dyn[2]
        assert new[0] <= 168


# ------------------------------------------------------------------ GPU
_LIVE = []


@pytest.fixture
def live():
    yield _LIVE
    while _LIVE:
        _LIVE.pop().close()


def _engine(kind, n, overrides=(), cc=None):
    """A TsidEngine of `kind` (its own conf, or the C conf `cc` in place of it)."""
    from common import make_conf
    from tsid_control_b200._capi import check
    from tsid_control_b200.engine import TsidEngine

    s = setup(kind, overrides=tuple(overrides))
    conf = make_conf(kind, overrides)
    if kind == "v1":
        e = TsidEngine(s["model"], conf, conf.lf_fixed_joint, conf.rf_fixed_joint, legacy=False, max_envs=n)
    else:
        e = TsidEngine(s["model"], conf, conf.lf_frame_name, conf.rf_frame_name, legacy=True, max_envs=n)
    _LIVE.append(e)
    if cc is not None:
        e.close()
        h = C.c_void_p()
        check(e.lib.tsidb_create(C.byref(e.cm), C.byref(cc), n, 0, C.byref(h)), "tsidb_create")
        e.h, e.cc = h, cc
    e.set_default_refs(s["refs"])
    return e


def _dev(e, *arrays):
    import torch

    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=e.device)  # noqa: E731
    return [({k: t(x) for k, x in a.items()} if isinstance(a, dict) else t(a)) for a in arrays]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,overrides", [("v1", ()), ("v0", ()), ("v1", TIGHT)])
def test_gains_grad_matches_emulator(kind, overrides, live):
    """2048-env walking batches (every contact mask, some envs in flight): tsidb_gains_grad on the GPU against the emulator
    on every env, NaN in every unread entry.  Bar: 1e-10 of each env's gradient norm (the GPU contracts to FMA)."""
    import torch

    n = 2048
    s, q, v, mask, refs = _inputs(kind, n, 201, overrides)
    mask[::97] = 0
    e = _engine(kind, n, overrides)
    dH, dg, dce0 = _weights(n, e.nv, mask, 202)
    qd, vd, md, rd, dHd, dgd, dcd = _dev(e, q, v, mask, refs, dH, dg, dce0)
    out = e.gains_grad(qd, vd, md, rd, {"H": dHd, "g": dgd, "ce0": dcd})
    flat = torch.cat([out[k] if k in out else torch.zeros(0) for k, _ in GAIN_FIELDS], dim=1).cpu().numpy()
    torch.cuda.synchronize()
    ref = EmuGainsGrad(s["cm"], s["cc"], s["refs"]).gains_grad(q, v, mask, refs, dH, dg, dce0)
    used = [c for k, nf in GAIN_FIELDS for c in range(COL[k], COL[k] + (e.na if k in ("kp_posture", "kd_posture") else nf))]
    ref = ref[:, used]
    err = float((np.abs(flat - ref).max(axis=1) / np.linalg.norm(ref, axis=1)).max())
    print(f"\ngains_grad {kind}{' tight' if overrides else ''}: GPU vs emulator {err:.1e} of the gradient's norm")
    assert err < 1e-10


def _tick_all(e, q, v, mask, refs, qd, vd, md, rd, dHd, dgd, dcd):
    """Every output a handle's gains reach, as numpy arrays: tick, compute_host, rollout, problem_data, refs_grad,
    state_grad, gains_grad."""
    import torch

    out = {}
    t = e.compute(qd, vd, md, rd)
    for k in ("tau", "ddq", "f", "status", "iters", "active_set"):
        out["tick_" + k] = getattr(t, k).cpu().numpy().copy()
    h = e.compute_host(q, v, mask, refs)
    for k, a in h.items():
        out["host_" + k] = np.array(a, copy=True)
    p = e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
    for k, a in p.items():
        out["prob_" + k] = a.cpu().numpy()
    grads = {"H": dHd, "g": dgd, "ce0": dcd}
    for k, a in e.refs_grad(qd, vd, md, rd, dgd, dcd).items():
        out["refs_" + k] = a.cpu().numpy()
    for k, a in e.state_grad(qd, vd, md, rd, {"g": dgd, "ce0": dcd}).items():
        out["state_" + k] = a.cpu().numpy()
    for k, a in e.gains_grad(qd, vd, md, rd, grads).items():
        out["gains_" + k] = a.cpu().numpy()
    n = 64
    e.gait_reset(n, dt=0.002, step_duration=0.8, step_length=0.1, step_height=0.03, com_height=float(refs["com"][0, 2]))
    r = e.rollout(qd[:n].clone(), vd[:n].clone(), 5, use_graph=False)
    torch.cuda.synchronize()
    for k in ("tau", "ddq", "f", "status"):
        out["rollout_" + k] = getattr(r, k).cpu().numpy().copy()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["v1", "v0"])
def test_set_gains_matches_a_fresh_handle_and_refuses(kind, live):
    """Setting the current values through the C setter changes no output by a bit, and through TsidEngine.set_gains is
    a no-op that leaves the gains version alone.  Setting new values (on v0 kp_am and a positive w_am among them, the
    AM task being on) gives, bit for bit, what a handle created with those values in its conf gives (tick,
    compute_host, rollout, problem_data, refs_grad, state_grad, gains_grad).  Every refused call returns < 0 and leaves
    every output as it was."""
    import torch

    from tsid_control_b200._capi import TsidbError, TsidbGains

    n = 512
    s, q, v, mask, refs = _inputs(kind, n, 211)
    e = _engine(kind, n)
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    dHd, dgd, dcd = _dev(e, *_weights(n, e.nv, mask, 212))
    dHd, dgd, dcd = (torch.nan_to_num(t) for t in (dHd, dgd, dcd))
    args = (q, v, mask, refs, qd, vd, md, rd, dHd, dgd, dcd)
    base = _tick_all(e, *args)
    lib = e.lib
    cur = TsidbGains()
    assert lib.tsidb_get_gains(e.h, C.byref(cur)) == 0
    assert lib.tsidb_set_gains(e.h, C.byref(cur)) == 0
    version = e._gains_version
    e.set_gains(e.gains())
    assert e._gains_version == version
    same = _tick_all(e, *args)
    for k in base:
        assert np.array_equal(base[k], same[k], equal_nan=True), k

    rng = np.random.default_rng(213)
    new = {k: t * torch.as_tensor(1 + 0.2 * rng.uniform(-1, 1, t.shape[0]), device=e.device) for k, t in e.gains().items()}
    e.set_gains(new)
    got = _tick_all(e, *args)
    cc = TsidbConf.from_buffer_copy(s["cc"])
    for k, t in new.items():
        vals = t.cpu().numpy()
        if vals.shape == (1,) and k.startswith("w_"):
            setattr(cc, k, float(vals[0]))
        else:
            for j, x in enumerate(vals):
                getattr(cc, k)[j] = float(x)
    assert e._gains_version == version + 1
    fresh = _tick_all(_engine(kind, n, cc=cc), *args)
    for k in got:
        assert np.array_equal(got[k], fresh[k], equal_nan=True), k
    assert not np.array_equal(got["tick_tau"], base["tick_tau"])

    assert lib.tsidb_get_gains(e.h, C.byref(cur)) == 0
    bad = []
    for field, val in (("w_foot", 0.0), ("w_com", -1.0), ("w_posture", 0.0), ("w_am", 0.0 if kind == "v0" else 1.0),
                       ("w_force_reg", -1e9),
                       ("kp_com", float("nan")), ("kd_posture", float("inf"))):
        g = TsidbGains.from_buffer_copy(cur)
        f = getattr(g, field)
        if isinstance(f, float):
            setattr(g, field, val)
        else:
            f[1] = val
        bad.append(g)
    for g in bad:
        assert lib.tsidb_set_gains(e.h, C.byref(g)) < 0
    assert lib.tsidb_set_gains(None, C.byref(cur)) < 0 and lib.tsidb_set_gains(e.h, None) < 0
    assert lib.tsidb_get_gains(e.h, None) < 0
    after = _tick_all(e, *args)
    for k in got:
        assert np.array_equal(got[k], after[k], equal_nan=True), k
    with pytest.raises(TsidbError, match="w_foot"):
        e.set_gains({"w_foot": torch.zeros(1, dtype=torch.float64)})
    with pytest.raises(ValueError, match="unknown"):
        e.set_gains({"kp": [1.0]})
    with pytest.raises(ValueError, match="expected"):
        e.set_gains({"kp_com": [1.0, 2.0]})


def _margin(prob, sol, count, margin=1e-3):
    """Envs whose solution has a strict-complementarity margin, so that small gain perturbations keep the working set."""
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
@pytest.mark.parametrize("kind", ["v1", "v0"])
def test_tick_layer_gains_jacobian_differences_and_sum(kind, live):
    """On envs with a complementarity margin, the Jacobian of tick_layer's tau, dv and f with respect to every gains
    tensor from its backward pass matches central differences to gradcheck's tolerances.  The gains are taken in relative
    coordinates gains * (1 + u), since w_force_reg is 1e-5.  (torch.autograd.gradcheck itself runs its perturbed forwards
    between the forward it differentiates and the backward, which tick_layer refuses by design.)  Central differences
    through the GPU forward agree with the per-env gains_grad along random relative directions on the envs whose working
    set stays fixed (gains and weights apart: see the step comment below); tick_layer's gradient of a shared gain equals the sum of the per-env gains_grad; the backward raises
    after an intervening set_gains; forward mode in the gains raises NotImplementedError."""
    import torch

    n = 1024
    s, q, v, mask, refs = _inputs(kind, n, 221, TIGHT)
    mask[::97] = 0
    e = _engine(kind, n, TIGHT)
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    g0 = {k: t for k, t in e.gains().items() if not (k in ("kp_am", "w_am") and not t.any())}
    prob = e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
    sol = e.qp_solve(prob)
    picked = _margin(prob, sol, 3)
    assert len(picked) == 3, picked
    idx = torch.as_tensor(picked, device=e.device)
    sub = (qd[idx].contiguous(), vd[idx].contiguous(), md[idx].contiguous())
    rsub = {k: t[idx].contiguous() for k, t in rd.items()}
    names = tuple(g0)

    def fn(*us):
        o = e.tick_layer(*sub, rsub, {k: g0[k] * (1 + u) for k, u in zip(names, us)})
        return o["tau"], o["dv"], o["f"]

    us = tuple(torch.zeros_like(g0[k]) for k in names)
    analytic = torch.autograd.functional.jacobian(fn, us)  # one forward, then one backward per output entry
    eps, worst = 1e-7, 0.0
    for j, u in enumerate(us):
        for c in range(u.numel()):
            up, um = [x.clone() for x in us], [x.clone() for x in us]
            up[j][c] += eps
            um[j][c] -= eps
            for o, (p_, m_) in enumerate(zip(fn(*up), fn(*um))):
                num = ((p_ - m_) / (2 * eps)).reshape(-1)
                ana = analytic[o][j].reshape(-1, u.numel())[:, c]
                assert torch.allclose(ana, num, rtol=1e-4, atol=1e-5), (names[j], c, o)
                worst = max(worst, float((ana - num).abs().max()))
    print(f"\ntick_layer gains Jacobian ({kind}, {len(picked)} envs) vs central differences: max |difference| {worst:.1e}")

    # per-env directional differences on the whole batch, and the shared gradient against the per-env sum
    rng = np.random.default_rng(222)
    gl = {k: t.clone().requires_grad_(True) for k, t in g0.items()}
    o = e.tick_layer(qd, vd, md, rd, gl)
    wt = {k: torch.as_tensor(rng.standard_normal(tuple(o[k].shape)), device=e.device) for k in ("tau", "dv", "f")}
    loss = sum((o[k] * wt[k]).sum() for k in wt)
    shared = torch.autograd.grad(loss, [gl[k] for k in names])
    gx = torch.zeros_like(sol["x"])
    gx[:, :e.nv] = wt["dv"]
    lf, rf = ((md.to(torch.int32) & b) != 0 for b in (1, 2))
    zero = torch.zeros((), dtype=gx.dtype, device=gx.device)
    gx[:, e.nv:e.nv + 12] = torch.where(lf[:, None], wt["f"][:, :12], torch.where(rf[:, None], wt["f"][:, 12:], zero))
    gx[:, e.nv + 12:e.nv + 24] = torch.where((lf & rf)[:, None], wt["f"][:, 12:], zero)
    qg = e.qp_grad(prob, sol, {"x": gx, "tau": wt["tau"]}, ("H", "g", "ce0"))
    per_env = e.gains_grad(qd, vd, md, rd, qg, names)
    for k, g in zip(names, shared):
        sm = per_env[k].sum(0)
        assert torch.allclose(g, sm, rtol=1e-12, atol=1e-12 * float(sm.abs().max())), k
    # Gains enter g and ce0 only, so the solves at +-h share H's factors and their differences are clean; weights change H,
    # whose refactorisation at +-h carries rounding of order eps cond(H) / h (the force block's smallest eigenvalues are
    # near hessian_reg): a larger step and a looser bar for them.  Measured on one B200: with one relative step of 1e-7
    # along gains and weights together the median relative errors were 1.2e-3 (v1) and 0.14 (v0, 99th percentile 34),
    # which failed a bar of 1e-5.  Split, with steps 1e-6 (gains) and 1e-4 (weights), v1 gave medians 1.1e-9 and 9.3e-5
    # (99th percentiles 1.9e-4 and 1.2e-2), v0 3.9e-5 for its gains (failing 1e-6) and, at 1e-4 for both, 7.4e-4 with a
    # 99th percentile of 0.36 for its weights (failing 0.1).  The legacy conf's solves are the worse conditioned, so its
    # steps are 1e-4 (gains) and 1e-3 (weights): medians 4.6e-7 and 6.0e-5, 99th percentiles 4.2e-4 and 3.6e-2.  The
    # bars sit above these by a factor of about 3 at the 99th percentile and 10 or more at the median.
    hg, hw = (1e-6, 1e-4) if kind == "v1" else (1e-4, 1e-3)
    for group, h, bars in (("gains", hg, (1e-5, 1e-2)), ("weights", hw, (1e-3, 1e-1))):
        sel = tuple(k for k in names if k.startswith("w_") == (group == "weights"))
        dirs = {k: torch.as_tensor(rng.standard_normal(tuple(g0[k].shape)), device=e.device) for k in sel}
        ad = sum((per_env[k] * g0[k] * dirs[k]).sum(dim=1) for k in sel)
        with torch.no_grad():
            lp = e.tick_layer(qd, vd, md, rd, {k: g0[k] * (1 + h * dirs[k]) for k in sel})
            act_p = e.qp_solve(e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS))["active"]
            lm = e.tick_layer(qd, vd, md, rd, {k: g0[k] * (1 - h * dirs[k]) for k in sel})
            act_m = e.qp_solve(e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS))["active"]
            e.set_gains(g0)
        fd = sum(((lp[k] - lm[k]) * wt[k]).sum(dim=1) for k in wt) / (2 * h)
        keep = (act_p == sol["active"]).all(dim=1) & (act_m == sol["active"]).all(dim=1) & (sol["status"] == 0) & \
            (lp["status"] == 0) & (lm["status"] == 0)
        rel = ((fd - ad).abs() / (1e-2 + ad.abs()))[keep].cpu().numpy()
        print(f"tick_layer {group} ({kind}) directional differences, relative step {h:g}: {int(keep.sum())}/{n} envs keep "
              f"their working set; relative error median {np.median(rel):.1e}, 99th percentile {np.quantile(rel, 0.99):.1e}")
        assert int(keep.sum()) >= 0.5 * n
        assert np.median(rel) < bars[0] and np.quantile(rel, 0.99) < bars[1]

    o = e.tick_layer(*sub, rsub, {k: t.clone().requires_grad_(True) for k, t in g0.items()})
    e.set_gains({})  # no change: the backward pass stays valid
    e.set_gains({"kp_com": g0["kp_com"] * 1.01})
    with pytest.raises(RuntimeError, match="set_gains"):
        o["tau"].sum().backward()
    e.set_gains(g0)
    with pytest.raises(NotImplementedError, match="forward mode"):
        import torch.autograd.forward_ad as fwAD

        with fwAD.dual_level():
            t = fwAD.make_dual(g0["kp_com"].clone(), torch.ones(3, dtype=torch.float64, device=e.device))
            e.tick_layer(*sub, rsub, {"kp_com": t})


@pytest.mark.gpu
def test_tick_layer_fit_recovers_gains(live):
    """torch.optim (L-BFGS) recovers CoM and posture gains perturbed by up to 5 % from the torques they produced, starting
    from the original gains, on the envs whose working set is the same at both: the loss falls by 10 orders of magnitude
    and the gains match to 1e-6 relative."""
    import torch

    n = 512
    s, q, v, mask, refs = _inputs("v1", n, 231)
    e = _engine("v1", n)
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    g0 = e.gains()
    names = ("kp_com", "kd_com", "kp_posture")
    gen = torch.Generator(device=e.device).manual_seed(232)
    true = {k: g0[k] * (1 + 0.05 * (2 * torch.rand(g0[k].shape, generator=gen, dtype=torch.float64, device=e.device) - 1))
            for k in names}
    active = lambda sub: e.qp_solve(e.problem_data(*sub, parts=e.PROBLEM_PARTS))["active"]  # noqa: E731
    a0 = active((qd, vd, md, rd))
    e.set_gains(true)
    a1 = active((qd, vd, md, rd))
    idx = torch.nonzero((a0 == a1).all(dim=1)).flatten()
    sub = (qd[idx].contiguous(), vd[idx].contiguous(), md[idx].contiguous(), {k: t[idx].contiguous() for k, t in rd.items()})
    target = e.tick_layer(*sub)["tau"].clone()
    us = {k: torch.zeros_like(g0[k]).requires_grad_(True) for k in names}
    opt = torch.optim.LBFGS(list(us.values()), lr=1.0, max_iter=100, history_size=100, tolerance_grad=1e-20,
                            tolerance_change=1e-30, line_search_fn="strong_wolfe")

    def loss_fn():
        return ((e.tick_layer(*sub, {k: g0[k] * (1 + u) for k, u in us.items()})["tau"] - target) ** 2).sum()

    def closure():
        opt.zero_grad()
        lo = loss_fn()
        lo.backward()
        return lo

    l0 = float(loss_fn().detach())
    for _ in range(4):
        opt.step(closure)
    l1 = float(loss_fn().detach())
    err = max(float(((g0[k] * (1 + us[k].detach()) - true[k]).abs() / true[k].abs()).max()) for k in names)
    print(f"\nfit of {names}: {len(idx)} envs, loss {l0:.2e} -> {l1:.2e}, largest relative gain error {err:.1e}")
    assert len(idx) >= n // 2
    assert l1 < 1e-10 * l0 and err < 1e-6


@pytest.mark.gpu
def test_tick_layer_graph_with_two_calls_sharing_gains(live):
    """Two tick_layer calls with the same gains tensors in one autograd graph (two chunks of a batch whose losses are
    summed, and a second tick from the state the first one's dv integrates to): one backward pass through both gives the
    sum of the gradients of the two calls taken alone.  Calls with different gains in one graph raise."""
    import torch

    n = 256
    s, q, v, mask, refs = _inputs("v1", n, 241)
    e = _engine("v1", n)
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    g0 = {k: t for k, t in e.gains().items() if k != "w_am"}
    half = n // 2
    parts = [tuple(x[sl].contiguous() for x in (qd, vd, md)) + ({k: t[sl].contiguous() for k, t in rd.items()},)
             for sl in (slice(0, half), slice(half, n))]
    gen = torch.Generator(device=e.device).manual_seed(242)
    w = [torch.randn((half, e.na), generator=gen, dtype=torch.float64, device=e.device) for _ in range(2)]

    def loss_of(i, gl):
        return (e.tick_layer(*parts[i], gains=gl)["tau"] * w[i]).sum()

    def grads(fn):
        gl = {k: t.clone().requires_grad_(True) for k, t in g0.items()}
        return dict(zip(gl, torch.autograd.grad(fn(gl), list(gl.values()))))

    both = grads(lambda gl: loss_of(0, gl) + loss_of(1, gl))
    alone = [grads(lambda gl, i=i: loss_of(i, gl)) for i in range(2)]
    for k in g0:
        want = alone[0][k] + alone[1][k]
        assert torch.allclose(both[k], want, rtol=1e-12, atol=1e-12 * float(want.abs().max())), k

    # a closed loop of two ticks: the second tick's state depends on the first tick's dv
    dt = 0.002
    wv = torch.randn((n, e.nv), generator=gen, dtype=torch.float64, device=e.device)

    def loop(gl):
        o1 = e.tick_layer(qd, vd, md, rd, gl)
        v1 = vd + dt * o1["dv"]
        o2 = e.tick_layer(qd, v1.contiguous(), md, rd, gl)
        return (o2["dv"] * wv).sum()

    g = grads(loop)
    assert all(torch.isfinite(t).all() for t in g.values())
    assert any(bool(t.abs().max() > 0) for t in g.values())

    gl = {k: t.clone().requires_grad_(True) for k, t in g0.items()}
    other = dict(gl, kp_com=gl["kp_com"] * 1.1)
    lo = loss_of(0, gl) + loss_of(1, other)
    with pytest.raises(RuntimeError, match="set_gains"):
        lo.backward()
    e.set_gains(g0)
