"""The assembled QP without the solve (tsidb_problem_data / TsidEngine.problem_data / HQPData of the mirror): every part
of every env against the oracle's dump of the same problem, and the tick's solution checked against the exported
problem with code that shares nothing with the kernels (a KKT certificate and an scipy solve)."""
import numpy as np
import pytest

import parity_log
from common import bits_to_rows, make_conf, setup
from emu_problem import EmuProblem
from oracle_py import CI_ACTUATION, CI_JOINT_BOUNDS, biped_orders
from tsid_control_b200 import synth

PARTS = ("H", "g", "CE", "ce0", "CI", "ci0")
BIG = 1e10  # open side of a two-sided row (Contact6d pyramid, base rows of TaskJointBounds)


def _metric(a, b):
    """The metric of test_dynamics_terms_match_oracle: max|a-b| / (1e-2 + max|b|)."""
    return float(np.max(np.abs(a - b)) / (1e-2 + np.max(np.abs(b)))) if np.size(b) else 0.0


def canonical_orders(orc, mask):
    """The export's order: contacts LF first; CI blocks [LF, RF, actuation, joint bounds] (those present)."""
    contacts = [f for f in (0, 1) if (mask >> f) & 1]
    ci = list(contacts) + ([CI_ACTUATION] if orc.cc.use_torque_bounds else []) + ([CI_JOINT_BOUNDS] if orc.cc.use_joint_bounds else [])
    return contacts, ci, orc.orders(mask)[2]


def compare_env(exp, i, dump, worst):
    """Env i of an export against an oracle dump in the same orders: sizes exact, padding exactly zero, every part within
    the metric (ci0: the finite bounds by the metric, the +-1e10 ones exactly)."""
    n, neq, nin = dump["n"], dump["neq"], dump["nin"]
    assert tuple(int(x) for x in exp["sizes"][i]) == (n, neq, nin)
    lead = {"H": (n, n), "g": (n,), "CE": (neq, n), "ce0": (neq,), "CI": (nin, n), "ci0": (nin,)}
    for k, shp in lead.items():
        a = exp[k][i]
        body = a[tuple(slice(0, m) for m in shp)]
        pad = a.copy()
        pad[tuple(slice(0, m) for m in shp)] = 0.0
        assert not pad.any(), f"{k}: padding is not zero"
        b = dump[k]
        if k == "ci0":
            big = np.abs(b) >= BIG
            assert np.array_equal(body[big], b[big])
            body, b = body[~big], b[~big]
        worst[k] = max(worst.get(k, 0.0), _metric(body, b))


# ------------------------------------------------------------------ CPU: the kernel bodies on the host emulator
@pytest.mark.parametrize("kind,maskval", [("v1", 3), ("v1", 1), ("v1", 2), ("v1", 0), ("v0", 3), ("v0", 1)])
def test_emulated_problem_export_matches_oracle(kind, maskval):
    s = setup(kind)
    orc = s["oracle"]
    n = 6
    q, v = synth.random_states(s["q0"], n, 51)
    step = (0.3, 0.2, 0.2, 0.5) if kind == "v1" else (0.1, 0.1275, 0.05, 0.7)
    _, refs = synth.walking_batch(s["refs"], n, 51, *step, float(s["refs"]["com"][2]))
    mask = np.full(n, maskval, np.uint8)
    exp = EmuProblem(s["cm"], s["cc"]).problem(q, v, mask, refs)
    worst = {}
    for i in range(n):
        r = {k: a[i] for k, a in refs.items()}
        d = orc.tick(q[i], v[i], maskval, r, dump=True, orders=canonical_orders(orc, maskval))["dump"]
        compare_env(exp, i, d, worst)
    print(f"\nemulated export vs oracle ({kind}, mask {maskval}):", {k: f"{x:.1e}" for k, x in worst.items()})
    assert all(x < 1e-10 for x in worst.values()), worst


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


def _batch(kind, n, seed, overrides=()):
    s = setup(kind, overrides=tuple(overrides))
    q, v = synth.random_states(s["q0"], n, seed)
    step = (0.3, 0.2, 0.2, 0.5) if kind == "v1" else (0.1, 0.1275, 0.05, 0.7)
    mask, refs = synth.walking_batch(s["refs"], n, seed, *step, float(s["refs"]["com"][2]))
    mask[::97] = 0  # some envs in flight
    return s, q, v, mask, refs


def _dev(e, q, v, mask, refs):
    import torch

    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=e.device)
    return t(q), t(v), t(mask), {k: t(a) for k, a in refs.items()}


def _export(e, q, v, mask, refs, **kw):
    import torch

    out = e.problem_data(*_dev(e, q, v, mask, refs), **kw)
    torch.cuda.synchronize()
    return {k: t.cpu().numpy() for k, t in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,overrides,n", [
    ("v1", (), 2048),
    ("v0", (), 2048),
    ("v1", (("tau_max_scaling", 0.08), ("v_max_scaling", 0.1)), 512),
])
def test_problem_export_matches_oracle(kind, overrides, n, live):
    """Every part of every env of a walking batch (per-env references, all four contact masks) against the oracle's
    dump of the problem in the export's orders; the tight-limit conf makes the actuation and joint-bound rows bind."""
    s, q, v, mask, refs = _batch(kind, n, 61, overrides)
    orc = s["oracle"]
    e = _controller(kind, n, overrides).engine
    exp = _export(e, q, v, mask, refs)
    assert set(np.unique(mask)) == {0, 1, 2, 3}
    worst = {}
    for i in range(n):
        m = int(mask[i])
        d = orc.tick(q[i], v[i], m, {k: a[i] for k, a in refs.items()}, dump=True, orders=canonical_orders(orc, m))["dump"]
        compare_env(exp, i, d, worst)
    name = f"problem_export_{kind}" + ("_tight_limits" if overrides else "")
    print(f"\n{name} vs oracle (max |a-b| / (1e-2 + max|b|)), {n} envs:", {k: f"{x:.1e}" for k, x in worst.items()})
    parity_log.record(name, worst)
    assert all(x < 1e-10 for x in worst.values()), worst


def _compact_rows(e, mask):
    """tsidb_ci_row numbering (block, side, i) -> row of the env's compact CI."""
    m = int(mask)
    blocks = [b for b in (0, 1) if (m >> b) & 1] + ([2] if e.cc.use_torque_bounds else []) + ([3] if e.cc.use_joint_bounds else [])
    rows, off = {}, 0
    for b in blocks:
        nr = (17, 17, e.na, e.nv)[b]
        for side in (0, 1):
            for i in range(nr):
                rows[(b, side, i)] = off + side * nr + i
        off += 2 * nr
    return rows


def kkt_residuals(H, g, CE, ce0, CI, ci0, x, lam):
    """Relative KKT residuals of (x, lam) for min 1/2 x'Hx + g'x s.t. CE x + ce0 = 0, CI x + ci0 >= 0 (mu by least
    squares).  Each residual is scaled by the size of the terms it sums (rows with a +-1e10 bound are never tight and
    are left out of the feasibility scale)."""
    eq = CE @ x + ce0
    s_eq = np.abs(CE) @ np.abs(x) + np.abs(ce0)
    sl = CI @ x + ci0
    s_in = np.abs(CI) @ np.abs(x) + np.where(np.abs(ci0) >= BIG, 0.0, np.abs(ci0))
    rhs = H @ x + g - CI.T @ lam
    mu = np.linalg.lstsq(CE.T, rhs, rcond=None)[0]
    st = rhs - CE.T @ mu
    s_st = np.abs(H) @ np.abs(x) + np.abs(g) + np.abs(CI.T) @ np.abs(lam) + np.abs(CE.T) @ np.abs(mu)
    act = lam != 0
    return {
        "equality": float(np.max(np.abs(eq) / (1e-2 + s_eq))),
        "feasibility": float(np.max(np.maximum(-sl, 0.0) / (1e-2 + s_in))),
        "dual": float(max(0.0, -lam.min()) / (1e-2 + np.abs(lam).max())),
        "complementarity": float(np.max(np.abs(sl[act]) / (1e-2 + s_in[act]))) if act.any() else 0.0,
        "stationarity": float(np.max(np.abs(st) / (1e-2 + s_st))),
    }


def scipy_qp(H, g, CE, ce0, CI, ci0):
    """The QP solved by scipy alone: SLSQP from x = 0, then the equality-constrained KKT system of the rows SLSQP left
    tight (SLSQP stops at its iteration limit on the ill-conditioned force block, cond(H) ~ 1e8, with the working set
    right but the wrench only to ~1e-3).  Returns x and (SLSQP status, tight rows)."""
    from scipy.optimize import minimize

    cons = [{"type": "eq", "fun": lambda y: CE @ y + ce0, "jac": lambda y: CE},
            {"type": "ineq", "fun": lambda y: CI @ y + ci0, "jac": lambda y: CI}]
    sol = minimize(lambda y: 0.5 * y @ H @ y + g @ y, np.zeros(len(g)), jac=lambda y: H @ y + g, constraints=cons,
                   method="SLSQP", options={"ftol": 1e-15, "maxiter": 1000})
    y = sol.x
    scale = 1.0 + np.abs(CI) @ np.abs(y) + np.where(np.abs(ci0) >= BIG, 0.0, np.abs(ci0))
    tight = (CI @ y + ci0) <= 1e-7 * scale
    A, b = np.vstack([CE, CI[tight]]), np.concatenate([ce0, ci0[tight]])
    K = np.block([[H, A.T], [A, np.zeros((len(b), len(b)))]])
    z = np.linalg.lstsq(K, np.concatenate([-g, -b]), rcond=None)[0]
    return z[:len(g)], (int(sol.status), int(tight.sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,bar", [("v1", 1e-8), ("v0", 1e-7)])
def test_tick_solution_certified_on_exported_problem(kind, bar, live):
    """The tick's solution x = (ddq, f of the feet in contact) and its multipliers (sol.lambda, mapped from tsidb_ci_row
    numbering onto the compact rows) satisfy the KKT conditions of the exported QP, for every env with status 0.  The
    legacy conf (fMin = 0, cond(H) ~ 1e8) is held to 1e-7.  For 16 envs the
    exported QP is also solved from scratch by scipy (SLSQP, then the KKT system of the rows it leaves tight): dv and tau
    agree with the tick."""
    import torch

    n = 1024
    s, q, v, mask, refs = _batch(kind, n, 62)
    e = _controller(kind, n).engine
    qd, vd, md, rd = _dev(e, q, v, mask, refs)
    t = e.compute(qd, vd, md, rd, aux=True)
    torch.cuda.synchronize()
    tick = {k: getattr(t, k).cpu().numpy().copy() for k in ("tau", "ddq", "f", "status", "lam", "lam_row")}
    exp = _export(e, q, v, mask, refs)
    worst, n_ok, scipy_err = {}, 0, {"ddq": 0.0, "tau": 0.0}
    ok = np.where(tick["status"] == 0)[0]
    assert len(ok) >= 0.95 * n
    for i in ok:
        n_, neq, nin = (int(x) for x in exp["sizes"][i])
        H, g = exp["H"][i][:n_, :n_], exp["g"][i][:n_]
        CE, ce0, CI, ci0 = exp["CE"][i][:neq, :n_], exp["ce0"][i][:neq], exp["CI"][i][:nin, :n_], exp["ci0"][i][:nin]
        m = int(mask[i])
        x = np.concatenate([tick["ddq"][i]] + [tick["f"][i][12 * f:12 * f + 12] for f in (0, 1) if (m >> f) & 1])
        lam = np.zeros(nin)
        used = tick["lam_row"][i] >= 0
        rows = _compact_rows(e, m)
        for r, l in zip(bits_to_rows(e.na, e.nv, [int(b) for b in tick["lam_row"][i][used]]), tick["lam"][i][used]):
            lam[rows[r]] = l
        for k, val in kkt_residuals(H, g, CE, ce0, CI, ci0, x, lam).items():
            worst[k] = max(worst.get(k, 0.0), val)
        n_ok += 1
        if n_ok <= 16:
            y, _ = scipy_qp(H, g, CE, ce0, CI, ci0)
            # tau = M_a dv - J_a^T f + h_a: the lower actuation rows are [M_a | -Jc_a^T] y - (tau_min - h_a)
            a0 = _compact_rows(e, m)[(2, 0, 0)]
            tau_y = CI[a0:a0 + e.na] @ y + ci0[a0:a0 + e.na] + e.cc.tau_min[:e.na]
            scipy_err["ddq"] = max(scipy_err["ddq"], _metric(y[:e.nv], tick["ddq"][i]))
            scipy_err["tau"] = max(scipy_err["tau"], _metric(np.asarray(tau_y), tick["tau"][i]))
    print(f"\nKKT residuals of the tick's solution on the exported QP ({kind}, {n_ok} envs):",
          {k: f"{x:.1e}" for k, x in worst.items()}, "scipy SLSQP vs tick:", {k: f"{x:.1e}" for k, x in scipy_err.items()})
    parity_log.record(f"problem_kkt_{kind}", {**worst, **{f"slsqp_{k}": x for k, x in scipy_err.items()}, "envs": n_ok})
    assert all(x < bar for x in worst.values()), worst
    assert all(x < 1e-6 for x in scipy_err.values()), scipy_err


@pytest.mark.gpu
def test_problem_export_leaves_the_tick_unchanged(live):
    """A problem_data call before and between two ticks (scheduling hint on) changes no output bit of the ticks; layout 1
    inputs give the same export bit for bit; a part passed as NULL is not written; bad arguments are refused."""
    import ctypes as C

    import torch

    from tsid_control_b200 import _capi

    n = 2048
    s, q, v, mask, refs = _batch("v1", n, 63)
    keys = ("tau", "ddq", "f", "status", "iters", "active_set")
    runs = []
    for with_export in (False, True):
        e = _controller("v1", n).engine
        e.set_sched_hint(True)
        args = _dev(e, q, v, mask, refs)
        outs = []
        for _ in range(2):
            if with_export:
                e.problem_data(*args)
            t = e.compute(*args)
            torch.cuda.synchronize()
            outs.append({k: getattr(t, k).cpu().numpy().copy() for k in keys})
        runs.append(outs)
    for a, b in zip(*runs):
        for k in keys:
            assert np.array_equal(a[k], b[k]), k

    # layout 1 ([dof][N]) inputs, a NULL part, errors: through the C ABI
    lib = e.lib
    qd, vd, md, rd = args
    nx, neq, nin = e.problem_sizes()
    assert (nx, neq, nin) == (50, 18, 160)
    ref = e.problem_data(qd, vd, md, rd)
    f64 = dict(dtype=torch.float64, device=e.device)
    out = {"H": torch.full((n, nx, nx), 7.0, **f64), "g": torch.full((n, nx), 7.0, **f64), "CE": torch.full((n, neq, nx), 7.0, **f64),
           "ce0": torch.full((n, neq), 7.0, **f64), "CI": torch.full((n, nin, nx), 7.0, **f64), "ci0": torch.full((n, nin), 7.0, **f64),
           "sizes": torch.full((n, 3), 7, dtype=torch.int32, device=e.device)}
    po = _capi.TsidbProblemOut(**{k: t.data_ptr() for k, t in out.items()})
    po.CI = None
    keep = [t.t().contiguous() for t in rd.values()]
    r = _capi.TsidbRefs(**{k: t.data_ptr() for k, t in zip(rd, keep)})
    qt, vt = qd.t().contiguous(), vd.t().contiguous()
    _capi.check(lib.tsidb_problem_data(e.h, n, 1, qt.data_ptr(), vt.data_ptr(), md.data_ptr(), C.byref(r), C.byref(po),
                                       e._stream()), "tsidb_problem_data")
    torch.cuda.synchronize()
    for k in ("H", "g", "CE", "ce0", "ci0", "sizes"):
        assert torch.equal(out[k], ref[k]), k
    assert bool((out["CI"] == 7.0).all())
    assert lib.tsidb_problem_data(e.h, n + 1, 0, qd.data_ptr(), vd.data_ptr(), None, None, C.byref(po), e._stream()) < 0
    assert b"max_envs" in lib.tsidb_last_error()
    assert lib.tsidb_problem_data(e.h, n, 0, qd.data_ptr(), vd.data_ptr(), None, None, None, e._stream()) < 0
    assert lib.tsidb_problem_data(e.h, n, 2, qd.data_ptr(), vd.data_ptr(), None, None, C.byref(po), e._stream()) < 0


def _mirror_compare(ctrl, s, orders, t, q, v, mask):
    """The mirror's HQPData of one robot against the oracle's dump of that robot's problem in the reference's orders."""
    hqp = ctrl.formulation.computeProblemData(t, q, v)
    refs = {k: t[0].cpu().numpy() for k, t in ctrl.refs.items()}
    d = s["oracle"].tick(q, v, mask, refs, dump=True, orders=orders)["dump"]
    worst = {}
    for k in PARTS:
        a, b = np.asarray(getattr(hqp, k)), d[k]
        assert a.shape == b.shape, (k, a.shape, b.shape)
        if k == "ci0":
            big = np.abs(b) >= BIG
            assert np.array_equal(a[big], b[big])
            a, b = a[~big], b[~big]
        worst[k] = _metric(a, b)
    return worst


@pytest.mark.gpu
def test_mirror_hqpdata_matches_oracle_in_reference_order(live):
    """HQPData of the drop-in formulation carries H, g, CE, ce0, CI, ci0 of the single-robot view in the reference's own
    variable and row order: Biped (legacy, RF contact first) and WalkController after removeRigidContact and
    addRigidContact of LF (the re-added contact goes last)."""
    s0 = setup("v0")
    b = _controller("v0", 1)
    q0, v0 = synth.random_states(s0["q0"], 1, 64)
    assert biped_orders(3)[1] == list(s0["oracle"].orders(3)[1])  # the legacy conf has no joint-bounds task
    w0 = _mirror_compare(b, s0, s0["oracle"].orders(3), 0.0, q0[0], v0[0], 3)

    s1 = setup("v1")
    c = _controller("v1", 1)
    name_lf = c.contactLF.name
    c.formulation.removeRigidContact(name_lf, 0.0)
    c.formulation.addRigidContact(c.contactLF, c.conf.w_forceRef, 1.0, 1)
    contacts = list(c._contact_order)
    assert contacts == [1, 0]
    ci = list(c._ci_order)
    cost = s1["oracle"].orders(3)[2]
    q1, v1 = synth.random_states(s1["q0"], 1, 65)
    w1 = _mirror_compare(c, s1, (contacts, ci, cost), 0.0, q1[0], v1[0], 3)
    print("\nmirror HQPData vs oracle: Biped", {k: f"{x:.1e}" for k, x in w0.items()},
          "WalkController (LF re-added)", {k: f"{x:.1e}" for k, x in w1.items()})
    parity_log.record("problem_mirror", {**{f"biped_{k}": x for k, x in w0.items()}, **{f"walk_{k}": x for k, x in w1.items()}})
    assert all(x < 1e-10 for x in list(w0.values()) + list(w1.values())), (w0, w1)
