"""Solving caller-supplied QPs (tsidb_qp_solve / TsidEngine.qp_solve) and the actuation map of the export (TA, ta0).

On CPU the kernel header's qp_env runs on the host warp emulator and is compared with the oracle's eiquadprog-fast on the
same arrays; on the GPU the batched solve of exported, modified and random problems is compared with the tick, the
oracle and KKT certificates computed here."""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import parity_log
from common import bits_to_rows, canonical_active, setup
from emu_qp import EmuProblemTA, emu_qp_solve
from oracle_qp import oracle_qp_solve
from test_problem_data import (BIG, _batch, _controller, _dev, canonical_orders, kkt_residuals, live,  # noqa: F401
                               scipy_qp)
from tsid_control_b200 import synth

RTOL, ATOL = 1e-8, 1e-10  # the parity bars
QP_KEYS = ("H", "g", "CE", "ce0", "CI", "ci0")


def _env(p, i):
    """Dense, unpadded arrays of env i of a padded problem dict."""
    n, neq, nin = (int(x) for x in p["sizes"][i])
    return (p["H"][i][:n, :n], p["g"][i][:n], p["CE"][i][:neq, :n], p["ce0"][i][:neq], p["CI"][i][:nin, :n],
            p["ci0"][i][:nin])


def _close(a, b):
    """The parity bars on a vector: max |a - b| <= 1e-10 + 1e-8 max |b|."""
    a, b = np.asarray(a), np.asarray(b)
    return bool(np.max(np.abs(a - b), initial=0.0) <= ATOL + RTOL * np.max(np.abs(b), initial=0.0))


def oracle_differences(p, sol, i, max_iter):
    """Env i of a solve against oracle_qp_solve on the same arrays -> (what differs, the oracle's result): status,
    iterations and the working set (rows and order) must be equal, x and the multipliers within the parity bars."""
    n, neq, _ = (int(x) for x in p["sizes"][i])
    o = oracle_qp_solve(*_env(p, i), max_iter)
    diff = [k for k, ok in (
        ("status", int(sol["status"][i]) == o["status"]), ("iters", int(sol["iters"][i]) == o["iters"]),
        ("active", np.array_equal(sol["active"][i][:n], o["active"]) and not (sol["active"][i][n:] != -1).any()),
        ("x", _close(sol["x"][i][:n], o["x"])), ("lambda", _close(sol["lambda"][i][:n], o["lambda"])),
        ("lambda_eq", _close(sol["lambda_eq"][i][:neq], o["lambda_eq"]))) if not ok]
    return diff, o


def compare_with_oracle(p, sol, max_iter, idx=None):
    """Every env (or those in idx) against the oracle (oracle_differences).  Returns [(env, what differs, oracle)]."""
    bad = []
    for i in (range(len(p["sizes"])) if idx is None else idx):
        diff, o = oracle_differences(p, sol, i, max_iter)
        if diff:
            bad.append((i, diff, o))
    return bad


def kkt_direct(H, g, CE, ce0, CI, ci0, x, active, lam, mu):
    """Relative KKT residuals of (x, lam, mu) with the solver's own multipliers (no fit): stationarity
    H x + g - CI' lam - CE' mu = 0, primal feasibility, dual feasibility, complementarity (scaled as kkt_residuals)."""
    lam_full = np.zeros(len(ci0))
    act = active[active >= 0]
    lam_full[act] = lam[:len(act)]
    eq = CE @ x + ce0
    s_eq = np.abs(CE) @ np.abs(x) + np.abs(ce0)
    sl = CI @ x + ci0
    s_in = np.abs(CI) @ np.abs(x) + np.where(np.abs(ci0) >= BIG, 0.0, np.abs(ci0))
    st = H @ x + g - CI.T @ lam_full - CE.T @ mu
    s_st = np.abs(H) @ np.abs(x) + np.abs(g) + np.abs(CI.T) @ np.abs(lam_full) + np.abs(CE.T) @ np.abs(mu)
    on = lam_full != 0
    return {
        "equality": float(np.max(np.abs(eq) / (1e-2 + s_eq))) if len(eq) else 0.0,
        "feasibility": float(np.max(np.maximum(-sl, 0.0) / (1e-2 + s_in))) if len(sl) else 0.0,
        "dual": float(max(0.0, -lam_full.min()) / (1e-2 + np.abs(lam_full).max())) if len(sl) else 0.0,
        "complementarity": float(np.max(np.abs(sl[on]) / (1e-2 + s_in[on]))) if on.any() else 0.0,
        "stationarity": float(np.max(np.abs(st) / (1e-2 + s_st))),
    }


def random_batch(sizes, n_max, neq_max, nin_max, seed, pad=np.nan):
    """Random strictly convex QPs with a feasible point, padded with `pad`: sizes [(n, neq, nin)] per env."""
    rng = np.random.default_rng(seed)
    N = len(sizes)
    p = {"H": np.full((N, n_max, n_max), pad), "g": np.full((N, n_max), pad), "CE": np.full((N, neq_max, n_max), pad),
         "ce0": np.full((N, neq_max), pad), "CI": np.full((N, nin_max, n_max), pad), "ci0": np.full((N, nin_max), pad),
         "sizes": np.array(sizes, np.int32).reshape(N, 3)}
    for e, (n, neq, nin) in enumerate(sizes):
        A = rng.standard_normal((n, n))
        p["H"][e, :n, :n] = A @ A.T / n + 0.5 * np.eye(n)
        p["g"][e, :n] = 3.0 * rng.standard_normal(n)
        xf = 0.3 * rng.standard_normal(n)
        CE = rng.standard_normal((neq, n))
        p["CE"][e, :neq, :n] = CE
        p["ce0"][e, :neq] = -CE @ xf
        CI = rng.standard_normal((nin, n))
        p["CI"][e, :nin, :n] = CI
        p["ci0"][e, :nin] = -CI @ xf + rng.uniform(0.0, 1.0, nin) * (rng.uniform(size=nin) < 0.7)
    return p


# ------------------------------------------------------------------ CPU: the kernel body on the host emulator
def _emulated_export(kind, maskval, n=4, seed=51):
    s = setup(kind)
    q, v = synth.random_states(s["q0"], n, seed)
    step = (0.3, 0.2, 0.2, 0.5) if kind == "v1" else (0.1, 0.1275, 0.05, 0.7)
    _, refs = synth.walking_batch(s["refs"], n, seed, *step, float(s["refs"]["com"][2]))
    mask = np.full(n, maskval, np.uint8)
    return s, q, v, refs, EmuProblemTA(s["cm"], s["cc"]).problem_ta(q, v, mask, refs)


@pytest.mark.parametrize("kind,maskval", [("v1", 3), ("v1", 1), ("v1", 2), ("v1", 0), ("v0", 3), ("v0", 1), ("v0", 2), ("v0", 0)])
def test_emulated_qp_solve_matches_oracle_on_exported_problems(kind, maskval):
    """The emulated export of walking problems, solved by the emulated qp_env, against oracle_qp_solve on the same
    arrays; the export's TA x + ta0 at the oracle tick's own x is the oracle's tau."""
    s, q, v, refs, p = _emulated_export(kind, maskval)
    orc, max_iter = s["oracle"], s["cc"].max_iter
    sol = emu_qp_solve(p, max_iter)
    assert not compare_with_oracle(p, sol, max_iter)
    assert (sol["status"] == 0).all()
    for i in range(len(q)):
        n = int(p["sizes"][i][0])
        r = orc.tick(q[i], v[i], maskval, {k: a[i] for k, a in refs.items()}, orders=canonical_orders(orc, maskval))
        assert np.all(p["TA"][i][:, n:] == 0.0)
        assert np.max(np.abs(p["TA"][i][:, :n] @ r["x"] + p["ta0"][i] - r["tau"])) < 1e-10
        assert np.max(np.abs(sol["tau"][i] - r["tau"])) < 1e-8 * (1.0 + np.abs(r["tau"]).max())


def _special_cases():
    """(name, dense problem, expected status) for the solver's exits."""
    rng = np.random.default_rng(7)
    cases = []
    cases.append(("n=1", (np.array([[2.0]]), np.array([1.0]), np.zeros((0, 1)), np.zeros(0), np.array([[1.0]]), np.array([0.25])), 0))
    A = rng.standard_normal((5, 5))
    cases.append(("unconstrained", (A @ A.T + np.eye(5), rng.standard_normal(5), np.zeros((0, 5)), np.zeros(0),
                                     np.zeros((0, 5)), np.zeros(0)), 0))
    CI = np.zeros((3, 4))
    CI[0, 1], CI[1, 1], CI[2, 0] = 1.0, -1.0, 1.0  # x1 >= 1 and x1 <= 0
    cases.append(("infeasible pair", (np.eye(4), np.zeros(4), np.zeros((0, 4)), np.zeros(0), CI, np.array([-1.0, 0.0, 5.0])), 1))
    CE = rng.standard_normal((3, 6))
    CE[2] = CE[0]
    cases.append(("duplicated equality", (np.eye(6), np.ones(6), CE, np.array([0.1, 0.2, 0.1]), np.zeros((0, 6)), np.zeros(0)), 4))
    cases.append(("indefinite H", (np.diag([1.0, -1.0, 2.0]), np.ones(3), np.zeros((0, 3)), np.zeros(0),
                                    np.eye(3), np.ones(3)), 1))
    return cases


def _pack(dense, n_max, neq_max, nin_max, pad=np.nan):
    N = len(dense)
    p = {"H": np.full((N, n_max, n_max), pad), "g": np.full((N, n_max), pad), "CE": np.full((N, neq_max, n_max), pad),
         "ce0": np.full((N, neq_max), pad), "CI": np.full((N, nin_max, n_max), pad), "ci0": np.full((N, nin_max), pad),
         "sizes": np.zeros((N, 3), np.int32)}
    for e, (H, g, CE, ce0, CI, ci0) in enumerate(dense):
        n, neq, nin = len(g), len(ce0), len(ci0)
        p["H"][e, :n, :n], p["g"][e, :n], p["CE"][e, :neq, :n], p["ce0"][e, :neq] = H, g, CE, ce0
        p["CI"][e, :nin, :n], p["ci0"][e, :nin] = CI, ci0
        p["sizes"][e] = (n, neq, nin)
    return p


def test_emulated_qp_solve_matches_oracle_on_random_problems():
    """Random dense QPs within the oracle's caps (53 / 18 / 172) with NaN in all padding, and the solver's exits:
    n = 1, no constraints, an infeasible pair of rows (status 1), a duplicated equality row (4), an indefinite H (1)."""
    rng = np.random.default_rng(3)
    sizes = [(int(n), int(rng.integers(0, min(n, 18) + 1)), int(rng.integers(0, 173))) for n in rng.integers(1, 54, 10)]
    sizes += [(53, 18, 172), (53, 0, 172), (18, 18, 40), (12, 3, 0)]
    rp = random_batch(sizes, 53, 18, 172, 11)
    cases = _special_cases()
    dense = [_env(rp, i) for i in range(len(sizes))] + [c[1] for c in cases]
    p = _pack(dense, 53, 18, 172)
    sol = emu_qp_solve(p, 1000)
    assert not compare_with_oracle(p, sol, 1000)
    expect = [0] * len(sizes) + [c[2] for c in cases]
    assert list(sol["status"]) == expect, list(zip([c[0] for c in cases], sol["status"][len(sizes):]))
    for i in np.where(sol["status"] != 0)[0]:
        assert not sol["x"][i].any() and (sol["active"][i] == -1).all() and not sol["lambda"][i].any()
        assert not sol["lambda_eq"][i].any()
    assert sol["iters"][:len(sizes)].max() > 5  # the working sets grow and shrink


def test_emulated_qp_solve_max_iter():
    """max_iter = 2 stops the solve after one added row: status 3 with x, the working set and the multipliers written,
    as the oracle reports them."""
    p = random_batch([(20, 4, 60), (30, 0, 100)], 30, 4, 100, 12)
    sol = emu_qp_solve(p, 2)
    assert list(sol["status"]) == [3, 3]
    assert not compare_with_oracle(p, sol, 2)
    assert all(np.isfinite(sol["x"][i][: p["sizes"][i][0]]).all() and sol["x"][i].any() for i in range(2))
    assert (sol["active"][:, 0] >= 0).all()


def test_emulated_qp_solve_rejects_sizes_beyond_strides():
    """An env whose sizes exceed its strides (or are negative / n = 0 / neq > n) gets status 4 and zero outputs; the
    others are solved as in a batch without it."""
    p = random_batch([(10, 2, 20)] * 6, 12, 3, 24, 13)
    p["sizes"][1] = (13, 2, 20)
    p["sizes"][2] = (10, 4, 20)
    p["sizes"][3] = (10, 2, 25)
    p["sizes"][4] = (0, 0, 0)
    p["sizes"][5] = (2, 3, 0)
    sol = emu_qp_solve(p, 1000)
    assert list(sol["status"]) == [0, 4, 4, 4, 4, 4]
    assert list(sol["iters"][1:]) == [0] * 5
    assert not sol["x"][1:].any() and (sol["active"][1:] == -1).all() and not sol["lambda_eq"][1:].any()
    one = emu_qp_solve({k: a[:1] for k, a in p.items()}, 1000)
    for k in one:
        assert np.array_equal(one[k][0], sol[k][0]), k


def test_qp_kernel_compiles_without_spills():
    """-Xptxas -v: the generic QP kernel and the export kernels keep everything in registers."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    src = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tsid_control_b200", "csrc", "tsidb.cu")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-cubin", "-Xptxas", "-v",
                            "-o", os.path.join(d, "t.cubin"), src], capture_output=True, text=True, check=True)
    props = re.findall(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       r.stderr)
    found = {name: (int(a), int(b), int(c)) for name, a, b, c in props}
    for kernel in ("tsidb_qp_kernel", "tsidb_problem_kernel"):
        hits = {k: v for k, v in found.items() if kernel in k}
        assert hits, kernel
        assert all(v == (0, 0, 0) for v in hits.values()), hits


# ------------------------------------------------------------------ GPU
def _to_dev(e, p):
    import torch

    return {k: torch.as_tensor(np.ascontiguousarray(a), device=e.device) for k, a in p.items()}


def _solve(e, p):
    import torch

    out = e.qp_solve(_to_dev(e, p))
    torch.cuda.synchronize()
    return {k: t.cpu().numpy() for k, t in out.items()}


def _export_ta(e, q, v, mask, refs):
    import torch

    out = e.problem_data(*_dev(e, q, v, mask, refs), parts=QP_KEYS + ("TA", "ta0"))
    torch.cuda.synchronize()
    return {k: t.cpu().numpy() for k, t in out.items()}


def _objective(H, g, x):
    return 0.5 * x @ H @ x + g @ x


def row_labels(cc, na, nv, mask, nin):
    """Compact CI row of an exported env -> (block, side, i) in tsidb_ci_row's terms; rows a caller appended after the
    export's are ("extra", 0, r)."""
    blocks = [b for b in (0, 1) if (mask >> b) & 1] + ([2] if cc.use_torque_bounds else []) + ([3] if cc.use_joint_bounds else [])
    out = [(b, side, i) for b in blocks for side in (0, 1) for i in range((17, 17, na, nv)[b])]
    return out + [("extra", 0, r) for r in range(nin - len(out))]


def certify_tie(p, i, labels, sol, other_x, other_active, other_kkt, bar):
    """Env i solved two ways with different working sets (or iteration counts) is a degenerate tie: the working sets
    agree once the degenerate contact corners are canonicalised (common.canonical_active, the rule of the tick's parity
    tests), both answers satisfy the KKT conditions within `bar` and reach the same objective."""
    nn, neq, _ = (int(x) for x in p["sizes"][i])
    ca = canonical_active([labels[r] for r in sol["active"][i] if r >= 0])
    cb = canonical_active([labels[r] for r in other_active if r >= 0])
    assert ca == cb, (i, sorted(ca ^ cb, key=str))
    H, g, CE, ce0, CI, ci0 = _env(p, i)
    ra = kkt_direct(H, g, CE, ce0, CI, ci0, sol["x"][i][:nn], sol["active"][i], sol["lambda"][i], sol["lambda_eq"][i][:neq])
    assert max(ra.values()) < bar and max(other_kkt.values()) < bar, (i, ra, other_kkt)
    fa, fb = _objective(H, g, sol["x"][i][:nn]), _objective(H, g, other_x)
    assert abs(fa - fb) <= bar * (1.0 + abs(fb)), (i, fa, fb)


def psi_tolerance(H, nin):
    """The total row violation eiquadprog-fast accepts as feasible (its psi stopping test): nin eps tr(H) tr(L^-T) 100."""
    return nin * np.finfo(float).eps * np.trace(H) * np.sum(1.0 / np.diag(np.linalg.cholesky(H))) * 100.0


def oracle_kkt(p, i, o):
    return kkt_direct(*_env(p, i), o["x"], o["active"], o["lambda"], o["lambda_eq"])


@pytest.mark.gpu
@pytest.mark.parametrize("kind,overrides,bar", [
    ("v1", (), 1e-8),
    ("v0", (), 1e-7),
    ("v1", (("tau_max_scaling", 0.08), ("v_max_scaling", 0.1)), 1e-8),
])
def test_qp_solve_round_trip_against_tick_and_oracle(kind, overrides, bar, live):
    """The export of 2048-env walking batches solved on the device.  Against the tick on the same inputs: status and
    working set equal (the tick's rows mapped through tsidb_ci_row onto the compact rows), dv, the contact wrenches T f
    and tau = TA x + ta0 within the parity bars (the bars of the tick's own parity tests: the corner forces of a
    cond(H) ~ 1e8 force block are only determined through their wrench).  Against oracle_qp_solve on the same arrays:
    status, iterations, working set in order, x and multipliers.  Every env that differs is a degenerate tie
    (certify_tie).  The returned multipliers certify every solution by the full KKT conditions (no fitted mu)."""
    import torch

    from common import force_generator

    n = 2048
    s, q, v, mask, refs = _batch(kind, n, 71, overrides)
    e = _controller(kind, n, overrides).engine
    args = _dev(e, q, v, mask, refs)
    t = e.compute(*args, aux=True)
    torch.cuda.synchronize()
    tick = {k: getattr(t, k).cpu().numpy().copy() for k in ("tau", "ddq", "f", "status", "lam", "lam_row")}
    p = _export_ta(e, q, v, mask, refs)
    sol = _solve(e, p)
    nv, T = e.nv, force_generator(e.cc)
    worst = {"dv": 0.0, "wrench": 0.0, "tau": 0.0}
    kkt = {}
    ties_tick, ties_oracle = [], []
    assert np.array_equal(sol["status"], tick["status"])
    assert (sol["status"] == 0).mean() >= 0.95
    scale = lambda b: 1e-2 + np.abs(b).max(initial=0.0)  # noqa: E731
    for i in np.where(sol["status"] == 0)[0]:
        nn, neq, nin = (int(x) for x in p["sizes"][i])
        m = int(mask[i])
        labels = row_labels(e.cc, e.na, nv, m, nin)
        rows = {lab: r for r, lab in enumerate(labels)}
        used = tick["lam_row"][i] >= 0
        tick_rows = [rows[r] for r in bits_to_rows(e.na, nv, [int(b) for b in tick["lam_row"][i][used]])]
        x = sol["x"][i][:nn]
        feet = [k for k in (0, 1) if (m >> k) & 1]
        f = np.concatenate([tick["f"][i][12 * k:12 * k + 12] for k in feet] or [np.zeros(0)])
        w, wt = (np.concatenate([T @ y[12 * j:12 * j + 12] for j in range(len(feet))] or [np.zeros(0)]) for y in (x[nv:], f))
        for k, val in kkt_direct(*_env(p, i), x, sol["active"][i], sol["lambda"][i], sol["lambda_eq"][i][:neq]).items():
            kkt[k] = max(kkt.get(k, 0.0), val)
        diff = [k for k, ok in (("active", sorted(tick_rows) == sorted(int(a) for a in sol["active"][i] if a >= 0)),
                                ("dv", _close(x[:nv], tick["ddq"][i])), ("wrench", _close(w, wt)),
                                ("tau", _close(sol["tau"][i], tick["tau"][i]))) if not ok]
        if diff:
            ties_tick.append((i, diff))
            lam = np.zeros(nin)
            lam[tick_rows] = tick["lam"][i][used]
            xt = np.concatenate([tick["ddq"][i], f])
            certify_tie(p, i, labels, sol, xt, np.array(tick_rows), kkt_residuals(*_env(p, i), xt, lam), bar)
            continue
        worst["dv"] = max(worst["dv"], np.abs(x[:nv] - tick["ddq"][i]).max() / scale(tick["ddq"][i]))
        worst["wrench"] = max(worst["wrench"], np.abs(w - wt).max(initial=0.0) / scale(wt))
        worst["tau"] = max(worst["tau"], np.abs(sol["tau"][i] - tick["tau"][i]).max() / scale(tick["tau"][i]))
    for i, diff, o in compare_with_oracle(p, sol, e.cc.max_iter):
        ties_oracle.append((i, diff))
        assert o["status"] == sol["status"][i] == 0, (i, o["status"], sol["status"][i])
        labels = row_labels(e.cc, e.na, nv, int(mask[i]), int(p["sizes"][i][2]))
        certify_tie(p, i, labels, sol, o["x"], o["active"], oracle_kkt(p, i, o), bar)
    name = f"qp_solve_{kind}" + ("_tight_limits" if overrides else "")
    print(f"\n{name}, {n} envs: vs tick", {k: f"{x:.1e}" for k, x in worst.items()}, "KKT", {k: f"{x:.1e}" for k, x in kkt.items()},
          f"degenerate ties vs tick {len(ties_tick)}, vs oracle {len(ties_oracle)}; iterations max {sol['iters'].max()}")
    for what, ties in (("tick", ties_tick), ("oracle", ties_oracle)):
        if ties:
            print(f"  differences vs {what}:", {k: sum(k in d for _, d in ties) for k in sorted({k for _, d in ties for k in d})})
    parity_log.record(name, {**worst, **{f"kkt_{k}": x for k, x in kkt.items()}, "ties_tick": len(ties_tick),
                             "ties_oracle": len(ties_oracle)})
    assert all(x < bar for x in kkt.values()), kkt
    assert all(x < bar for x in worst.values()), worst


@pytest.mark.gpu
def test_qp_solve_modified_problem(live):
    """The v1 export with five joint-acceleration bounds |ddq_j| <= a appended as rows and a soft bound on one more
    joint through a slack variable s >= 0 (ddq_j0 <= a + s, cost 50 s^2): n <= 51, nin <= 172, odd stride.  Equal to
    oracle_qp_solve on the same arrays (status, iterations, working set, x and multipliers); the hard bounds hold."""
    n = 1024
    s, q, v, mask, refs = _batch("v1", n, 72)
    e = _controller("v1", n).engine
    p0 = _export_ta(e, q, v, mask, refs)
    nv, na = e.nv, e.na
    joints, j0, a = (6, 9, 12, 15, 18), 21, 4.0
    nm, ninm = p0["g"].shape[1] + 1, p0["ci0"].shape[1] + 2 * len(joints) + 2
    N = n
    p = {"H": np.zeros((N, nm, nm)), "g": np.zeros((N, nm)), "CE": np.zeros((N, 18, nm)), "ce0": p0["ce0"].copy(),
         "CI": np.zeros((N, ninm, nm)), "ci0": np.zeros((N, ninm)), "TA": np.zeros((N, na, nm)), "ta0": p0["ta0"].copy(),
         "sizes": p0["sizes"].copy()}
    for i in range(N):
        nn, neq, nin = (int(x) for x in p0["sizes"][i])
        p["H"][i, :nn, :nn] = p0["H"][i, :nn, :nn]
        p["H"][i, nn, nn] = 100.0
        p["g"][i, :nn] = p0["g"][i, :nn]
        p["CE"][i, :neq, :nn] = p0["CE"][i, :neq, :nn]
        p["CI"][i, :nin, :nn] = p0["CI"][i, :nin, :nn]
        p["ci0"][i, :nin] = p0["ci0"][i, :nin]
        r = nin
        for j in joints:
            p["CI"][i, r, j], p["ci0"][i, r] = 1.0, a
            p["CI"][i, r + 1, j], p["ci0"][i, r + 1] = -1.0, a
            r += 2
        p["CI"][i, r, j0], p["CI"][i, r, nn], p["ci0"][i, r] = -1.0, 1.0, a
        p["CI"][i, r + 1, nn] = 1.0
        p["TA"][i, :, :nn] = p0["TA"][i, :, :nn]
        p["sizes"][i] = (nn + 1, neq, r + 2)
    sol = _solve(e, p)
    assert (sol["status"] == 0).mean() >= 0.95
    bad = compare_with_oracle(p, sol, e.cc.max_iter)
    kkt = {}
    for i in np.where(sol["status"] == 0)[0]:
        nn, neq, _ = (int(x) for x in p["sizes"][i])
        for k, val in kkt_direct(*_env(p, i), sol["x"][i][:nn], sol["active"][i], sol["lambda"][i], sol["lambda_eq"][i][:neq]).items():
            kkt[k] = max(kkt.get(k, 0.0), val)
    print(f"\nmodified v1 export, {N} envs: KKT", {k: f"{x:.1e}" for k, x in kkt.items()}, f"differences vs oracle {len(bad)}",
          [(i, d) for i, d, _ in bad[:8]])
    for i, _, o in bad:
        # eiquadprog itself ends some of these envs with residuals up to ~1e-6 (the bound rows run parallel to the
        # joint-bound rows): each env is held to 1e-8 or twice the oracle's own residual on it, whichever is larger
        ro = oracle_kkt(p, i, o)
        certify_tie(p, i, row_labels(e.cc, na, nv, int(mask[i]), int(p["sizes"][i][2])), sol, o["x"], o["active"], ro,
                    max(1e-8, 2 * max(ro.values())))
    ok = sol["status"] == 0
    ddq = sol["x"][ok][:, :nv]
    slack = np.array([sol["x"][i][int(p["sizes"][i][0]) - 1] for i in np.where(ok)[0]])
    # the new rows hold as every row of an eiquadprog solution does: to within the violation its psi test accepts
    tol = np.array([psi_tolerance(_env(p, i)[0], int(p["sizes"][i][2])) for i in np.where(ok)[0]])
    assert (np.abs(ddq[:, list(joints)]).max(axis=1) <= a + tol).all()
    assert (slack >= -tol).all()
    binding = (np.abs(np.abs(ddq[:, list(joints)]) - a) < 1e-9).any(axis=1).sum()
    taus = np.einsum("nrk,nk->nr", p["TA"][ok], sol["x"][ok]) + p["ta0"][ok]
    assert np.abs(taus - sol["tau"][ok]).max() < 1e-9 * (1 + np.abs(taus).max())
    print(f"bound binding in {binding} envs, slack > 0 in {(slack > 1e-9).sum()}")
    assert binding > 0


@pytest.mark.gpu
def test_qp_solve_random_problems_at_the_caps(live):
    """A random batch at the caps (n = 64, neq = 20, nin = 512, NaN padding elsewhere) has no oracle: every env is
    certified by the KKT conditions with the returned multipliers, and 16 envs by the scipy solve of test_problem_data."""
    N = 256
    rng = np.random.default_rng(21)
    sizes = [(64, 20, 512)] * (N // 2) + [(int(n), int(rng.integers(0, 21)), int(rng.integers(0, 513)))
                                          for n in rng.integers(20, 65, N // 2)]
    p = random_batch(sizes, 64, 20, 512, 22)
    e = _controller("v1", 64).engine
    sol = _solve(e, p)
    assert (sol["status"] == 0).all(), np.unique(sol["status"], return_counts=True)
    kkt, sc = {}, 0.0
    for i in range(N):
        nn, neq, _ = sizes[i]
        res = kkt_direct(*_env(p, i), sol["x"][i][:nn], sol["active"][i], sol["lambda"][i], sol["lambda_eq"][i][:neq])
        for k, val in res.items():
            kkt[k] = max(kkt.get(k, 0.0), val)
        if i < 16:
            y, _ = scipy_qp(*_env(p, i))
            sc = max(sc, np.abs(y - sol["x"][i][:nn]).max() / (1e-2 + np.abs(y).max()))
    print(f"\nrandom QPs at the caps, {N} envs: KKT", {k: f"{x:.1e}" for k, x in kkt.items()}, f"scipy {sc:.1e}, "
          f"iterations max {sol['iters'].max()}, working set max {(sol['active'] >= 0).sum(axis=1).max()}")
    assert all(x < 1e-8 for x in kkt.values()), kkt
    assert sc < 1e-6


@pytest.mark.gpu
def test_qp_solve_per_env_errors_and_bad_arguments(live):
    """An env with sizes above its strides gets status 4 and zero outputs while its neighbours' results are bit-identical
    to a batch without it; the host refuses strides above the caps, misaligned and null arrays and tau without TA."""
    import ctypes as C

    import torch

    from tsid_control_b200 import _capi

    e = _controller("v1", 64).engine
    p = random_batch([(30, 6, 80)] * 5, 32, 8, 96, 31)
    ref = _solve(e, {k: np.delete(a, 2, axis=0) for k, a in p.items()})
    p["sizes"][2] = (33, 6, 80)
    sol = _solve(e, p)
    assert sol["status"][2] == 4 and sol["iters"][2] == 0
    assert not sol["x"][2].any() and (sol["active"][2] == -1).all() and not sol["lambda"][2].any() and not sol["lambda_eq"][2].any()
    for k in ref:
        assert np.array_equal(np.delete(sol[k], 2, axis=0), ref[k]), k

    lib = e.lib
    d = _to_dev(e, p)
    f64 = dict(dtype=torch.float64, device=e.device)
    o = {"x": torch.empty((5, 32), **f64), "status": torch.empty(5, dtype=torch.int32, device=e.device)}
    tau = torch.empty((5, e.na), **f64)

    def call(n_envs=5, n_max=32, neq_max=8, nin_max=96, drop=(), shift=None, out_drop=(), with_tau=False):
        po = _capi.TsidbProblemOut(**{k: (t.data_ptr() + ((2 if k == "sizes" else 4) if k == shift else 0)) for k, t in d.items() if k not in drop})
        qo = _capi.TsidbQpOut(**{k: t.data_ptr() for k, t in o.items() if k not in out_drop})
        if with_tau:
            qo.tau = tau.data_ptr()
        rc = lib.tsidb_qp_solve(e.h, n_envs, n_max, neq_max, nin_max, C.byref(po), C.byref(qo), e._stream())
        return rc, lib.tsidb_last_error()

    for kw, msg in ((dict(n_max=65), b"TSIDB_QP_MAX_N"), (dict(nin_max=513), b"TSIDB_QP_MAX_NIN"),
                    (dict(neq_max=33), b"neq_max <= n_max"), (dict(n_envs=0), b"n_envs"),
                    (dict(shift="H"), b"aligned"), (dict(shift="sizes"), b"aligned"), (dict(drop=("H",)), b"required"),
                    (dict(drop=("CI",)), b"CI and ci0"), (dict(out_drop=("x",)), b"required"), (dict(with_tau=True), b"tau needs TA")):
        rc, err = call(**kw)
        assert rc < 0 and msg in err, (kw, rc, err)
    torch.cuda.synchronize()
    with pytest.raises(TypeError):
        e.qp_solve({**d, "H": d["H"].float()})
    with pytest.raises(ValueError):
        e.qp_solve({k: t for k, t in d.items() if k != "ci0"})


@pytest.mark.gpu
def test_qp_solve_is_independent_of_the_tick(live):
    """Two solves of the same input are bit-identical; a solve between two ticks (scheduling hint on) changes no output
    bit of the second tick; a solve on a side stream while a tick of the same handle runs on the main stream gives the
    results it gives alone; problem_data with the default parts returns what it returns with TA and ta0 requested."""
    import torch

    n = 8192
    s, q, v, mask, refs = _batch("v1", n, 73)
    keys = ("tau", "ddq", "f", "status", "iters", "active_set")
    runs, probs = [], []
    for with_solve in (False, True):
        e = _controller("v1", n).engine
        e.set_sched_hint(True)
        args = _dev(e, q, v, mask, refs)
        prob = e.problem_data(*args, parts=QP_KEYS + ("TA", "ta0"))
        outs = []
        for _ in range(2):
            if with_solve:
                e.qp_solve(prob)
            t = e.compute(*args)
            torch.cuda.synchronize()
            outs.append({k: getattr(t, k).cpu().numpy().copy() for k in keys})
        runs.append(outs)
    for a, b in zip(*runs):
        for k in keys:
            assert np.array_equal(a[k], b[k]), k

    alone = {k: t.cpu().numpy() for k, t in e.qp_solve(prob).items()}
    again = {k: t.cpu().numpy() for k, t in e.qp_solve(prob).items()}
    for k in alone:
        assert np.array_equal(alone[k], again[k]), k
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=e.device)
    side.wait_stream(torch.cuda.current_stream(e.device))
    t = e.compute(*args)
    with torch.cuda.stream(side):
        conc = e.qp_solve(prob)
    torch.cuda.synchronize()
    for k in alone:
        assert np.array_equal(alone[k], conc[k].cpu().numpy()), k
    for k in keys:
        assert np.array_equal(getattr(t, k).cpu().numpy(), runs[0][1][k]), k

    dflt = e.problem_data(*args)
    assert set(dflt) == set(QP_KEYS) | {"sizes"}
    for k in dflt:
        assert torch.equal(dflt[k], prob[k]), k
