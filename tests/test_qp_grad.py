"""Differentiating the batched QP solve (tsidb_qp_grad / TsidEngine.qp_grad / TsidEngine.qp_layer).

Every check compares with qp_grad_ref, a numpy restatement of the adjoint that solves the transposed KKT system of the
final working set densely (it shares no code with the kernel's Cholesky + Householder path).  qp_grad_ref itself is
checked against central differences of the oracle's eiquadprog.  On CPU the kernel header's qp_grad_env runs on the host
warp emulator; on the GPU the batched call, torch.autograd.gradcheck of qp_layer, finite differences through the GPU
solve and an optimisation through qp_layer are checked."""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import parity_log
from emu_qp import emu_qp_solve
from emu_qp_grad import emu_qp_grad
from oracle_qp import oracle_qp_solve
from test_problem_data import _batch, _controller, _dev, live  # noqa: F401
from test_qp_solve import _emulated_export, _env, _export_ta, _solve, _to_dev, random_batch

RTOL, ATOL = 1e-8, 1e-10  # the parity bars
PARTS = ("H", "g", "CE", "ce0", "CI", "ci0", "TA", "ta0")
GRADS = ("x", "lambda", "lambda_eq", "tau")


def qp_grad_ref(H, CE, CI, x, active, lam, lam_eq, xb=None, lb=None, leb=None, TA=None, taub=None):
    """The adjoint of one solved QP from dense, unpadded arrays: with G = [CE; CI_W], nu = [lam_eq; lam_W] and the
    incoming gradients xb (+ TA' taub) and nub = [leb; lb_W], solve [[H, G'], [G, 0]] [p; q] = [xb; -nub] (H from its lower
    triangle, as the solve reads it) and return dL/d of H, g, CE, ce0, CI, ci0, TA, ta0 (zeros where not reached)."""
    n, neq, nin = len(x), len(lam_eq), CI.shape[0]
    W = [int(a) for a in active if a >= 0]
    w, m = len(W), neq + len(W)
    G = np.vstack([CE, CI[W]]) if m else np.zeros((0, n))
    nu = np.concatenate([lam_eq, lam[:w]])
    xb = np.zeros(n) if xb is None else np.array(xb[:n], dtype=float)
    nub = np.concatenate([np.zeros(neq) if leb is None else leb[:neq], np.zeros(w) if lb is None else lb[:w]])
    if taub is not None:
        xb = xb + TA.T @ taub
    Hl = np.tril(H) + np.tril(H, -1).T
    K = np.block([[Hl, G.T], [G, np.zeros((m, m))]])
    rhs = np.concatenate([xb, -nub])
    s = np.linalg.solve(K, rhs)
    # cond(K) reaches 1e9 on the exported problems (the force block of H): iterative refinement with residuals in
    # extended precision makes the reference accurate to the data rather than to LU's backward error
    Kl, rl = K.astype(np.longdouble), rhs.astype(np.longdouble)
    for _ in range(3):
        s = s + np.linalg.solve(K, (rl - Kl @ s.astype(np.longdouble)).astype(float))
    p, q = s[:n], s[n:]
    P = -np.outer(p, x)
    out = {"H": np.tril(P + P.T, -1) + np.diag(np.diag(P)), "g": -p,
           "CE": np.outer(nu[:neq], p) - np.outer(q[:neq], x), "ce0": -q[:neq],
           "CI": np.zeros((nin, n)), "ci0": np.zeros(nin)}
    out["CI"][W] = np.outer(nu[neq:], p) - np.outer(q[neq:], x)
    out["ci0"][W] = -q[neq:]
    if TA is not None:
        out["TA"] = np.zeros_like(TA) if taub is None else np.outer(taub, x)
        out["ta0"] = np.zeros(TA.shape[0]) if taub is None else np.array(taub, dtype=float)
    return out


def ref_batch(p, sol, grads):
    """qp_grad_ref of every env of a padded batch, embedded in zero padding -> (dict of padded parts, expected status)."""
    N = len(p["sizes"])
    out = {k: np.zeros(p[k].shape) for k in PARTS if k in p}
    status = np.full(N, 4, np.int32)
    for i in range(N):
        if sol["status"][i] != 0:
            continue
        n, neq, nin = (int(v) for v in p["sizes"][i])
        gi = {k: (grads[k][i] if k in grads else None) for k in GRADS}
        r = qp_grad_ref(p["H"][i][:n, :n], p["CE"][i][:neq, :n], p["CI"][i][:nin, :n], sol["x"][i][:n], sol["active"][i][:n],
                        sol["lambda"][i], sol["lambda_eq"][i][:neq], gi["x"], gi["lambda"], gi["lambda_eq"],
                        p["TA"][i][:, :n] if "TA" in p else None, gi["tau"])
        for k, lead in (("H", (n, n)), ("g", (n,)), ("CE", (neq, n)), ("ce0", (neq,)), ("CI", (nin, n)), ("ci0", (nin,)),
                        ("TA", (-1, n)), ("ta0", (-1,))):
            if k in out:
                out[k][i][tuple(slice(0, d) if d >= 0 else slice(None) for d in lead)] = r[k]
        status[i] = 0
    return out, status


def compare(out, ref, status, parts=None, rtol=RTOL):
    """Status equal; every part of every env within the parity bars of the reference and exactly zero where the reference
    is (padding, rows outside the working set, envs not differentiated).  Returns the worst relative error per part."""
    assert np.array_equal(out["status"], status), (np.where(out["status"] != status)[0][:10], out["status"][:10])
    worst = {}
    for k in (parts or ref):
        a, b = out[k], ref[k]
        for i in range(len(a)):
            err = np.max(np.abs(a[i] - b[i]), initial=0.0)
            scale = np.max(np.abs(b[i]), initial=0.0)
            assert err <= ATOL + rtol * scale, (k, i, err, scale)
            assert np.all(a[i][b[i] == 0.0] == 0.0), (k, i)
            worst[k] = max(worst.get(k, 0.0), err / (1e-300 + scale))
    return worst


def random_grads(p, seed, pad=np.nan):
    """Random incoming gradients x, lambda, lambda_eq (and tau when the problem has TA) with `pad` beyond each env's
    sizes and working set (nothing there may be read)."""
    rng = np.random.default_rng(seed)
    N, nm = p["g"].shape
    neqm = p["ce0"].shape[1]
    g = {"x": rng.standard_normal((N, nm)), "lambda": rng.standard_normal((N, nm)), "lambda_eq": rng.standard_normal((N, neqm))}
    for i in range(N):
        n, neq, _ = (int(v) for v in p["sizes"][i])
        g["x"][i][n:] = pad
        g["lambda_eq"][i][neq:] = pad
    if "TA" in p:
        g["tau"] = rng.standard_normal((N, p["TA"].shape[1]))
    return g


def poison_solution(p, sol):
    """The solution with NaN beyond each env's x, working set and equality multipliers (nothing there may be read)."""
    s = {k: np.array(a, copy=True) for k, a in sol.items()}
    for i in range(len(s["status"])):
        n, neq, _ = (int(v) for v in p["sizes"][i])
        s["x"][i][n:] = np.nan
        s["lambda"][i][int((s["active"][i] >= 0).sum()):] = np.nan
        s["lambda_eq"][i][neq:] = np.nan
    return s


def augment(p0, nv):
    """The export with five joint-acceleration bounds |ddq_j| <= 4 appended as rows and a soft bound on one more joint
    through a slack variable s >= 0 (ddq_j0 <= 4 + s, cost 50 s^2): one more variable, odd stride."""
    joints, j0, a = (6, 9, 12, 15, 18), 21, 4.0
    N = len(p0["sizes"])
    nm, ninm = p0["g"].shape[1] + 1, p0["ci0"].shape[1] + 2 * len(joints) + 2
    na = p0["TA"].shape[1]
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
    return p


# ------------------------------------------------------------------ CPU: the kernel body on the host emulator
@pytest.mark.parametrize("kind,maskval", [("v1", 3), ("v1", 1), ("v1", 2), ("v1", 0), ("v0", 3), ("v0", 1), ("v0", 2), ("v0", 0)])
def test_emulated_qp_grad_matches_reference_on_exported_problems(kind, maskval):
    """Emulated exports of walking problems (every contact mask), solved by the emulated qp_env, differentiated by the
    emulated qp_grad_env with random incoming gradients for x, lambda, lambda_eq and tau."""
    s, q, v, refs, p = _emulated_export(kind, maskval)
    sol = emu_qp_solve(p, s["cc"].max_iter)
    assert (sol["status"] == 0).all()
    grads = random_grads(p, 5 + maskval)
    out = emu_qp_grad(p, poison_solution(p, sol), grads)
    worst = compare(out, *ref_batch(p, sol, grads))
    print(f"\nemulated qp_grad vs reference ({kind}, mask {maskval}):", {k: f"{x:.1e}" for k, x in worst.items()})


def test_emulated_qp_grad_matches_reference_on_random_problems():
    """Random dense QPs with NaN in all padding (problem, solution and incoming gradients), a part requested alone, and
    gradients of only x: the rest counts as zero."""
    rng = np.random.default_rng(8)
    sizes = [(int(n), int(rng.integers(0, min(n, 18) + 1)), int(rng.integers(0, 120))) for n in rng.integers(1, 54, 10)]
    sizes += [(53, 18, 172), (53, 0, 172), (18, 18, 40), (12, 3, 0), (64, 20, 300)]
    p = random_batch(sizes, 64, 20, 300, 9)
    sol = emu_qp_solve(p, 1000)
    assert (sol["status"] == 0).all()
    assert (sol["active"] >= 0).sum(axis=1).max() > 5
    grads = random_grads(p, 10)
    out = emu_qp_grad(p, poison_solution(p, sol), grads)
    worst = compare(out, *ref_batch(p, sol, grads))
    print("\nemulated qp_grad vs reference, random problems:", {k: f"{x:.1e}" for k, x in worst.items()})
    only = {"x": grads["x"]}
    out = emu_qp_grad(p, sol, only, parts=("ci0",))
    assert set(out) == {"ci0", "status"}
    compare(out, *ref_batch(p, sol, only), parts=("ci0",))


def test_emulated_qp_grad_matches_reference_on_a_modified_export():
    """The v1 export with bound rows and a slack variable appended (odd stride n_max = 51)."""
    s, q, v, refs, p0 = _emulated_export("v1", 3)
    p = augment(p0, 26)
    sol = emu_qp_solve(p, s["cc"].max_iter)
    assert (sol["status"] == 0).all()
    grads = random_grads(p, 12)
    out = emu_qp_grad(p, poison_solution(p, sol), grads)
    worst = compare(out, *ref_batch(p, sol, grads))
    print("\nemulated qp_grad vs reference, modified export:", {k: f"{x:.1e}" for k, x in worst.items()})


def error_batch():
    """Eight solved random envs and the same batch with envs 1-7 made undifferentiable: a non-OPTIMAL solve status, sizes
    above the strides, an out-of-range working-set entry, a duplicated entry, neq + |W| > n, -1 padding before an entry
    and two identical working-set rows."""
    p = random_batch([(12, 2, 30)] * 8, 14, 3, 32, 41)
    sol = emu_qp_solve(p, 1000)
    assert (sol["status"] == 0).all() and ((sol["active"] >= 0).sum(axis=1) >= 2).all()
    bp, bs = {k: a.copy() for k, a in p.items()}, {k: a.copy() for k, a in sol.items()}
    bs["status"][1] = 1
    bp["sizes"][2] = (15, 2, 30)
    bs["active"][3][0] = 30
    bs["active"][4][1] = bs["active"][4][0]
    bs["active"][5][:11] = np.arange(11)
    bs["active"][6][1], bs["active"][6][2] = -1, 5
    r0, r1 = bs["active"][7][:2]
    bp["CI"][7][r1] = bp["CI"][7][r0]
    return p, sol, bp, bs


def test_emulated_qp_grad_errors_give_zero_gradients():
    """Each undifferentiable env gets status 4 and zero gradients; env 0 gets what it gets alone."""
    p, sol, bp, bs = error_batch()
    grads = random_grads(p, 42, pad=0.0)
    out = emu_qp_grad(bp, bs, grads)
    assert list(out["status"]) == [0] + [4] * 7
    for k in PARTS[:6]:
        assert not out[k][1:].any(), k
    alone = emu_qp_grad({k: a[:1] for k, a in p.items()}, {k: a[:1] for k, a in sol.items()}, {k: a[:1] for k, a in grads.items()})
    for k in alone:
        assert np.array_equal(alone[k][0], out[k][0]), k


def _margin_problems(count, seed):
    """Random QPs whose oracle solution has a strict-complementarity margin: active multipliers and inactive slacks at
    least 1e-4 of their scale, a non-empty working set."""
    rng = np.random.default_rng(seed)
    found = []
    while len(found) < count:
        n = int(rng.integers(4, 12))
        sz = (n, int(rng.integers(0, 4)), int(rng.integers(4, 16)))
        p = random_batch([sz], n, max(sz[1], 1), sz[2], int(rng.integers(1 << 30)))
        d = _env(p, 0)
        o = oracle_qp_solve(*d, 1000)
        W = [int(a) for a in o["active"] if a >= 0]
        if o["status"] != 0 or not W:
            continue
        slack = d[4] @ o["x"] + d[5]
        inactive = np.delete(slack, W)
        lam = o["lambda"][:len(W)]
        if lam.min() < 1e-4 * (1 + np.abs(lam).max()) or (len(inactive) and inactive.min() < 1e-4 * (1 + np.abs(slack).max())):
            continue
        TA = rng.standard_normal((3, n))
        found.append((d, TA, rng.standard_normal(3), o))
    return found


def test_reference_matches_finite_differences_of_the_oracle():
    """qp_grad_ref against central differences of oracle_qp_solve along random directions in every part, on problems
    with a strict-complementarity margin whose working set is unchanged at +-eps: 1e-6 relative."""
    rng = np.random.default_rng(17)
    worst = 0.0
    for d, TA, ta0, o in _margin_problems(6, 18):
        H, g, CE, ce0, CI, ci0 = d
        n, neq, nin = len(g), len(ce0), len(ci0)
        W = sorted(int(a) for a in o["active"] if a >= 0)
        xb, lb, leb, taub = rng.standard_normal(n), rng.standard_normal(n), rng.standard_normal(neq), rng.standard_normal(3)

        def loss(args):
            r = oracle_qp_solve(*args[:6], 1000)
            act = [int(a) for a in r["active"] if a >= 0]
            assert r["status"] == 0 and sorted(act) == W
            lam_rows = np.zeros(nin)
            lam_rows[act] = r["lambda"][:len(act)]
            lb_rows = np.zeros(nin)
            lb_rows[[int(a) for a in o["active"] if a >= 0]] = lb[:len(W)]
            return xb @ r["x"] + leb @ r["lambda_eq"] + lb_rows @ lam_rows + taub @ (args[6] @ r["x"] + args[7])

        ref = qp_grad_ref(H, CE, CI, o["x"], o["active"], o["lambda"], o["lambda_eq"], xb, lb, leb, TA, taub)
        args = [H, g, CE, ce0, CI, ci0, TA, ta0]
        for k, name in enumerate(PARTS):
            if args[k].size == 0:
                continue
            dirn = rng.standard_normal(args[k].shape)
            eps = 1e-5
            plus, minus = list(args), list(args)
            plus[k], minus[k] = args[k] + eps * dirn, args[k] - eps * dirn
            fd = (loss(plus) - loss(minus)) / (2 * eps)
            an = float(np.sum(ref[name] * dirn))
            scale = float(np.sum(np.abs(ref[name] * dirn)))
            err = abs(fd - an) / max(abs(an), scale)
            worst = max(worst, err)
            assert err < 1e-6, (name, fd, an, scale)
    print(f"\nqp_grad_ref vs central differences of the oracle: worst {worst:.1e}")


def test_qp_grad_kernel_compiles_without_spills():
    """-Xptxas -v: the QP gradient kernel keeps everything in registers."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    src = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tsid_control_b200", "csrc", "tsidb.cu")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-cubin", "-Xptxas", "-v",
                            "-o", os.path.join(d, "t.cubin"), src], capture_output=True, text=True, check=True)
    m = re.search(r"Function properties for \S*tsidb_qp_grad_kernel\S*\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads", r.stderr)
    assert m and m.groups() == ("0", "0", "0"), m and m.groups()


# ------------------------------------------------------------------ GPU
def _grad(e, p, sol, grads, parts=None):
    import torch

    out = e.qp_grad(_to_dev(e, p), _to_dev(e, sol), _to_dev(e, grads), parts)
    torch.cuda.synchronize()
    return {k: t.cpu().numpy() for k, t in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,overrides,rtol", [
    ("v1", (), 1e-8),
    ("v0", (), 1e-8),
    ("v1", (("tau_max_scaling", 0.08), ("v_max_scaling", 0.1)), 1e-7),
])
def test_qp_grad_matches_reference_on_walking_batches(kind, overrides, rtol, live):
    """2048-env walking batches: export with TA, qp_solve, qp_grad with random incoming gradients for x, lambda,
    lambda_eq and tau; every part of every env against qp_grad_ref (exact to the data) within the parity bars.  With the
    tight limits the working sets stack torque and joint-velocity rows on the contact rows, cond(KKT) reaches 1e9, and
    the equality-row gradients (-q) of a few envs carry the 1e-8 relative error a backward-stable fp64 solve of such a
    system has: 1e-7 there, the bar test_qp_solve holds the solve's own outputs to for v0."""
    n = 2048
    s, q, v, mask, refs = _batch(kind, n, 81, overrides)
    e = _controller(kind, n, overrides).engine
    p = _export_ta(e, q, v, mask, refs)
    sol = _solve(e, p)
    assert (sol["status"] == 0).mean() >= 0.95
    grads = random_grads(p, 82, pad=0.0)
    out = _grad(e, p, sol, grads)
    ref, status = ref_batch(p, sol, grads)
    worst = compare(out, ref, status, rtol=rtol)
    name = f"qp_grad_{kind}" + ("_tight_limits" if overrides else "")
    print(f"\n{name}, {n} envs: vs qp_grad_ref", {k: f"{x:.1e}" for k, x in worst.items()},
          f"differentiated {(out['status'] == 0).sum()}, working set max {(sol['active'] >= 0).sum(axis=1).max()}")
    parity_log.record(name, worst)


def _pack_margin(e, count, seed):
    """_margin_problems packed into one zero-padded batch, with a random TA [na, n] and ta0 per env."""
    rng = np.random.default_rng(seed)
    probs = _margin_problems(count, seed)
    nm = max(len(d[1]) for d, *_ in probs)
    neqm = max(max(len(d[3]) for d, *_ in probs), 1)
    ninm = max(len(d[5]) for d, *_ in probs)
    N, na = len(probs), e.na
    p = {"H": np.zeros((N, nm, nm)), "g": np.zeros((N, nm)), "CE": np.zeros((N, neqm, nm)), "ce0": np.zeros((N, neqm)),
         "CI": np.zeros((N, ninm, nm)), "ci0": np.zeros((N, ninm)), "TA": np.zeros((N, na, nm)), "ta0": np.zeros((N, na)),
         "sizes": np.zeros((N, 3), np.int32)}
    for i, (d, *_) in enumerate(probs):
        H, g, CE, ce0, CI, ci0 = d
        nn, neq, nin = len(g), len(ce0), len(ci0)
        p["H"][i, :nn, :nn], p["g"][i, :nn], p["CE"][i, :neq, :nn], p["ce0"][i, :neq] = H, g, CE, ce0
        p["CI"][i, :nin, :nn], p["ci0"][i, :nin] = CI, ci0
        p["TA"][i, :, :nn] = rng.standard_normal((na, nn))
        p["ta0"][i] = rng.standard_normal(na)
        p["sizes"][i] = (nn, neq, nin)
    return p


def _layer_fn(e, p, keys):
    """keys' tensors -> (x, lambda, lambda_eq, tau) of qp_layer, the other parts fixed."""
    def fn(*ts):
        prob = dict(p)
        prob.update(zip(keys, ts))
        out = e.qp_layer(prob)
        return out["x"], out["lambda"], out["lambda_eq"], out["tau"]
    return fn


@pytest.mark.gpu
def test_qp_layer_gradcheck_on_random_problems(live):
    """torch.autograd.gradcheck of qp_layer with respect to H, g, CE, ce0, CI, ci0, TA and ta0 on a small random batch
    whose solutions have a strict-complementarity margin."""
    import torch

    e = _controller("v1", 64).engine
    p = _to_dev(e, _pack_margin(e, 4, 91))
    keys = PARTS
    inputs = tuple(p[k].clone().requires_grad_(True) for k in keys)
    assert torch.autograd.gradcheck(_layer_fn(e, p, keys), inputs, eps=1e-6, atol=1e-6, rtol=1e-5)


def _margin_envs(p, sol, count, margin):
    """Up to `count` envs of a solved batch, those with a working set first, whose solution has a strict-complementarity
    margin: multipliers of the working set above `margin` times max(1, their largest), slacks of the other rows above
    `margin` times their scale.  (Most walking envs have none: their contact pyramids put rows with zero multiplier in
    the working set and rows with zero slack outside it.)"""
    picked = []
    for i in np.where(sol["status"] == 0)[0]:
        H, g, CE, ce0, CI, ci0 = _env(p, i)
        w = int((sol["active"][i] >= 0).sum())
        lam = sol["lambda"][i][:w]
        slack = np.delete(CI @ sol["x"][i][:len(g)] + ci0, sol["active"][i][:w])
        if lam.min(initial=1.0) > margin * max(1.0, np.abs(lam).max(initial=0.0)) and \
                slack.min(initial=1.0) > margin * (1 + np.abs(ci0[np.abs(ci0) < 1e9]).max(initial=0.0)):
            picked.append((w == 0, int(p["sizes"][i][0]), int(i)))
    return [i for *_, i in sorted(picked)][:count]


@pytest.mark.gpu
def test_qp_layer_gradcheck_on_exported_walking_envs(live):
    """gradcheck of qp_layer with respect to g and ci0 on three exported walking envs whose solutions have a
    complementarity margin (_margin_envs; the tight-limit conf gives envs whose working sets hold limit rows)."""
    import torch

    n = 1024
    tight = (("tau_max_scaling", 0.08), ("v_max_scaling", 0.1))
    s, q, v, mask, refs = _batch("v1", n, 92, tight)
    e = _controller("v1", n, tight).engine
    p = _export_ta(e, q, v, mask, refs)
    sol = _solve(e, p)
    envs = _margin_envs(p, sol, 3, 1e-3)
    assert len(envs) == 3, envs
    sub = _to_dev(e, {k: a[envs] for k, a in p.items()})
    keys = ("g", "ci0")
    fn = _layer_fn(e, sub, keys)
    inputs = tuple(sub[k].clone().requires_grad_(True) for k in keys)
    jac = torch.autograd.functional.jacobian(lambda *t: torch.cat([o.reshape(-1) for o in fn(*t)]), inputs)
    scale = max(float(j.abs().max()) for j in jac)
    print(f"\nwalking envs {envs} (n = {[int(p['sizes'][i][0]) for i in envs]}, working set "
          f"{[int((sol['active'][i] >= 0).sum()) for i in envs]}): max |d out / d (g, ci0)| {scale:.2e}")
    assert torch.autograd.gradcheck(fn, inputs, eps=1e-6, atol=1e-6 * scale, rtol=1e-4)


@pytest.mark.gpu
def test_qp_grad_directional_differences_through_the_gpu_solve(live):
    """Central differences of L = xb.x + taub.tau through the GPU qp_solve on a walking batch, along random directions
    in g (scaled to its entries) and in ci0 (on the rows of each env's working set, the only rows x depends on), against
    qp_grad's directional derivative, on the envs whose working set is the same at theta +- eps d; such envs must be the
    large majority (degenerate contact corners, rows of zero slack, change their working set in the others).  The error
    is taken relative to the larger of |derivative| and the sum of its absolute terms.  The KKT systems of the contact
    envs have cond ~ 4e8, so the solve's own rounding (up to ~1e-8 in x) against a perturbation of 1e-7 sets the
    accuracy of a difference quotient: the bars are on the median (1e-6) and the 90th percentile (1e-4), with every env
    within 0.1; the multiplier gradients are checked against qp_grad_ref and by gradcheck instead."""
    n = 2048
    s, q, v, mask, refs = _batch("v1", n, 93)
    e = _controller("v1", n).engine
    p = _export_ta(e, q, v, mask, refs)
    sol = _solve(e, p)
    rng = np.random.default_rng(94)
    grads = {"x": rng.standard_normal(sol["x"].shape), "tau": rng.standard_normal(sol["tau"].shape)}
    out = _grad(e, p, sol, grads)
    W = lambda so, i: sorted(int(a) for a in so["active"][i] if a >= 0)  # noqa: E731
    loss = lambda so: np.einsum("ij,ij->i", grads["x"], so["x"]) + np.einsum("ij,ij->i", grads["tau"], so["tau"])  # noqa: E731
    for k in ("g", "ci0"):
        scale = 1e-3 + np.where(np.abs(p[k]) < 1e9, np.abs(p[k]), 0.0)
        d = rng.standard_normal(p[k].shape) * (scale if k == "g" else 1.0 + scale)
        if k == "ci0":
            rows = np.zeros_like(d)
            for i in range(n):
                rows[i, W(sol, i)] = 1.0
            d *= rows
        eps = 1e-7
        sp, sm = (_solve(e, {**p, k: p[k] + sgn * eps * d}) for sgn in (1.0, -1.0))
        same = [i for i in range(n) if sol["status"][i] == 0 and sp["status"][i] == 0 and sm["status"][i] == 0
                and W(sp, i) == W(sol, i) == W(sm, i)]
        fd = (loss(sp) - loss(sm)) / (2 * eps)
        an = np.sum((out[k] * d).reshape(n, -1), axis=1)
        sc = np.sum(np.abs(out[k] * d).reshape(n, -1), axis=1)
        err = np.abs(fd - an)[same] / np.maximum(np.maximum(np.abs(an), sc), 1e-300)[same]
        q50, q90 = np.median(err), np.quantile(err, 0.9)
        print(f"\n{k}: working set unchanged in {len(same)} of {n} envs; directional derivative vs central differences: "
              f"median {q50:.1e}, 90 % {q90:.1e}, 99 % {np.quantile(err, 0.99):.1e}, max {err.max():.1e}")
        assert len(same) >= 0.75 * n
        assert q50 < 1e-6 and q90 < 1e-4 and err.max() < 0.1, (k, q50, q90, err.max())


@pytest.mark.gpu
def test_qp_layer_fits_a_slack_cost_with_torch_optim(live):
    """A learnable weight w = exp(theta) on the cost of an appended slack variable (the soft bound ddq_j0 <= a + s of the
    modified export) is fitted with Adam so that tau reaches the tau of a target weight: within 60 steps the loss falls
    below 5 % of its start."""
    import torch

    n = 64
    s, q, v, mask, refs = _batch("v1", n, 96)
    e = _controller("v1", n).engine
    p0 = _export_ta(e, q, v, mask, refs)
    p = augment(p0, e.nv)
    sol = _solve(e, p)
    keep = np.where((sol["status"] == 0) & (sol["x"][np.arange(n), p["sizes"][:, 0] - 1] > 1e-6))[0][:16]
    assert len(keep) >= 4
    base = _to_dev(e, {k: a[keep] for k, a in p.items()})
    slack = torch.as_tensor(p["sizes"][keep, 0] - 1, device=e.device, dtype=torch.long)
    rows = torch.arange(len(keep), device=e.device)

    def tau_of(theta):
        H = base["H"].clone()
        H = H.index_put((rows, slack, slack), torch.exp(theta).expand(len(keep)))
        return e.qp_layer({**base, "H": H})["tau"]

    with torch.no_grad():
        target = tau_of(torch.tensor(np.log(20.0), dtype=torch.float64, device=e.device))
    theta = torch.tensor(np.log(100.0), dtype=torch.float64, device=e.device, requires_grad=True)
    opt = torch.optim.Adam([theta], lr=0.05)
    losses = []
    for _ in range(60):
        opt.zero_grad()
        loss = ((tau_of(theta) - target) ** 2).sum()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    print(f"\nslack weight fit: loss {losses[0]:.3e} -> {losses[-1]:.3e}, w = {float(torch.exp(theta.detach())):.2f} (target 20)")
    assert losses[-1] < 0.05 * losses[0]


@pytest.mark.gpu
def test_qp_grad_plumbing(live):
    """Per-env errors (as on the emulator), argument refusals, a NULL part is not written, bit-identical repeats, a
    qp_grad on a side stream beside a tick gives what it gives alone, and later ticks do not change."""
    import ctypes as C

    import torch

    from tsid_control_b200 import _capi

    e = _controller("v1", 64).engine
    p, sol, bp, bs = error_batch()
    grads = random_grads(p, 42, pad=0.0)
    out = _grad(e, bp, bs, grads)
    assert list(out["status"]) == [0] + [4] * 7
    assert all(not out[k][1:].any() for k in PARTS[:6])
    compare({k: a[:1] for k, a in out.items()}, *ref_batch({k: a[:1] for k, a in p.items()}, {k: a[:1] for k, a in sol.items()},
                                                              {k: a[:1] for k, a in grads.items()}), parts=PARTS[:6])

    d, ds, dg = _to_dev(e, p), _to_dev(e, sol), _to_dev(e, grads)
    f64 = dict(dtype=torch.float64, device=e.device)
    sentinel = {k: torch.full_like(d[k], 7.0) for k in PARTS[:6]}
    st = torch.empty(8, dtype=torch.int32, device=e.device)
    tau = torch.zeros((8, e.na), **f64)

    def call(n_envs=8, n_max=14, neq_max=3, nin_max=32, drop=(), sol_drop=(), gin_extra=None, gout_extra=None, shift=None,
             outs=("g",), status=True):
        po = _capi.TsidbProblemOut(**{k: t.data_ptr() + (4 if k == shift else 0) for k, t in d.items() if k not in drop})
        so = _capi.TsidbQpOut(**{k: t.data_ptr() for k, t in ds.items() if k not in sol_drop and k != "iters"})
        gi = _capi.TsidbQpOut(**{k: t.data_ptr() for k, t in dg.items()}, **(gin_extra or {}))
        go = _capi.TsidbProblemOut(**{k: sentinel[k].data_ptr() for k in outs}, **(gout_extra or {}))
        rc = e.lib.tsidb_qp_grad(e.h, n_envs, n_max, neq_max, nin_max, C.byref(po), C.byref(so), C.byref(gi), C.byref(go),
                                 st.data_ptr() if status else None, e._stream())
        return rc, e.lib.tsidb_last_error()

    for kw, msg in ((dict(n_max=65), b"TSIDB_QP_MAX_N"), (dict(nin_max=513), b"TSIDB_QP_MAX_NIN"),
                    (dict(neq_max=15), b"neq_max <= n_max"), (dict(n_envs=0), b"n_envs"), (dict(shift="H"), b"aligned"),
                    (dict(drop=("H",)), b"required"), (dict(sol_drop=("active",)), b"required"), (dict(status=False), b"required"),
                    (dict(drop=("CI",)), b"CI and ci0"), (dict(sol_drop=("lambda_eq",)), b"lambda_eq"),
                    (dict(gin_extra={"tau": tau.data_ptr()}), b"needs TA"), (dict(gin_extra={"active": st.data_ptr()}), b"NULL"),
                    (dict(gout_extra={"sizes": st.data_ptr()}), b"NULL")):
        rc, err = call(**kw)
        assert rc < 0 and msg in err, (kw, rc, err)
    rc, err = call(outs=("g",))
    torch.cuda.synchronize()
    assert rc == 0, err
    assert np.array_equal(sentinel["g"].cpu().numpy(), _grad(e, p, sol, grads)["g"])
    for k in ("H", "CE", "ce0", "CI", "ci0"):
        assert bool((sentinel[k] == 7.0).all()), k
    with pytest.raises(TypeError):
        e.qp_grad(d, ds, {**dg, "x": dg["x"].float()})
    with pytest.raises(ValueError):
        e.qp_grad(d, ds, dg, parts=("TA",))
    with pytest.raises(ValueError):
        e.qp_grad(d, {k: t for k, t in ds.items() if k != "active"}, dg)

    n = 8192
    s, q, v, mask, refs = _batch("v1", n, 97)
    keys = ("tau", "ddq", "f", "status", "iters", "active_set")
    runs = []
    for with_grad in (False, True):
        e = _controller("v1", n).engine
        e.set_sched_hint(True)
        args = _dev(e, q, v, mask, refs)
        prob = e.problem_data(*args, parts=PARTS)
        so = e.qp_solve(prob)
        gr = {"x": torch.ones_like(so["x"]), "tau": torch.ones_like(so["tau"])}
        outs = []
        for _ in range(2):
            if with_grad:
                e.qp_grad(prob, so, gr)
            t = e.compute(*args)
            torch.cuda.synchronize()
            outs.append({k: getattr(t, k).cpu().numpy().copy() for k in keys})
        runs.append(outs)
    for a, b in zip(*runs):
        for k in keys:
            assert np.array_equal(a[k], b[k]), k
    alone = {k: t.cpu().numpy() for k, t in e.qp_grad(prob, so, gr).items()}
    again = {k: t.cpu().numpy() for k, t in e.qp_grad(prob, so, gr).items()}
    for k in alone:
        assert np.array_equal(alone[k], again[k]), k
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=e.device)
    side.wait_stream(torch.cuda.current_stream(e.device))
    t = e.compute(*args)
    with torch.cuda.stream(side):
        conc = e.qp_grad(prob, so, gr)
    torch.cuda.synchronize()
    for k in alone:
        assert np.array_equal(alone[k], conc[k].cpu().numpy()), k
    for k in keys:
        assert np.array_equal(getattr(t, k).cpu().numpy(), runs[0][1][k]), k
