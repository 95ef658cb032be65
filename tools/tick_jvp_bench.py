"""Time of the forward derivative of the tick (TsidEngine.tick_jvp / tick_jacobian, tsidb_tick_jvp) on the walking65536
workload.

    python tools/tick_jvp_bench.py [--n 65536] [--iters 5] [--warmup 1]

On the inputs of bench.py's walking65536 (same seed) it times, with CUDA events over --iters calls after --warmup and
tick_layer's forward (problem_data + qp_solve) held fixed: tick_jvp with one per-env direction in (q, v); tick_jacobian's
JVP in (q, v) (nq + nv shared identity columns); the JVP in every input (q, v and all references); and, for comparison,
one tick_layer backward with q, v and every reference requiring grad, which is the cost of one reverse-mode row of the
Jacobian.  The bytes the JVP writes follow from the shapes.  The card's name, power limit and clock are read in the same
run.  Needs a CUDA device; there is no CPU path.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

def gpu_info() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:  # noqa: BLE001
        return f"nvidia-smi unavailable ({exc}); torch: {torch.cuda.get_device_name(0)}"


def timed(fn, warmup: int, iters: int):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(iters):
        start.record()
        fn()
        stop.record()
        stop.synchronize()
        times.append(start.elapsed_time(stop))
    return float(np.median(times)), min(times), max(times)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tick_jvp_bench: no CUDA device")
    from tsid_control_b200 import synth
    from tsid_control_b200.ctrl.conf import RobotConfig
    from tsid_control_b200.ctrl.WalkController import WalkController

    n = args.n
    conf = RobotConfig()
    conf.max_envs = n
    ctrl = WalkController(conf, n_envs=n)
    e = ctrl.engine
    q, v = synth.random_states(ctrl.q, n, 0)  # the seed of bench.py's walking65536 (rank 0)
    mask, refs = synth.walking_batch(ctrl.default_refs, n, 0, 0.3, 0.2, 0.2, 0.5, float(ctrl.default_refs["com"][2]))
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=e.device)  # noqa: E731
    qd, vd, md, rd = dev(q), dev(v), dev(mask), {k: dev(a) for k, a in refs.items()}
    print(f"GPU: {gpu_info()}")
    print(f"workload: walking, robot/v1, {n} envs, masks {dict(zip(*np.unique(mask, return_counts=True)))}")
    gen = torch.Generator(device=e.device).manual_seed(0)
    rnd = lambda *s: torch.randn(s, generator=gen, dtype=torch.float64, device=e.device)  # noqa: E731
    prob = e.problem_data(qd, vd, md, rd, parts=e.PROBLEM_PARTS + e.ACTUATION_PARTS)
    sol = e.qp_solve(prob)
    nx = prob["g"].shape[1]
    dims = dict(e._ref_dims, q=e.nq, v=e.nv)

    def eye(keys):
        K = sum(dims[k] for k in keys)
        m, out, c = torch.eye(K, dtype=torch.float64, device=e.device), {}, 0
        for k in keys:
            out[k] = m[:, c:c + dims[k]].contiguous()
            c += dims[k]
        return out, K

    def report(what, tangents, per_env_dirs):
        o = e.tick_jvp(qd, vd, md, rd, tangents, prob, sol)
        ok = int((o["status"] == 0).sum())
        ms, lo, hi = timed(lambda: e.tick_jvp(qd, vd, md, rd, tangents, prob, sol), args.warmup, args.iters)
        written = n * per_env_dirs * (nx + e.na) * 8 + 4 * n
        print(f"{what}: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f}); {per_env_dirs} directions, "
              f"{written / 1e9:.3f} GB written (x' {nx}, tau' {e.na} doubles per env and direction); {ok} of {n} envs "
              f"differentiated")
        return ms

    report("tick_jvp, one per-env direction in (q, v)", {"q": rnd(n, 1, e.nq), "v": rnd(n, 1, e.nv)}, 1)
    t, K = eye(("q", "v"))
    ms_qv = report("tick_jacobian's JVP in (q, v)", t, K)
    t, K = eye(("q", "v") + tuple(k for k, _ in e._ref_dims))
    report("tick_jacobian's JVP in q, v and every reference", t, K)
    t, K = eye(tuple(k for k, _ in e._ref_dims))
    report("tick_jacobian's JVP in the references alone (no tangent K1 pass)", t, K)

    leaves = {k: t.clone().requires_grad_(True) for k, t in rd.items()}
    qs, vs = qd.clone().requires_grad_(True), vd.clone().requires_grad_(True)
    out = e.tick_layer(qs, vs, md, leaves)
    w = {k: rnd(*out[k].shape) for k in ("tau", "dv", "f")}
    loss = sum((out[k] * w[k]).sum() for k in w)
    inputs = list(leaves.values()) + [qs, vs]
    ms, lo, hi = timed(lambda: torch.autograd.grad(loss, inputs, retain_graph=True), args.warmup, args.iters)
    rows = e.na + e.nv + 24
    print(f"tick_layer backward (q, v and every reference; one reverse-mode row): {ms:.3f} ms per call (median of "
          f"{args.iters}, min {lo:.3f}, max {hi:.3f}); {rows} such rows for a Jacobian: {rows * ms:.0f} ms; the (q, v) "
          f"Jacobian by forward mode costs {ms_qv / ms:.2f} rows")
    print(f"GPU after the runs: {gpu_info()}")
    e.close()


if __name__ == "__main__":
    main()
