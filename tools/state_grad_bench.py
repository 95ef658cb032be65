"""Time of the gradient with respect to the state (TsidEngine.state_grad / tsidb_state_grad, TsidEngine.tick_layer) on
the walking65536 workload.

    python tools/state_grad_bench.py [--n 65536] [--iters 10] [--warmup 2]

On the inputs of bench.py's walking65536 (same seed) it times, with CUDA events over --iters calls after --warmup:
tsidb_state_grad alone with random dL/d of all eight parts of the export, writing dL/dq and dL/dv; qp_grad of the
tick_layer's forward solve for all eight parts; tick_layer's backward pass from random dL/dtau, dL/ddv and dL/df with
every reference tensor requiring grad, once without and once with q and v requiring grad; and the tick on the same
inputs for scale.  The card's name, power limit and clock are read in the same run.  Needs a CUDA device; there is no
CPU path.
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
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("state_grad_bench: no CUDA device")
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
    parts = e.PROBLEM_PARTS + e.ACTUATION_PARTS
    prob = e.problem_data(qd, vd, md, rd, parts=parts)
    grads = {k: rnd(*prob[k].shape) for k in parts}
    ms, lo, hi = timed(lambda: e.state_grad(qd, vd, md, rd, grads), args.warmup, args.iters)
    print(f"tsidb_state_grad (all eight parts -> dq, dv): {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, "
          f"max {hi:.3f}); {ms * 1e3 / n:.3f} us per env, {e.nq + e.nv} tangent passes of K1 per env")

    sol = e.qp_solve(prob)
    gin = {"x": rnd(*sol["x"].shape), "tau": rnd(n, e.na)}
    ms, lo, hi = timed(lambda: e.qp_grad(prob, sol, gin, parts), args.warmup, args.iters)
    print(f"qp_grad (all eight parts): {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f})")

    for with_state in (False, True):
        leaves = {k: t.clone().requires_grad_(True) for k, t in rd.items()}
        qs, vs = (qd.clone().requires_grad_(True), vd.clone().requires_grad_(True)) if with_state else (qd, vd)
        out = e.tick_layer(qs, vs, md, leaves)
        w = {k: rnd(*out[k].shape) for k in ("tau", "dv", "f")}
        loss = sum((out[k] * w[k]).sum() for k in w)
        inputs = list(leaves.values()) + ([qs, vs] if with_state else [])

        def backward(loss=loss, inputs=inputs):
            torch.autograd.grad(loss, inputs, retain_graph=True)

        ms, lo, hi = timed(backward, args.warmup, args.iters)
        what = "every reference, q and v" if with_state else "every reference, q and v without grad"
        print(f"tick_layer backward ({what}): {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f})")
        del out, loss, leaves
    ms, lo, hi = timed(lambda: e.compute(qd, vd, md, rd), args.warmup, args.iters)
    print(f"tick on the same inputs: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f})")
    print(f"GPU after the runs: {gpu_info()}")
    e.close()


if __name__ == "__main__":
    main()
