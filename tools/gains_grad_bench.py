"""Time of the gradient with respect to the task gains and weights (TsidEngine.gains_grad / tsidb_gains_grad,
TsidEngine.set_gains, TsidEngine.tick_layer with gains) on the walking65536 workload.

    python tools/gains_grad_bench.py [--n 65536] [--iters 20] [--warmup 3] [--log profiles/gains_grad/gains_grad_bench.log]

On the inputs of bench.py's walking65536 (same seed) it times, with CUDA events over --iters calls after --warmup:
tsidb_gains_grad alone with random dL/dH, dL/dg and dL/dce0; tick_layer's backward pass from random dL/dtau, dL/ddv and
dL/df with every gains tensor and every reference tensor requiring grad (qp_grad for H, g and ce0, refs_grad, gains_grad
and the sum over envs), against the same backward with the references alone (qp_grad for g and ce0, refs_grad);
set_gains on the host clock (it synchronises the device); and the tick on the same inputs for scale.  gains_grad's bytes
(q, v, mask, references, the H blocks, g columns and ce0 rows it reads, the gradients it writes) are counted from the
shapes.  The card's name, power limit and clock are read in the same run; the output also goes to --log.  Needs a CUDA
device; there is no CPU path.
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

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


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
    import time

    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log", default=os.path.join(ROOT, "profiles", "gains_grad", "gains_grad_bench.log"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gains_grad_bench: no CUDA device")
    from tsid_control_b200 import synth
    from tsid_control_b200.ctrl.conf import RobotConfig
    from tsid_control_b200.ctrl.WalkController import WalkController

    lines = []

    def say(msg: str) -> None:
        print(msg, flush=True)
        lines.append(msg)

    n = args.n
    conf = RobotConfig()
    conf.max_envs = n
    ctrl = WalkController(conf, n_envs=n)
    e = ctrl.engine
    q, v = synth.random_states(ctrl.q, n, 0)  # the seed of bench.py's walking65536 (rank 0)
    mask, refs = synth.walking_batch(ctrl.default_refs, n, 0, 0.3, 0.2, 0.2, 0.5, float(ctrl.default_refs["com"][2]))
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=e.device)  # noqa: E731
    qd, vd, md, rd = dev(q), dev(v), dev(mask), {k: dev(a) for k, a in refs.items()}
    say(f"GPU: {gpu_info()}")
    say(f"workload: walking, robot/v1, {n} envs, masks {dict(zip(*np.unique(mask, return_counts=True)))}")

    nx, neq, _ = e.problem_sizes()
    gen = torch.Generator(device=e.device).manual_seed(0)
    rnd = lambda *s: torch.randn(s, generator=gen, dtype=torch.float64, device=e.device)  # noqa: E731
    grads = {"H": rnd(n, nx, nx), "g": rnd(n, nx), "ce0": rnd(n, neq)}
    nc = (mask & 1).astype(np.int64) + ((mask >> 1) & 1)
    nref = 9 + 24 + 24 + 12 + 12 + e.na
    reads = 8 * (n * (e.nq + e.nv + nref + e.nv + e.nv * e.nv) + int((6 * nc).sum()) + int((144 * nc).sum())) + n
    writes = 8 * n * 84
    ms, lo, hi = timed(lambda: e.gains_grad(qd, vd, md, rd, grads), args.warmup, args.iters)
    say(f"tsidb_gains_grad (all 84 columns): {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f}); "
        f"read {reads / 1e6:.1f} MB, written {writes / 1e6:.1f} MB (from shapes); "
        f"{(reads + writes) / (ms * 1e-3) / 1e9:.0f} GB/s = {100 * (reads + writes) / (ms * 1e-3) / HBM_BYTES_PER_S:.1f} % "
        f"of 7.7 TB/s")
    del grads
    ms, lo, hi = timed(lambda: e.refs_grad(qd, vd, md, rd, rnd(n, nx), rnd(n, neq)), args.warmup, args.iters)
    say(f"tsidb_refs_grad for comparison (with two randn fills): {ms:.3f} ms per call (median of {args.iters})")

    g0 = e.gains()
    for with_gains in (False, True):
        leaves = {k: t.clone().requires_grad_(True) for k, t in rd.items()}
        gl = {k: t.clone().requires_grad_(True) for k, t in g0.items()} if with_gains else None
        out = e.tick_layer(qd, vd, md, leaves, gl)
        w = {k: rnd(*out[k].shape) for k in ("tau", "dv", "f")}
        loss = sum((out[k] * w[k]).sum() for k in w)
        wrt = list(leaves.values()) + (list(gl.values()) if gl else [])

        def backward():
            torch.autograd.grad(loss, wrt, retain_graph=True)

        ms, lo, hi = timed(backward, args.warmup, args.iters)
        what = "gains and references (qp_grad H, g, ce0 + refs_grad + gains_grad)" if with_gains else \
            "references alone (qp_grad g, ce0 + refs_grad)"
        say(f"tick_layer backward, {what}: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f})")
        del out, loss

    times = []
    for i in range(args.warmup + args.iters):
        t0 = time.perf_counter()
        e.set_gains(g0)
        if i >= args.warmup:
            times.append(1e3 * (time.perf_counter() - t0))
    say(f"set_gains (host clock, synchronises the device): {np.median(times):.3f} ms per call (median of {args.iters}, "
        f"min {min(times):.3f}, max {max(times):.3f})")
    ms, lo, hi = timed(lambda: e.compute(qd, vd, md, rd), args.warmup, args.iters)
    say(f"tick on the same inputs: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f})")
    say(f"GPU after the runs: {gpu_info()}")
    e.close()
    if args.log:
        os.makedirs(os.path.dirname(os.path.abspath(args.log)), exist_ok=True)
        with open(args.log, "w") as fh:
            fh.write("# python tools/gains_grad_bench.py " + " ".join(sys.argv[1:]) + "\n" + "\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
