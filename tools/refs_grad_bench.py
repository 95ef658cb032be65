"""Time of the gradient through the task references (TsidEngine.refs_grad / tsidb_refs_grad, TsidEngine.tick_layer) on
the walking65536 workload.

    python tools/refs_grad_bench.py [--n 65536] [--iters 20] [--warmup 3]

On the inputs of bench.py's walking65536 (same seed) it times, with CUDA events over --iters calls after --warmup:
tsidb_refs_grad alone with random dL/dg and dL/dce0 writing all six reference gradients; tick_layer's forward pass
(problem_data with the actuation map, then qp_solve); its backward pass (qp_grad for g and ce0, then refs_grad) from
random dL/dtau, dL/ddv and dL/df with every reference tensor requiring grad; and the tick on the same inputs for scale.
refs_grad's bytes (q, v, mask, references, the dg columns and dce0 rows it reads, the gradients it writes) are counted
from the shapes.  The card's name, power limit and clock are read in the same run.  Needs a CUDA device; there is no CPU
path.
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
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("refs_grad_bench: no CUDA device")
    from tsid_control_b200 import synth
    from tsid_control_b200.ctrl.conf import RobotConfig
    from tsid_control_b200.ctrl.WalkController import WalkController
    from tsid_control_b200.engine import REF_KEYS

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

    nx, neq, _ = e.problem_sizes()
    gen = torch.Generator(device=e.device).manual_seed(0)
    rnd = lambda *s: torch.randn(s, generator=gen, dtype=torch.float64, device=e.device)  # noqa: E731
    dg, dce0 = rnd(n, nx), rnd(n, neq)
    nc = (mask & 1).astype(np.int64) + ((mask >> 1) & 1)
    dims = dict(zip(REF_KEYS, (9, 24, 24, 12, 12, e.na)))
    reads = 8 * (n * (e.nq + e.nv + sum(dims.values()) + e.nv) + int((6 * nc).sum())) + n
    writes = 8 * n * sum(dims.values())
    ms, lo, hi = timed(lambda: e.refs_grad(qd, vd, md, rd, dg, dce0), args.warmup, args.iters)
    print(f"tsidb_refs_grad (all six references): {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f}); "
          f"read {reads / 1e6:.1f} MB, written {writes / 1e6:.1f} MB (from shapes); "
          f"{(reads + writes) / (ms * 1e-3) / 1e9:.0f} GB/s = {100 * (reads + writes) / (ms * 1e-3) / HBM_BYTES_PER_S:.1f} % "
          f"of 7.7 TB/s")

    leaves = {k: t.clone().requires_grad_(True) for k, t in rd.items()}
    ms, lo, hi = timed(lambda: e.tick_layer(qd, vd, md, leaves), args.warmup, args.iters)
    print(f"tick_layer forward (problem_data with TA, ta0 + qp_solve): {ms:.3f} ms per call (median of {args.iters}, "
          f"min {lo:.3f}, max {hi:.3f})")
    out = e.tick_layer(qd, vd, md, leaves)
    w = {k: rnd(*out[k].shape) for k in ("tau", "dv", "f")}
    loss = sum((out[k] * w[k]).sum() for k in w)

    def backward():
        torch.autograd.grad(loss, list(leaves.values()), retain_graph=True)

    ms, lo, hi = timed(backward, args.warmup, args.iters)
    st = out["status"].cpu().numpy()
    print(f"tick_layer backward (qp_grad g, ce0 + refs_grad, every reference): {ms:.3f} ms per call (median of {args.iters}, "
          f"min {lo:.3f}, max {hi:.3f}); solve status 0 on {(st == 0).sum()} of {n}")
    ms, lo, hi = timed(lambda: e.compute(qd, vd, md, rd), args.warmup, args.iters)
    print(f"tick on the same inputs: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f})")
    print(f"GPU after the runs: {gpu_info()}")
    e.close()


if __name__ == "__main__":
    main()
