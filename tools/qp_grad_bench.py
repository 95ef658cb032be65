"""Time of the adjoint of the generic QP solve (TsidEngine.qp_grad / tsidb_qp_grad) on the exported walking65536 problems.

    python tools/qp_grad_bench.py [--n 65536] [--iters 20] [--warmup 3]

On the workload of bench.py's walking65536 (same seed) it exports every env's QP with the actuation map, solves it once
with tsidb_qp_solve and times, with CUDA events over --iters calls after --warmup: tsidb_qp_grad with incoming gradients
for x, lambda, lambda_eq and tau writing every part (H, g, CE, ce0, CI, ci0, TA, ta0), the same writing g, ce0 and ci0
only, and tsidb_qp_solve on the same inputs for scale.  For each gradient call it reports ms per call, the bytes it
reads and writes (a model computed from the shapes and each env's (n, neq, nin) and working-set size) and the achieved
GB/s against the B200's 7.7 TB/s.  The card's name, power limit and clock are read in the same run.  Needs a CUDA
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
PARTS = ("H", "g", "CE", "ce0", "CI", "ci0", "TA", "ta0")


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


def grad_bytes(sizes: np.ndarray, active: np.ndarray, n_max: int, neq_max: int, nin_max: int, na: int, parts) -> tuple:
    """(read, written) bytes of tsidb_qp_grad with all four incoming gradients on OPTIMAL envs: sizes, status and the
    env's n working-set entries; the lower triangle of H, the CE rows and the working set's CI rows; x, the multipliers
    and their incoming gradients; TA and tau's gradient.  Written: the requested parts at their strides and status."""
    n, neq = (sizes[:, k].astype(np.int64) for k in range(2))
    w = (active >= 0).sum(axis=1).astype(np.int64)
    reads = 12 + 4 + 4 * n + 8 * (n * (n + 1) // 2 + (neq + w) * n + 2 * (n + neq + w) + na + na * n)
    stride = {"H": n_max * n_max, "g": n_max, "CE": neq_max * n_max, "ce0": neq_max, "CI": nin_max * n_max, "ci0": nin_max,
              "TA": na * n_max, "ta0": na}
    writes = 4 + 8 * sum(stride[k] for k in parts)
    return int(reads.sum()), int(writes * len(n))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("qp_solve_bench: no CUDA device")
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

    nx, neq, nin = e.problem_sizes()
    na = e.na
    prob = e.problem_data(qd, vd, md, rd, parts=PARTS)
    sol = e.qp_solve(prob)
    torch.cuda.synchronize()
    status = sol["status"].cpu().numpy()
    active = sol["active"].cpu().numpy()
    sizes = prob["sizes"].cpu().numpy()
    print(f"solve status {dict(zip(*np.unique(status, return_counts=True)))}, working set mean {(active >= 0).sum(1).mean():.2f} "
          f"max {(active >= 0).sum(1).max()}, n_max {nx}, neq_max {neq}, nin_max {nin}")
    gen = torch.Generator(device=e.device).manual_seed(0)
    grads = {k: torch.randn(sol[k].shape, generator=gen, dtype=torch.float64, device=e.device)
             for k in ("x", "lambda", "lambda_eq", "tau")}
    for parts in (PARTS, ("g", "ce0", "ci0")):
        out = e.qp_grad(prob, sol, grads, parts)
        ms, lo, hi = timed(lambda: e.qp_grad(prob, sol, grads, parts), args.warmup, args.iters)
        st = out["status"].cpu().numpy()
        rd_b, wr_b = grad_bytes(sizes, active, nx, neq, nin, na, parts)
        tot = rd_b + wr_b
        print(f"tsidb_qp_grad ({', '.join(parts)}): {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f}); "
              f"differentiated {(st == 0).sum()} of {n}; read {rd_b / 1e9:.3f} GB, written {wr_b / 1e9:.3f} GB (model from "
              f"shapes and working sets); {tot / (ms * 1e-3) / 1e9:.0f} GB/s = {100 * tot / (ms * 1e-3) / HBM_BYTES_PER_S:.1f} % "
              f"of 7.7 TB/s")
        del out

    ms, lo, hi = timed(lambda: e.qp_solve(prob), args.warmup, args.iters)
    print(f"tsidb_qp_solve on the same inputs: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f})")
    print(f"GPU after the runs: {gpu_info()}")
    e.close()


if __name__ == "__main__":
    main()
