"""Time of the generic QP solve (TsidEngine.qp_solve / tsidb_qp_solve) on the exported walking65536 problems.

    python tools/qp_solve_bench.py [--n 65536] [--iters 20] [--warmup 3]

On the workload of bench.py's walking65536 (same seed) it times, with CUDA events over --iters calls after --warmup:
the export with the actuation map (problem_data with H, g, CE, ce0, CI, ci0, TA, ta0), tsidb_qp_solve on that export
(x, multipliers, working set and tau), and the tick on the same inputs for context.  For each call it reports ms per
call and the bytes the call moves, computed from the shapes, each env's (n, neq, nin) and the solve's measured
iteration counts (the violation scan reads the env's CI rows and ci0 once per pass), and the achieved GB/s against the
B200's 7.7 TB/s.  The card's name and power limit are read in the same run.  Needs a CUDA device; there is no CPU path.
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


def solve_bytes(sizes: np.ndarray, iters: np.ndarray, status: np.ndarray, n_max: int, neq_max: int, na: int) -> int:
    """Bytes tsidb_qp_solve reads and writes: sizes 12 B; the lower triangle of H, g, CE and ce0 once; per pass of the
    active-set loop (one per iteration) the env's CI rows and ci0, plus one CI row per pick; TA rows and ta0 for tau; the
    outputs at their strides."""
    n, neq, nin = (sizes[:, k].astype(np.int64) for k in range(3))
    it = iters.astype(np.int64)
    written = (status == 0) | (status == 3)
    reads = 12 + 8 * (n * (n + 1) // 2 + n + neq * n + neq)
    reads += 8 * it * (nin * n + nin + n)
    reads += np.where(written, 8 * (na * n + na), 0)
    writes = 8 * (2 * n_max + neq_max + na) + 4 * (n_max + 2)
    return int(reads.sum() + writes * len(n))


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
    ms, lo, hi = timed(lambda: e.problem_data(qd, vd, md, rd, parts=PARTS), args.warmup, args.iters)
    stored = n * 8 * (nx * nx + nx + neq * nx + neq + nin * nx + nin + na * nx + na) + n * 12
    print(f"export with TA, ta0: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f}); stored "
          f"{stored / 1e9:.3f} GB; {stored / (ms * 1e-3) / 1e9:.0f} GB/s = {100 * stored / (ms * 1e-3) / HBM_BYTES_PER_S:.1f} % "
          f"of 7.7 TB/s")

    out = e.qp_solve(prob)
    ms, lo, hi = timed(lambda: e.qp_solve(prob), args.warmup, args.iters)
    sizes, iters, status = prob["sizes"].cpu().numpy(), out["iters"].cpu().numpy(), out["status"].cpu().numpy()
    moved = solve_bytes(sizes, iters, status, nx, neq, na)
    print(f"tsidb_qp_solve: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f}); status "
          f"{dict(zip(*np.unique(status, return_counts=True)))}, iterations mean {iters.mean():.2f} max {iters.max()}; "
          f"moved {moved / 1e9:.3f} GB (model from shapes and iterations); {moved / (ms * 1e-3) / 1e9:.0f} GB/s = "
          f"{100 * moved / (ms * 1e-3) / HBM_BYTES_PER_S:.1f} % of 7.7 TB/s")

    ms, lo, hi = timed(lambda: e.compute(qd, vd, md, rd), args.warmup, args.iters)
    print(f"tick on the same inputs: {ms:.3f} ms per call (median of {args.iters}, min {lo:.3f}, max {hi:.3f}) = "
          f"{n / (ms * 1e-3) / 1e6:.2f} M ticks/s (L2 not flushed between calls)")
    e.close()


if __name__ == "__main__":
    main()
