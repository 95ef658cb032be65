"""Time of the QP export (TsidEngine.problem_data / tsidb_problem_data) on the walking65536 workload.

    python tools/problem_data_bench.py [--n 65536] [--iters 30] [--warmup 5]

Per part set (all six parts; H, g, CE, ce0 only) it reports ms per call (CUDA events over --iters calls after --warmup),
the bytes the call stores (the padded arrays, and the part of them inside each env's (n, neq, nin) from `sizes`), the
achieved store rate and its share of the B200's 7.7 TB/s HBM bandwidth.  A call is the dynamics kernel followed by the
export kernel; the dynamics kernel's time in a regular tick (set_timing / last_tick_ms) is reported next to it.  The
card's name and power limit are read in the same run.  Needs a CUDA device; there is no CPU path.
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


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("problem_data_bench: no CUDA device")
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
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=e.device)
    qd, vd, md, rd = dev(q), dev(v), dev(mask), {k: dev(a) for k, a in refs.items()}
    print(f"GPU: {gpu_info()}")
    print(f"workload: walking, robot/v1, {n} envs, masks {dict(zip(*np.unique(mask, return_counts=True)))}")

    # the dynamics kernel of a regular tick (stage timing: the tick runs stage by stage on one stream)
    e.set_timing(True)
    dyn = []
    for i in range(args.warmup + args.iters):
        e.compute(qd, vd, md, rd)
        ms = e.last_tick_ms()
        if i >= args.warmup:
            dyn.append(ms["dynamics"])
    e.set_timing(False)
    dyn_ms = float(np.median(dyn))
    print(f"tick dynamics kernel: median {dyn_ms:.3f} ms over {len(dyn)} ticks")

    nx, neq, nin = e.problem_sizes()
    for parts in (("H", "g", "CE", "ce0", "CI", "ci0"), ("H", "g", "CE", "ce0")):
        out = None
        for _ in range(args.warmup):
            out = e.problem_data(qd, vd, md, rd, parts=parts)
        torch.cuda.synchronize()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = []
        for _ in range(args.iters):
            start.record()
            out = e.problem_data(qd, vd, md, rd, parts=parts)
            stop.record()
            stop.synchronize()
            times.append(start.elapsed_time(stop))
        ms = float(np.median(times))
        sz = out["sizes"].cpu().numpy().astype(np.int64)
        per_env_pad = {"H": nx * nx, "g": nx, "CE": neq * nx, "ce0": neq, "CI": nin * nx, "ci0": nin}
        per_env_used = {"H": sz[:, 0] ** 2, "g": sz[:, 0], "CE": sz[:, 1] * sz[:, 0], "ce0": sz[:, 1],
                        "CI": sz[:, 2] * sz[:, 0], "ci0": sz[:, 2]}
        stored = n * 8 * sum(per_env_pad[k] for k in parts) + n * 12
        used = 8 * int(sum(per_env_used[k].sum() for k in parts)) + n * 12
        rate = stored / (ms * 1e-3)
        print(f"parts {','.join(parts)}: {ms:.3f} ms per call (median of {args.iters}, min {min(times):.3f}, max {max(times):.3f}); "
              f"stored {stored / 1e9:.3f} GB ({used / 1e9:.3f} GB inside the envs' sizes); "
              f"{rate / 1e9:.0f} GB/s = {100 * rate / HBM_BYTES_PER_S:.1f} % of 7.7 TB/s for the whole call; "
              f"export kernel alone ~{ms - dyn_ms:.3f} ms (call minus the tick's dynamics kernel) = "
              f"{stored / ((ms - dyn_ms) * 1e-3) / 1e9:.0f} GB/s, {100 * stored / ((ms - dyn_ms) * 1e-3) / HBM_BYTES_PER_S:.1f} %")
        del out
        torch.cuda.empty_cache()
    e.close()


if __name__ == "__main__":
    main()
