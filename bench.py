#!/usr/bin/env python
"""bench.py — TSID QP ticks/s (robot/v1, batch 65536 per GPU) and tick latency.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores
    python bench.py --config {standing4096,walking65536,legacy16384,mixed1M} [--data replay]
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as .npy

One "step" = one TSID tick (computeProblemData + solve + decode, ref:main.py:119-127) of every env of the
batch.  The headline workload (default) is BASELINE.json configs[2]: robot/v1 LIPM walking, 65536 envs per GPU
with per-env contact phases (20 % double support, 40 % / 40 % single support), swing-foot and CoM references and
random perturbed states (SURVEY.md §8d, seed 0).  Weak scaling: every rank owns its own 65536 envs; the only
collective is the all-gather of the per-tick diagnostics.  --config selects the other BASELINE configs
(configs[1] standing, configs[3] legacy OP3, configs[4] v0+v1 mixed 1 M envs sharded by env index: strong
scaling); --data replay times ticks over states RECORDED from a closed-loop device rollout (tick -> integrate ->
gait phase machine), one recorded step per timed step, instead of independent random states.

Rank 0 prints ONE JSON line.  `value` is measured with inputs resident in HBM, CUDA events around every
step on the launching stream, an L2 flush between steps (outside the events), max over ranks.  `e2e` is the
same tick through the host-buffer entry point tsidb_compute_host (pinned host buffers, H2D, kernels, D2H inside
the timed region); `e2e_device_refs` is the deployment the device gait makes possible: references and contact
phases stay on the device (tsidb_compute_host_devrefs), only q and v are uploaded per tick.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "tsid_qp_ticks_per_sec"
UNIT = "ticks/s"

# parts: (controller kind, share of the envs) — 'v1' = WalkController + ctrl/conf.py, 'v0' = legacy Biped + op3_conf;
# n: envs per GPU (weak scaling) or in total (strong scaling)
CONFIGS = {
    "standing4096": dict(parts=[("v1", 1.0)], n=4096, mode="standing", scaling="weak",
                         workload="robot/v1 double-support standing balance (BASELINE configs[1]): 4096 envs/GPU, seed 0"),
    "walking65536": dict(parts=[("v1", 1.0)], n=65536, mode="walking", scaling="weak",
                         workload="robot/v1 LIPM walking (BASELINE configs[2]): 65536 envs/GPU, 20% DS / 40% SS-L / 40% SS-R, seed 0"),
    "legacy16384": dict(parts=[("v0", 1.0)], n=16384, mode="walking", scaling="weak",
                        workload="legacy OP3 model (robot/v0 + op3_conf) walking (BASELINE configs[3]): 16384 envs/GPU, "
                                 "single/double-support contact switching, seed 0"),
    "mixed1M": dict(parts=[("v0", 0.5), ("v1", 0.5)], n=1 << 20, mode="walking", scaling="strong",
                    workload="robot/v0 + robot/v1 mixed walking (BASELINE configs[4]): 1048576 envs in total, first half v0 "
                             "(op3_conf), second half v1, contiguous by model, sharded by env index over the GPUs, seed 0"),
}
GAIT = {"v1": (0.3, 0.2, 0.2, 0.5), "v0": (0.1, 0.1275, 0.05, 0.7)}  # ref:ctrl/conf.py:24-28, ref:legacy/op3_conf.py:9-12
CHUNK = 131072  # envs per handle call (workspace 30 KB per env)
DUMP_FIELDS = ("tau", "ddq", "f", "status", "iters", "active_set")  # what TsidEngine.compute hands the bench's tick
DUMP_BYTES = 60 << 20  # array bytes of --dump-outputs over all ranks; with the .npy headers the files stay under 64 MB


# ----------------------------------------------------------------------------------------------
def algorithmic_flops(kind: str, mask: np.ndarray, iters: np.ndarray) -> dict:
    """SURVEY.md §8(d): F/tick = F_dyn + F_asm + F_fact(n) + equality phase + per_iter * it (1 FMA = 2 flop);
    it = active-set iterations that attempted a constraint change = iterations - 1 (the last pass only checks
    feasibility).  v1: DS 0.50 M + 0.020 M it, SS 0.22 M + 0.012 M it; v0: DS 0.46 M + 0.018 M it, SS 0.20 M +
    0.011 M it; flight from the same formula (n = nv, m_e = 6).  Split by the kernel that does the work:
    dynamics+assembly 28 k (F_dyn 20 k + F_asm 8 k), the factorisation and equality phase (elimination kernel,
    which also builds the null-space basis), the iterations (active-set kernel)."""
    nc = (mask & 1) + ((mask >> 1) & 1)
    if kind == "v1":
        base = np.where(nc == 2, 0.50e6, np.where(nc == 1, 0.22e6, 0.075e6))
        per = np.where(nc == 2, 0.020e6, np.where(nc == 1, 0.012e6, 0.0075e6))
    else:
        base = np.where(nc == 2, 0.46e6, np.where(nc == 1, 0.20e6, 0.065e6))
        per = np.where(nc == 2, 0.018e6, np.where(nc == 1, 0.011e6, 0.0065e6))
    it = np.maximum(iters.astype(np.float64) - 1.0, 0.0)
    dyn = 28e3 * len(mask)
    return {"dynamics": float(dyn), "eliminate": float(base.sum() - dyn), "activeset": float((per * it).sum()),
            "tick": float((base + per * it).sum())}


HBM_BYTES_PER_TICK = 1832.0  # SURVEY.md §8(d): 1240 B in + 592 B out (v1, double support)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
def make_workload(kind: str, mode: str, n: int, seed: int, q_stand: np.ndarray, refs0: dict):
    from tsid_control_b200 import synth

    q, v = synth.random_states(q_stand, n, seed)
    if mode == "standing":
        return q, v, np.full(n, 3, np.uint8), {k: np.tile(a, (n, 1)) for k, a in refs0.items()}
    mask, refs = synth.walking_batch(refs0, n, seed, *GAIT[kind], float(refs0["com"][2]))
    return q, v, mask, refs


def shard_parts(cfg: dict, rank: int, world: int):
    """[(kind, n_envs, seed)] this rank owns.  Weak scaling: the whole config per rank.  Strong scaling (mixed1M): the
    global env range is cut by contiguous env index (sharding.shard_range); a rank's slice is split by model."""
    if cfg["scaling"] == "weak":
        return [(cfg["parts"][0][0], cfg["n"], 1000 * rank)]
    from tsid_control_b200.sharding import shard_range

    lo, hi = shard_range(cfg["n"], rank, world)
    out, start = [], 0
    for kind, frac in cfg["parts"]:
        end = start + int(round(frac * cfg["n"]))
        a, b = max(lo, start), min(hi, end)
        if b > a:
            out.append((kind, b - a, 7 * a + 1))  # the seed depends on the global offset only
        start = end
    return out


def run_reference(args) -> None:
    """The reference algorithm (restated CPU port: oracle/, -O3 AVX2 build) on all host threads, on the SAME config:
    every step is one tick of the whole per-GPU batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from common import setup

    cfg = dict(CONFIGS[args.config])
    if args.batch:
        cfg["n"] = args.batch
    cores = os.cpu_count() or 1
    runs, total = [], 0
    for kind, n, seed in shard_parts(cfg, 0, 1):
        if cfg["scaling"] == "strong":
            n = min(n, 32768)  # mixed1M: a bounded sample per model (the whole config needs > 10 s per step on a host)
        s = setup(kind, "liboracle_fast.so")
        q, v, mask, refs = make_workload(kind, cfg["mode"], n, seed, s["q0"], s["refs"])
        runs.append(s["oracle"].timed_batch(q, v, mask, refs, cores))
        total += n
    for _ in range(max(1, args.warmup)):
        for r in runs:
            r()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        for r in runs:
            r()
        times.append(time.perf_counter() - t0)
    val = total * len(times) / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": cfg["scaling"],
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["workload"], "name": args.config, "envs_per_step": total},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{total} envs of the workload per step (the whole per-GPU batch), {cores} threads, restated "
                                   "CPU port of pinocchio+tsid+eiquadprog-fast (oracle/, -O3 x86-64-v3); the reference's own "
                                   "binaries cannot be installed in this image"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def pin_rank_to_cores(local: int, world: int) -> list:
    """One slice of the host cores per rank (the ranks of a box share one NUMA node here: topology shows every GPU
    with the same CPU affinity): the pinned staging buffers are first-touched from the slice that feeds them."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        if world > 1 and len(cores) >= world:
            per = len(cores) // world
            mine = cores[local * per:(local + 1) * per]
            os.sched_setaffinity(0, mine)
            return mine
        return cores
    except Exception:
        return []


class Shard:
    """One (model, env range) of this rank: controller, device-resident inputs, host copies."""

    def __init__(self, kind, n, seed, mode, local, torch):
        if kind == "v1":
            from tsid_control_b200.ctrl.conf import RobotConfig
            from tsid_control_b200.ctrl.WalkController import WalkController

            conf = RobotConfig()
            conf.device, conf.max_envs = local, min(n, CHUNK)
            self.ctrl = WalkController(conf, n_envs=1)
        else:
            import importlib
            import types

            from tsid_control_b200.legacy.biped import Biped

            mod = importlib.import_module("tsid_control_b200.legacy.op3_conf")
            conf = types.SimpleNamespace(**{k: getattr(mod, k) for k in dir(mod) if not k.startswith("_")})
            conf.device, conf.max_envs = local, min(n, CHUNK)
            self.ctrl = Biped(conf, n_envs=1)
        self.kind, self.n, self.eng, self.dev = kind, n, self.ctrl.engine, self.ctrl.device
        self.q, self.v, self.mask, self.refs = make_workload(kind, mode, n, seed, self.ctrl.q, self.ctrl.default_refs)
        t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=self.dev)
        self.qd, self.vd, self.md = t(self.q), t(self.v), t(self.mask)
        self.rd = {k: t(a) for k, a in self.refs.items()}
        self.chunks = [(o, min(o + CHUNK, n)) for o in range(0, n, CHUNK)]
        self.torch = torch

    def set_inputs(self, qd, vd, md, rd):
        self.qd, self.vd, self.md, self.rd = qd, vd, md, rd

    def tick(self, keep=False):
        """One tick of every env of the shard (a handle call per chunk of <= CHUNK envs); returns (status, iters).
        self.outs: the TickOutput of every chunk.  With one chunk that is the engine's buffers (valid until the next
        tick); with several each call overwrites the previous chunk's buffers, so keep=True copies them (inside the
        tick) and otherwise self.outs is None."""
        if len(self.chunks) == 1:
            o = self.eng.compute(self.qd, self.vd, self.md, self.rd, want_active=True)
            self.outs = [o]
            return o.status, o.iters
        outs, self.outs = [], [] if keep else None
        for lo, hi in self.chunks:
            o = self.eng.compute(self.qd[lo:hi], self.vd[lo:hi], self.md[lo:hi], {k: r[lo:hi] for k, r in self.rd.items()})
            outs.append((o.status.clone(), o.iters.clone()))
            if keep:
                from tsid_control_b200.engine import TickOutput

                self.outs.append(TickOutput(**{k: getattr(o, k).clone() for k in DUMP_FIELDS}))
        return self.torch.cat([a for a, _ in outs]), self.torch.cat([b for _, b in outs])


def dump_outputs(out_dir: str, shards, prefix: str, limit: int) -> None:
    """The outputs of the shards' last tick as out_dir/<prefix><kind>_<field>.npy, float64: tau, ddq, f, status, iters,
    active_set as [N, 6] (each of its three 64-bit words as low and high 32 bits, exact in float64) and env, the env index
    within the shard of every row.  Above `limit` bytes every shard keeps the same share of its envs, drawn with a fixed
    seed: with the same arguments the rows are the same envs on the same inputs from run to run."""
    import torch

    bytes_per_env = [8 * (s.eng.na + s.eng.nv + 24 + 2 + 6 + 1) for s in shards]
    total = sum(s.n * b for s, b in zip(shards, bytes_per_env))
    os.makedirs(out_dir, exist_ok=True)
    for s in shards:
        env = np.arange(s.n)
        if total > limit:
            env = np.sort(np.random.default_rng(0).choice(s.n, s.n * limit // total, replace=False))
        idx = torch.as_tensor(env, device=s.dev)
        out = {f: torch.cat([getattr(o, f) for o in s.outs], dim=1 if f == "active_set" else 0) for f in DUMP_FIELDS}
        out = {f: (t[:, idx].T if f == "active_set" else t[idx]).cpu().numpy() for f, t in out.items()}
        words = out["active_set"].view(np.uint64)
        out["active_set"] = np.stack([words & 0xFFFFFFFF, words >> 32], axis=-1).reshape(len(env), 6)
        out["env"] = env
        for f, a in out.items():
            np.save(os.path.join(out_dir, f"{prefix}{s.kind}_{f}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="walking65536", choices=sorted(CONFIGS),
                    help="BASELINE.json config (the metric is quoted on walking65536)")
    ap.add_argument("--data", default="synthetic", choices=["synthetic", "replay"],
                    help="replay: states, contact phases and references recorded from a closed-loop device rollout")
    ap.add_argument("--batch", type=int, default=0, help="override the config's env count (the metric is quoted at the config's own size)")
    ap.add_argument("--replay-stride", type=int, default=5,
                    help="--data replay: control steps (2 ms each) between consecutive snapshots; 1 = consecutive ticks of a controller")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true",
                    help="profiling runs only: skip the end-to-end and latency legs (the line then has no e2e)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the outputs of the last one (tau, ddq, f, status, iters, active_set) "
                         "as DIR/<kind>_<name>.npy, float64, at most 64 MB in all (above that a fixed, seeded sample of the "
                         "envs); configs of more than 131072 envs per model copy each chunk's outputs inside that step")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
        return

    sys.dont_write_bytecode = True  # the tree may be read-only: the modules imported below leave no __pycache__ in it
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    my_cores = pin_rank_to_cores(local, world)  # before CUDA and the pinned allocations exist

    import torch
    import torch.distributed as dist

    import __graft_entry__ as ge

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the TSID tick has no CPU fallback (use --impl reference for the CPU port)")
    if rank == 0:
        ge.build()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    from tsid_control_b200.engine import fp64_peak_tflops
    from tsid_control_b200.sharding import gather_diagnostics

    cfg = dict(CONFIGS[args.config])
    if args.batch:
        cfg["n"] = args.batch
    parts = shard_parts(cfg, rank, world)
    shards = [Shard(kind, n, seed, cfg["mode"], local, torch) for kind, n, seed in parts]
    dev = shards[0].dev
    n_local = sum(s.n for s in shards)
    n_global = cfg["n"] * world if cfg["scaling"] == "weak" else cfg["n"]
    n_pad = -(-cfg["n"] // world) if cfg["scaling"] == "strong" else cfg["n"]  # equal-length shards for the all-gather
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)  # 256 MiB > 126 MB L2
    diag_out = torch.empty((world * n_pad, 2), dtype=torch.int32, device=dev) if world > 1 else None
    diag_st = torch.zeros(n_pad, dtype=torch.int32, device=dev)
    diag_it = torch.zeros(n_pad, dtype=torch.int32, device=dev)

    # ---- replay data: record a closed-loop rollout (tick -> integrate -> gait step on the device), one snapshot per step
    replay, fails = None, 0
    if args.data == "replay":
        if len(shards) != 1 or len(shards[0].chunks) != 1:
            raise SystemExit("--data replay records one rollout per rank: use a single-model config of at most 131072 envs per GPU")
        s = shards[0]
        conf = s.ctrl.conf
        rng = np.random.Generator(np.random.PCG64(12345 + rank))
        phase0 = torch.as_tensor(rng.uniform(0, 1, s.n), device=dev)
        vcmd = torch.as_tensor(np.c_[rng.uniform(-0.3, 0.3, s.n), rng.uniform(-0.1, 0.1, s.n)], device=dev)
        L, W, Hh, T = GAIT[s.kind]
        s.eng.gait_reset(s.n, dt=float(conf.dt), step_duration=T, step_length=L, step_height=Hh,
                         com_height=float(s.ctrl.default_refs["com"][2]), phase0=phase0, vcmd=vcmd)
        qr, vr = s.qd.clone(), s.vd.clone()
        vr *= 0.2  # start near rest: the recorded states are what the controller itself produces afterwards
        post = s.rd["posture"]
        snaps = []
        s.eng.rollout(qr, vr, 25, use_graph=True)  # run in
        for _ in range(max(args.steps, 8)):
            gs = s.eng.gait_state()
            snaps.append((qr.clone(), vr.clone(), gs["mask"].clone(),
                          {"com": gs["com"].clone(), "foot_lf": gs["foot_lf"].clone(), "foot_rf": gs["foot_rf"].clone(),
                           "contact_lf": gs["contact_lf"].clone(), "contact_rf": gs["contact_rf"].clone(), "posture": post}))
            s.eng.rollout(qr, vr, max(1, args.replay_stride), use_graph=True)  # 10 ms of closed loop between snapshots by default
        torch.cuda.synchronize()
        replay = snaps
        fails = int((s.eng.gait_state()["fails"] > 0).sum().item())

    # Scheduling hint (tsidb_set_sched_hint): envs of a contact class ordered by their iteration counts in the previous
    # tick.  A synthetic batch that is ticked again unchanged would make that forecast exact, so the headline of the
    # synthetic workloads is measured with the hint OFF; a replayed rollout (consecutive snapshots 10 ms apart) gives it
    # the forecast a controller has, and is measured with it ON.  The other setting is timed afterwards and reported.
    hint_main = replay is not None
    for s in shards:
        s.eng.set_sched_hint(hint_main)

    step_no = [0]

    def step(keep=False):
        if replay is not None:
            shards[0].set_inputs(*replay[step_no[0] % len(replay)])
            step_no[0] += 1
        off = 0
        res = []
        for s in shards:
            st, it = s.tick(keep)
            res.append((st, it))
            if world > 1:
                diag_st[off:off + s.n] = st
                diag_it[off:off + s.n] = it
            off += s.n
        if world > 1:
            gather_diagnostics(diag_st, diag_it, diag_out)
        return res

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    fp64_peak = fp64_peak_tflops(local)

    sampler = ClockSampler(local)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    step_no[0] = 0
    launches0 = sum(s.eng.launch_count() for s in shards)
    evs = []
    iters_seen, mask_seen = [], []
    for i in range(args.steps):
        flush.zero_()  # evict the inputs from L2 (outside the timed events)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = step(keep=bool(args.dump_outputs) and i == args.steps - 1)
        e1.record()
        evs.append((e0, e1))
        if replay is not None:  # the iteration histogram differs from step to step: keep them all (outside the events)
            iters_seen.append(res[0][1].cpu().numpy().copy())
            mask_seen.append(shards[0].md.cpu().numpy().copy())
    torch.cuda.synchronize()
    if args.dump_outputs:  # before any other tick reuses the output buffers
        dump_outputs(args.dump_outputs, shards, f"rank{rank}_" if world > 1 else "", DUMP_BYTES // world)
    if world > 1:
        dist.barrier()
    launches = sum(s.eng.launch_count() for s in shards) - launches0
    ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = sum(ms)
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = n_global * args.steps / (total_ms * 1e-3)

    def timed_value(k):
        """ticks/s over k more steps with the current hint setting (same flush, events and max over ranks)."""
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ev = []
        for _ in range(k):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step()
            b.record()
            ev.append((a, b))
        torch.cuda.synchronize()
        tot = sum(a.elapsed_time(b) for a, b in ev)
        if world > 1:
            tt = torch.tensor([tot], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            tot = float(tt.item())
        return n_global * k / (tot * 1e-3)

    status_np = np.concatenate([st.cpu().numpy() for st, _ in res])
    iters_np = np.concatenate([it.cpu().numpy() for _, it in res])
    if replay is not None:
        fl = [algorithmic_flops(shards[0].kind, m, i) for m, i in zip(mask_seen, iters_seen)]
        flops = {k: float(np.mean([f[k] for f in fl])) for k in fl[0]}
    else:
        fl = [algorithmic_flops(s.kind, s.mask, it.cpu().numpy()) for s, (_, it) in zip(shards, res)]
        flops = {k: float(sum(f[k] for f in fl)) for k in fl[0]}
    step_ms = statistics.mean(ms)
    # per-kernel durations: CUDA events recorded by the library between its launches, on the launching stream,
    # in separate (untimed) steps with the same L2 flush so the events do not perturb `value`
    kms = {}
    if all(len(s.chunks) == 1 for s in shards):  # the library keeps the events of a handle's last call only
        for s in shards:
            s.eng.set_timing(True)
        per_kernel = {}
        for _ in range(max(3, min(args.steps, 10))):
            flush.zero_()
            step()
            acc = {}
            for s in shards:
                for k, t in s.eng.last_tick_ms().items():
                    acc[k] = acc.get(k, 0.0) + t
            for k, t in acc.items():
                per_kernel.setdefault(k, []).append(t)
        for s in shards:
            s.eng.set_timing(False)
        kms = {k: statistics.mean(v) for k, v in per_kernel.items()}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_ach = HBM_BYTES_PER_TICK * n_local / (step_ms * 1e-3) / 1e9
    kernels = []
    if kms:
        for g in ("dynamics", "eliminate", "activeset"):
            t = kms[g]
            tf = flops[g] / (t * 1e-3) / 1e12
            kernels.append({"kernel": g, "ms": t, "algorithmic_flops_per_launch": flops[g], "achieved": tf,
                            "frac": tf / fp64_peak if fp64_peak else None,
                            "traffic": traffic.get(g) if args.config == "walking65536" else None})
    dom = max(kernels, key=lambda k: k["ms"]) if kernels else None
    tick_tf = flops["tick"] / (step_ms * 1e-3) / 1e12

    # ---- e2e: host buffers through the C ABI (H2D + kernels + D2H inside the call) ----
    # inputs live in pinned host memory (the contract's "from pinned host memory"), results land in pinned
    # host memory; the library cuts the batch into chunks so the copies run under the kernels
    e2e = e2e_dev = e2e_tau = None
    lat = None
    lat_by_class = {}
    if not args.no_e2e:
        e2e_steps = max(3, min(args.steps, 10))
        host = []
        for s in shards:
            for lo, hi in s.chunks:
                hq, hv, hm = s.eng.pin(s.q[lo:hi]), s.eng.pin(s.v[lo:hi]), s.eng.pin(s.mask[lo:hi])
                hr = {k: s.eng.pin(a[lo:hi]) for k, a in s.refs.items()}
                dm = torch.as_tensor(s.mask[lo:hi], device=dev)
                dr = {k: torch.as_tensor(np.ascontiguousarray(a[lo:hi]), device=dev) for k, a in s.refs.items()}
                host.append((s, hq, hv, hm, hr, s.eng.host_buffers(hi - lo, pinned=True), dm, dr))

        def e2e_pass(device_refs):
            outs = []
            for s, hq, hv, hm, hr, hout, dm, dr in host:
                if device_refs:
                    outs.append(s.eng.compute_host_devrefs(hq, hv, dm, dr, out=hout, tau_only=(device_refs == "tau"),
                                                           want_active=(device_refs != "tau")))
                else:
                    outs.append(s.eng.compute_host(hq, hv, hm, hr, out=hout))
            return outs

        results = {}
        for device_refs in (False, True, "tau"):
            for _ in range(2):
                e2e_pass(device_refs)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                ho = e2e_pass(device_refs)
            t_e2e = time.perf_counter() - t0
            if replay is None:
                assert np.array_equal(np.concatenate([o["status"] for o in ho]), status_np), "e2e path disagrees with the device path"
                assert np.array_equal(np.concatenate([o["iters"] for o in ho]), iters_np), "e2e path disagrees with the device path"
            if world > 1:
                t = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                t_e2e = float(t.item())
            results[device_refs] = n_global * e2e_steps / t_e2e
        h2d_full = sum(s.n * (8 * (s.eng.nq + s.eng.nv + 9 + 24 + 24 + 12 + 12 + s.eng.na) + 1) for s in shards)
        h2d_dev = sum(s.n * 8 * (s.eng.nq + s.eng.nv) for s in shards)
        d2h = sum(s.n * (8 * (s.eng.na + s.eng.nv + 24) + 4 + 4 + 24) for s in shards)
        e2e = {"value": results[False], "unit": UNIT, "h2d_bytes_per_step": h2d_full, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
               "api": "tsidb_compute_host via TsidEngine.compute_host: q, v, contact mask and every reference from pinned host buffers, "
                      "results into pinned host buffers, 4 chunks over 3 streams (copies overlap the kernels)"}
        d2h_tau = sum(s.n * (8 * s.eng.na + 4 + 4) for s in shards)
        e2e_tau = {"value": results["tau"], "unit": UNIT, "h2d_bytes_per_step": h2d_dev, "d2h_bytes_per_step": d2h_tau, "steps": e2e_steps,
                   "api": "tsidb_compute_host_devrefs with ddq = f = active_set = NULL: q and v up, tau, status and iters down (what "
                          "ref:main.py:126 sends to the actuators); references on the device"}
        e2e_dev = {"value": results[True], "unit": UNIT, "h2d_bytes_per_step": h2d_dev, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                   "api": "tsidb_compute_host_devrefs: q and v from pinned host buffers; references and contact phases resident on the "
                          "device (the gait state the device phase machine keeps), results into pinned host buffers"}

    # ---- the other setting of the scheduling hint (see above), on every rank ----
    for s in shards:
        s.eng.set_sched_hint(not hint_main)
    value_other = timed_value(max(3, min(args.steps, 10)))
    for s in shards:
        s.eng.set_sched_hint(hint_main)
    sched_hint = {
        "headline": "on" if hint_main else "off", "value_on": value if hint_main else value_other,
        "value_off": value_other if hint_main else value, "unit": UNIT,
        "note": ("envs of a contact class ordered by their iteration counts in the previous tick (tsidb_set_sched_hint; never "
                 "changes a result).  " +
                 ("Replayed rollout: the previous tick is the snapshot 10 ms earlier, the forecast a controller has - headline with it."
                  if hint_main else
                  "Synthetic batch ticked again unchanged: the forecast would be exact, so value / e2e are measured WITHOUT it; "
                  "value_on is the same loop with it."))}

    # the sampler ran from the start of the timed region to here: the GPU was under the same tick load throughout
    # (timed steps, per-kernel timing steps, end-to-end steps), which gives nvidia-smi time for several samples
    clocks = sampler.stop()
    clocks["window"] = "timed steps + per-kernel timing steps + end-to-end steps"

    # ---- single-env tick latency (the reference's own operating point: one robot per call), measured after the clock sampler
    # has stopped: its nvidia-smi polls (a subprocess every few ms, driver queries) added ~20 us to a 77 us call ----
    if not args.no_e2e:
        if rank == 0:
            # p50 over TICKS: 96 different envs of the workload (its contact-class mix), one at a time; per env the median
            # of 9 calls after 3 warm-ups.  A tick's latency follows its active-set iteration count (1 .. ~35), so one
            # env's number says little: the distribution over states is what a controller sees
            s = shards[-1]
            per_env, per_cls = [], {"double_support": [], "single_support": [], "flight": []}
            for i0 in range(min(96, s.n)):
                qc, vc, mc = s.qd[i0:i0 + 1].contiguous(), s.vd[i0:i0 + 1].contiguous(), s.md[i0:i0 + 1].contiguous()
                rc = {k: t[i0:i0 + 1].contiguous() for k, t in s.rd.items()}
                tc = []
                for i in range(12):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    s.eng.compute(qc, vc, mc, rc)
                    torch.cuda.synchronize()
                    tc.append(time.perf_counter() - t0)
                us = statistics.median(tc[3:]) * 1e6
                per_env.append(us)
                m_ = int(s.mask[i0])
                per_cls["double_support" if m_ == 3 else ("flight" if m_ == 0 else "single_support")].append(us)
            lat = statistics.median(per_env)
            lat_by_class = {k: statistics.median(v) for k, v in per_cls.items() if v}
            lat_by_class["p90_all"] = sorted(per_env)[int(0.9 * (len(per_env) - 1))]
            lat_by_class["envs"] = len(per_env)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": total_ms / args.steps, "p50_ms_per_step": statistics.median(ms), "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64", "data": args.data,
        "config": {"workload": cfg["workload"], "name": args.config, "envs_per_gpu": n_local, "global_envs": n_global,
                   "l2_flush_between_steps": True,
                   "timing": "CUDA events per step on the launching stream, flush outside the events, max over ranks",
                   "collective": "all_gather of int32[N_local,2] diagnostics per step" if world > 1 else "none (1 GPU)",
                   "host_cores_of_rank0": len(my_cores)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "solver": {"mean_iters": float(iters_np.mean()), "max_iters": int(iters_np.max()),
                   "status_optimal_frac": float((status_np == 0).mean())},
        "sched_hint": sched_hint,
        "tick_latency_1env_us_p50": lat,
        "tick_latency_1env_us_p50_by_class": lat_by_class or None,
    }
    if replay is not None:
        line["config"]["replay"] = (f"{len(replay)} snapshots of a closed-loop device rollout (tsidb_rollout: tick -> integrate_dv -> gait "
                                    f"phase machine), {max(1, args.replay_stride)} control steps apart after a 25-step run-in; envs that ever failed a tick: {fails}")
    if e2e:
        line["e2e"] = e2e
        line["e2e_device_refs"] = e2e_dev
        line["e2e_tau_only"] = e2e_tau
    if dom:
        line["roofline"] = {
            "bound": "fp64", "achieved": dom["achieved"], "peak": fp64_peak, "unit": "TFLOP/s", "frac": dom["frac"],
            "traffic": dom["traffic"], "kernel": dom["kernel"], "kernel_ms": dom["ms"],
            "algorithmic_flops_per_launch": dom["algorithmic_flops_per_launch"],
            "peak_source": "measured on this GPU by tsidb_fp64_peak (dependent-free DFMA chains); MEASURED_PEAKS.json has no FP64 "
                           "entry; the path is FP64- and shared-memory-bound, not HBM- or tensor-bound (SURVEY.md §8d, DESIGN.md §4)",
            "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full capture in profiles/ "
                              "(profiles/dram_traffic.json)" if traffic else None,
            "tick": {"achieved": tick_tf, "frac": tick_tf / fp64_peak if fp64_peak else None, "ms": step_ms,
                     "algorithmic_flops_per_step": flops["tick"],
                     "launches": "class sort (2) + dynamics + per contact class: elimination (with the null-space basis) + active set"},
            "kernels": kernels, "kernel_ms_all": kms,
            "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                    "algorithmic_bytes_per_tick": HBM_BYTES_PER_TICK,
                    "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}}
    if not args.no_cpu_baseline:
        from common import setup

        s0 = shards[-1]
        so = setup(s0.kind, "liboracle_fast.so")
        cores = os.cpu_count() or 1
        sample = min(s0.n, max(256, min(8192, 512 * cores)))
        run = so["oracle"].timed_batch(s0.q[:sample], s0.v[:sample], s0.mask[:sample], {k: a[:sample] for k, a in s0.refs.items()}, cores)
        run()
        reps, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < 10.0 and reps < 50:
            run()
            reps += 1
        dt = time.perf_counter() - t0
        # single-thread latency of one tick
        run1 = so["oracle"].timed_batch(s0.q[:64], s0.v[:64], s0.mask[:64], {k: a[:64] for k, a in s0.refs.items()}, 1)
        run1()
        t1 = time.perf_counter()
        run1()
        lat_cpu = (time.perf_counter() - t1) / 64 * 1e6
        line["cpu_baseline"] = {"value": sample * reps / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"first {sample} envs of the workload x {reps} passes on {cores} threads; restated CPU port "
                                          "(oracle/, -O3 x86-64-v3), not the reference binaries", "tick_latency_1thread_us": lat_cpu}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
