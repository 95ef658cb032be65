"""bench.py --dump-outputs: the files hold what the timed tick computed on the bench's own seeded inputs."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from common import assert_parity, compare_outputs, setup

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_of_a_sampled_multi_chunk_batch_match_the_oracle(tmp_path):
    """300000 envs: three handle calls per step (CHUNK = 131072, a ragged last one) and more than the dump's byte budget,
    so the dump is a seeded sample.  Rows spread over all three chunks are checked against the oracle on the inputs the
    bench generates (make_workload, seed 0 for rank 0)."""
    n = 300000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", str(n),
                        "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["envs_per_gpu"] == n

    files = sorted(os.path.basename(p) for p in glob.glob(os.path.join(tmp_path, "*.npy")))
    assert files == sorted(f"v1_{k}.npy" for k in bench.DUMP_FIELDS + ("env",))
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in files) <= 64e6
    d = {f[3:-4]: np.load(os.path.join(tmp_path, f)) for f in files}
    assert all(a.dtype == np.float64 for a in d.values())
    env = d["env"].astype(np.int64)
    assert 0 < len(env) < n and (np.diff(env) > 0).all() and env[0] >= 0 and env[-1] < n
    assert env[-1] >= 2 * bench.CHUNK  # the sample reaches the last chunk

    s = setup("v1")
    q, v, mask, refs = bench.make_workload("v1", "walking", n, 0, s["q0"], s["refs"])
    rows = np.linspace(0, len(env) - 1, 512).astype(np.int64)
    e = env[rows]
    words = d["active_set"][rows].astype(np.uint64).reshape(-1, 3, 2)
    out = {"tau": d["tau"][rows], "ddq": d["ddq"][rows], "f": d["f"][rows],
           "status": d["status"][rows].astype(np.int32), "iters": d["iters"][rows].astype(np.int32),
           "active_set": ((words[..., 1] << np.uint64(32)) | words[..., 0]).view(np.int64).T}
    res, _ = compare_outputs("v1", q[e], v[e], mask[e], {k: a[e] for k, a in refs.items()}, out)
    assert_parity(res)
