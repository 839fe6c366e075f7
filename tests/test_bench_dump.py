"""bench.py --dump-outputs: the files hold what the timed path returned in its LAST step (the query batch of step
warmup + steps - 1), and the same arguments give the same inputs, hence the same outputs, from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, NQ, K, STEPS, WARMUP = 60_000, 3000, 10, 3, 2


def run_bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(STEPS), "--warmup", str(WARMUP),
           "--n", str(N), "--nq", str(NQ), "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    return line, np.load(os.path.join(out_dir, "scores.npy")), np.load(os.path.join(out_dir, "ids.npy"))


def test_dump_outputs_hold_the_last_timed_step_and_repeat(tmp_path):
    import torch
    from vearch_b200 import synth
    line, scores, ids = run_bench(tmp_path / "a")
    assert line["steps"] == STEPS and line["warmup"] == WARMUP
    assert sorted(os.listdir(tmp_path / "a")) == ["ids.npy", "scores.npy"]
    assert scores.dtype == np.float32 and ids.dtype == np.float64 and scores.shape == ids.shape == (NQ, K)
    assert (ids >= 0).all() and (ids < N).all() and (np.diff(scores, axis=1) >= 0).all()
    # IVF-PQ with exact re-rank on integer-valued data: each score is the exact L2 distance between the returned
    # vector and the query of the last timed batch (bench.py seeds: database 1234 + chunk, queries 4321 + batch)
    db = synth.sift_like_torch(N, 128, seed=1234, device="cuda:0")
    xq = synth.sift_like_torch(NQ, 128, seed=4321 + WARMUP + STEPS - 1, device="cuda:0")
    vec = db[torch.from_numpy(ids.astype(np.int64)).cuda()]
    exact = ((vec - xq[:, None, :]) ** 2).sum(-1).cpu().numpy()
    assert np.array_equal(exact, scores)
    _, scores2, ids2 = run_bench(tmp_path / "b")
    assert np.array_equal(scores2, scores) and np.array_equal(ids2, ids)
