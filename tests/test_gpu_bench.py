"""bench.py end to end at a small size: --steps sets the number of timed steps, and --dump-outputs writes what the timed
paths returned in their last step (the MSM result and the batch verifier's decisions)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_bench_steps_and_dump_outputs(tmp_path):
    dump = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3", "--lgn", "12", "--strong", "",
           "--verify-proofs", "64", "--verify-reps", "1", "--verify-prover-check", "1", "--dump-outputs", str(dump)]
    env = dict(os.environ, BP_BENCH_NO_SWEEP="1")          # no size sweep, no CPU baseline of the MSM leg
    out = subprocess.run(cmd, cwd=tmp_path, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-4000:])
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    msm = np.load(dump / "msm_result.npy")
    assert msm.dtype == np.float64 and msm.shape == (2, 8)
    assert msm.astype("<u4").tobytes().hex() == line["result"]
    assert line["verify"]["decisions_ok"] is True, line["verify"]
    accept = np.load(dump / "verify_accept.npy")
    assert accept.dtype == np.float32
    assert accept.tolist() == [0.0 if i % 16 == 15 else 1.0 for i in range(64)]      # the bench corrupts every 16th proof
