"""`bench.py --dump-outputs`: the last timed decode step's logits and states as float .npy files -- the same bits from two runs
with the same arguments, and the oracle's logits and states for the same seeded tokens."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from ai00_server_b200 import synth
from oracle import rwkv_numpy as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRESET, BATCH, PROMPT, WARMUP, STEPS = "tiny6", 3, 5, 3, 4


def rel_err(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def run_bench(out_dir):
    env = dict(os.environ, B200RWKV_BENCH_PROMPT=str(PROMPT), B200RWKV_BENCH_SKIP_EXACT="1")
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--preset", PRESET, "--batch", str(BATCH), "--steps", str(STEPS),
           "--warmup", str(WARMUP), "--cpu-steps", "0", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == STEPS
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in os.listdir(out_dir)) <= 64 << 20
    return {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def test_dump_outputs_are_reproducible_and_match_the_oracle(tmp_path):
    a, b = run_bench(tmp_path / "a"), run_bench(tmp_path / "b")
    assert sorted(a) == ["logits", "state"]
    for k in a:
        assert a[k].dtype == np.float32 and np.array_equal(a[k], b[k]), k
    import bench
    shape = synth.PRESETS[PRESET]
    n = PROMPT + WARMUP + STEPS                        # the prompt, then one token per warm-up and timed step
    toks = bench.make_tokens(PROMPT + 2 * (WARMUP + STEPS) + 8, BATCH, shape.V)
    orc = O.Oracle(O.parse_st(synth.make_st(shape, 0)), "f16")
    assert a["logits"].shape == (BATCH, shape.V)
    for s in range(BATCH):
        want, state = orc.run(toks[s, :n].tolist(), orc.state_init())
        assert rel_err(a["logits"][s], want[0]) <= 1e-3 and a["logits"][s].argmax() == want[0].argmax(), s
        assert rel_err(a["state"][s], state) <= 1e-3, s
