"""bench.py --dump-outputs: the arrays it writes are what the timed step (config[1]: n=3, 65,536 envs, fixed
random actions, H=1000) computed, checked on sampled environments against the CPU oracle."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_match_oracle(O, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-ars",
                          "--no-cpu", "--no-sustained", "--dump-outputs", str(tmp_path)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["final_state.npy", "returns.npy"]
    ret, fin = np.load(tmp_path / "returns.npy"), np.load(tmp_path / "final_state.npy")
    n, B, H = 3, 65536, 1000
    assert ret.dtype == fin.dtype == np.float64 and ret.shape == (B,) and fin.shape == (B, 2 * n + 2)
    actions = np.random.default_rng(0).uniform(-5, 5, (B, n - 1))   # bench.py's inputs on rank 0
    idx = np.concatenate([[0, 1, 63, 64, B - 1], np.random.default_rng(1).integers(0, B, 27)])
    want_r, want_f = O.rollout_fixed_batch(O.make_params(n=n), O.GYM, actions[idx], H)
    np.testing.assert_array_less(np.abs(ret[idx] - want_r), 1e-6 * np.maximum(1e-3, np.abs(want_r)))
    assert np.max(np.abs(fin[idx] - want_f)) < 1e-8 * max(1.0, np.max(np.abs(want_f)))
