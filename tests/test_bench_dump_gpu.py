"""bench.py --dump-outputs: the outputs of the last timed train step land as float .npy files (at most 64 MB), and two runs with
the same arguments write identical arrays, so that two builds of the project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests._util import ROOT

pytestmark = pytest.mark.gpu


def _bench(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3", "--alt", "0",
                        "--extras", "0", "--no-cpu", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_are_written_and_repeatable(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    runs = [tmp_path / "a", tmp_path / "b"]
    for d in runs:
        assert _bench(d)["steps"] == 2
    names = sorted(os.listdir(runs[0]))
    assert names == ["grads_sample.npy", "loss.npy", "loss_terms.npy", "params_sample.npy"]
    assert sum(os.path.getsize(runs[0] / n) for n in names) <= 64 << 20
    for n in names:
        a, b = np.load(runs[0] / n), np.load(runs[1] / n)
        assert a.dtype == np.float32 and np.all(np.isfinite(a)), n
        assert np.array_equal(a, b), n
    assert np.load(runs[0] / "loss.npy") == np.load(runs[0] / "loss_terms.npy")[0]
