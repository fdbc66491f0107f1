"""Window supplier (zeggs_b200.data.WindowDataset) against the reference dataset (ZEGGS/dataset.py:9-204) on a synthetic
processed_data.npz with the reference's schema (data_pipeline.py:650-684): same sliding windows, same style-example windows
(edge clamping, tail repetition), same one-hot labels.  What the reference returned is stored in tests/golden/dataset_windows.npz
(oracle/make_golden.py dataset): window rows and range indices as they are, every returned tensor as a fingerprint of its bytes."""
import os

import numpy as np
import pytest
import torch

from tests import _fixtures as fx
from zeggs_b200.data import KEYS, WindowDataset


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    return fx.write_processed_data(str(tmp_path_factory.mktemp("ds")))


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "dataset_windows.npz"))


@pytest.mark.parametrize("window,ex_len", [(64, 128), (100, 256), (64, 64)])
def test_windows_and_examples_match_reference(files, golden, window, ex_len):
    ddef, dproc = files
    tag = f"w{window}_ex{ex_len}"
    ours = WindowDataset(ddef, dproc, window, "example", ex_len, seed=0)
    assert len(ours) == int(golden[tag + "_len"])
    rs = np.random.RandomState(window)
    idx = list(rs.randint(0, len(ours), size=40)) + [0, len(ours) - 1]
    assert np.array_equal(idx, golden[tag + "_idx"])
    for j, i in enumerate(idx):
        ref_rows, ref_digest = golden[tag + "_R"][j], golden[tag + "_digest"][j]
        start, ri = int(ours.starts[i]), int(ours.rng_idx[i])
        rows = torch.arange(start, start + window)
        assert np.array_equal(rows.numpy(), ref_rows) and ri == int(golden[tag + "_S"][j])
        assert np.array_equal(fx.digest(ours.X[rows].numpy()), ref_digest[0])
        for k, key in enumerate(KEYS):
            assert np.array_equal(fx.digest(ours.Y[key][rows].numpy()), ref_digest[1 + k]), key
        ex = ours._example(start, ri)
        assert np.array_equal(fx.digest(ex.numpy()), ref_digest[10])


def test_label_batches_and_host_batches(files, golden):
    ddef, dproc = files
    ref_L = torch.from_numpy(golden["label_w64_L"])
    ours = WindowDataset(ddef, dproc, 64, "label", 128, seed=5)
    assert len(ours) == len(ref_L)
    b = ours.sample_host_batch(6)
    assert b["style"].shape == (6, 3) and torch.all(b["style"].sum(1) == 1)
    assert b["audio"].shape == (6, 64, 81) and b["lpos"].shape == (6, 64, 75, 3)
    # every sampled label is the label of the range its window came from
    ours2 = WindowDataset(ddef, dproc, 64, "label", 128, seed=5)
    idx = ours2.rs.randint(0, len(ours2.starts), size=6)
    for r, i in enumerate(idx):
        assert torch.equal(b["style"][r], ref_L[int(i)])
