"""CPU unit test of the per-frame loss math shared by the CUDA kernels (csrc/loss_frame.cuh): the header is
compiled as HOST code into a scratch harness (tests/host/loss_host.cu) and checked against the oracle's
autograd (train.py:277-421 restated in oracle/model_oracle.py).  No GPU involved."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import model_oracle as mo
from tests._util import NAMES, ROOT
from zeggs_b200 import synth

Q_CH = 2496
GROUPS = [  # (start, n, term, w, dterm, dw)
    (0, 3, 0, 0.1, -1, 0), (3, 9, 1, 10.0, -1, 0), (12, 3, 2, 0.1, -1, 0), (15, 3, 3, 5.0, -1, 0),
    (18, 225, 4, 15.0, 12, 7.0), (243, 450, 5, 15.0, 13, 8.0), (693, 225, 6, 10.0, -1, 0), (918, 225, 7, 7.0, -1, 0),
    (1143, 225, 8, 0.1, 14, 0.06), (1368, 675, 9, 3.0, 15, 1.25), (2043, 225, 10, 0.06, -1, 0), (2268, 225, 11, 1.25, -1, 0),
    (2493, 3, 16, 10.0, -1, 0)]


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("host") / "libzeggs_loss_host.so")
    src = os.path.join(ROOT, "tests", "host", "loss_host.cu")
    r = subprocess.run(["/usr/local/cuda/bin/nvcc", "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-o", out, src],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("nvcc host harness build failed: " + r.stderr[-400:])
    return C.CDLL(out)


def pack(w):
    B, T = w["root_vel"].shape[:2]
    return np.concatenate([w[k].reshape(B, T, -1) for k in ("root_vel", "root_vrt", "lpos", "ltxy", "lvel", "lvrt")], axis=2)


def P(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("B,T", [(2, 5), (4, 7)])
def test_loss_frame_math_matches_oracle_autograd(harness, B, T):
    st = synth.load_stats()
    parents = st["parents"].astype(np.int32)
    dt = float(st["dt"])
    O = synth.make_pose_windows(B, T, seed=31)
    W = synth.make_pose_windows(B, T, seed=32)
    gaze = W["gaze_pos"]
    n = B * T
    stride = (n + 31) // 32 * 32
    Qs, Yss = [], []
    for X in (O, W):
        Ys = np.zeros((1131, stride), np.float32)
        Ys[:, :n] = pack(X).reshape(n, 1131).T
        Q = np.zeros((Q_CH, stride), np.float32)
        harness.loss_forward_host(P(Ys), C.c_size_t(stride), C.c_size_t(n), T, P(np.ascontiguousarray(X["root_rot"].reshape(n, 4))),
                                  P(np.ascontiguousarray(X["root_pos"].reshape(n, 3))), P(np.ascontiguousarray(gaze.reshape(n, 3))), P(parents), P(Q))
        Qs.append(Q); Yss.append(Ys)
    D = (Qs[0] - Qs[1])[:, :n].reshape(Q_CH, B, T)
    terms = np.zeros(17)
    G = np.zeros((Q_CH, stride), np.float32)
    g = np.zeros((Q_CH, B, T))
    for s, c, term, w, dterm, dw in GROUPS:
        d = D[s:s + c]
        terms[term] += w * np.abs(d).mean()
        g[s:s + c] += w * np.sign(d) / d.size
        if dterm >= 0:
            e = (d[:, :, 1:] - d[:, :, :-1]) / dt
            terms[dterm] += dw * np.abs(e).mean()
            ge = dw * np.sign(e) / e.size / dt
            g[s:s + c, :, 1:] += ge
            g[s:s + c, :, :-1] -= ge
    G[:, :n] = (g / 18.0).reshape(Q_CH, n)
    gYs = np.zeros((1131, stride), np.float32)
    dpos = np.zeros((n, 3), np.float32); dq = np.zeros((n, 4), np.float32); dqp = np.zeros((n, 4), np.float32)
    harness.loss_backward_host(P(Yss[0]), P(Qs[0]), P(G), C.c_size_t(stride), C.c_size_t(n), T,
                               P(np.ascontiguousarray(O["root_rot"].reshape(n, 4))), P(np.ascontiguousarray(O["root_pos"].reshape(n, 3))),
                               P(np.ascontiguousarray(gaze.reshape(n, 3))), P(parents), P(gYs), P(dpos), P(dq), P(dqp))
    dq = dq.reshape(B, T, 4); dqp = dqp.reshape(B, T, 4)
    dq_tot = dq.copy()
    dq_tot[:, 0] += dqp[:, 0]
    dq_tot[:, :-1] += dqp[:, 1:]
    # oracle
    Ot = [torch.from_numpy(O[k]).clone().requires_grad_(True) for k in NAMES]
    Wt = [torch.from_numpy(W[k]) for k in NAMES]
    loss, L = mo.train_losses(Ot, Wt, torch.from_numpy(gaze), st["parents"], dt)
    grads = torch.autograd.grad(loss, Ot)
    for i, k in enumerate(mo.LOSS_NAMES):
        assert abs(terms[i] - float(L[k])) <= 2e-5 * max(1e-3, abs(float(L[k]))), k
    assert abs(terms.sum() / 18 - loss.item()) <= 2e-5 * abs(loss.item())
    ref_gY = np.concatenate([grads[i].numpy().reshape(B, T, -1) for i in range(2, 8)], axis=2)
    got_gY = gYs[:, :n].T.reshape(B, T, 1131)
    for name, lo, hi in (("vel", 0, 3), ("vrt", 3, 6), ("lpos", 6, 231), ("ltxy", 231, 681), ("lvel", 681, 906), ("lvrt", 906, 1131)):
        err = np.abs(got_gY[..., lo:hi] - ref_gY[..., lo:hi]).max()
        sc = np.abs(ref_gY[..., lo:hi]).max()
        assert err <= 3e-4 * sc, (name, err, sc)
    assert np.abs(dpos.reshape(B, T, 3) - grads[0].numpy()).max() <= 3e-4 * np.abs(grads[0].numpy()).max()
    assert np.abs(dq_tot - grads[1].numpy()).max() <= 3e-4 * np.abs(grads[1].numpy()).max()
