"""Deterministic synthetic inputs for the generate_gesture end-to-end tests: a 75-joint BVH on the shipped skeleton (bone names /
parents of data_definition.json, offsets = mean local joint positions of stats.npz) with small-angle random-walk rotations, and a
16 kHz int16 WAV.  Pure numpy + '%f' text, so the dev container (where the reference produces the golden) and the GPU box (where
the CUDA path is checked against it) write byte-identical files."""
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
DATA = os.path.join(os.path.dirname(HERE), "ubisoft-laforge-zeroeggs_b200", "data")


def skeleton():
    with open(os.path.join(DATA, "data_definition_v1.json")) as f:
        return json.load(f)


def make_synthetic_bvh(path, frames=420, seed=31):
    from zeggs_b200 import bvhio, synth
    d = skeleton()
    st = synth.load_stats()
    J = len(d["parents"])
    rs = np.random.RandomState(seed)
    offsets = st["anim_input_mean"][6:6 + 3 * J].reshape(J, 3).astype(np.float64)
    rot = np.cumsum(rs.randn(frames, J, 3) * 0.35, axis=0)                       # degrees, random walk
    rot += 12.0 * np.sin(np.arange(frames)[:, None, None] / 37.0 + rs.rand(1, J, 3) * 6.28)
    rot[:, 0] = np.cumsum(rs.randn(frames, 3) * 0.2, axis=0) + np.array([0.0, 25.0, 0.0])   # hips: a slow turn
    pos = np.repeat(offsets[None], frames, axis=0)
    pos[:, 0] = np.array([0.0, 92.0, 0.0]) + np.cumsum(rs.randn(frames, 3) * 0.3, axis=0) * np.array([1.0, 0.05, 1.0])
    bvhio.save_bvh(path, pos.astype(np.float32), rot.astype(np.float32), d["parents"], d["bone_names"], "zyx", d["dt"])
    return path


def write_processed_data(d):
    """A 900-frame processed_data.npz with the reference's schema (data_pipeline.py:650-684) plus its data_definition.json, in
    directory `d`; the 120-frame middle range is short enough to exercise the style-example clamping and tail repetition."""
    from zeggs_b200 import synth
    from zeggs_b200.data import KEYS
    st = synth.load_stats()
    rs = np.random.RandomState(3)
    N = 900
    data = {"X_audio_features": rs.randn(N, 81).astype(np.float32)}
    win = synth.make_pose_windows(1, N, seed=4)
    for k in KEYS:
        data["Y_" + k] = win[k][0]
    ranges = np.array([[0, 300], [300, 420], [420, 900]], dtype=np.int64)
    data.update(ranges_train=ranges, ranges_valid=ranges[:1], ranges_train_labels=np.array([0, 2, 1]),
                ranges_valid_labels=np.array([0]))
    for k in ("audio_input_mean", "audio_input_std", "anim_input_mean", "anim_input_std", "anim_output_mean", "anim_output_std"):
        data[k] = st[k]
    np.savez(os.path.join(d, "processed_data.npz"), **data)
    details = dict(bone_names=[f"b{i}" for i in range(75)], label_names=["Neutral", "Happy", "Sad"],
                   parents=[int(p) for p in st["parents"]], dt=float(st["dt"]))
    with open(os.path.join(d, "data_definition.json"), "w") as f:
        json.dump(details, f)
    return os.path.join(d, "data_definition.json"), os.path.join(d, "processed_data.npz")


def digest(x):
    """16-byte fingerprint (uint8[16]) of an array's dtype, shape and bytes: equal fingerprints <=> bit-identical arrays."""
    import hashlib
    a = np.ascontiguousarray(np.asarray(x))
    return np.frombuffer(hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).digest()[:16], dtype=np.uint8)


def make_wav(path, seconds=4.0, seed=32):
    from scipy.io import wavfile
    from zeggs_b200 import synth
    x = synth.make_waveforms(1, int(16000 * seconds), seed=seed)[0]
    wavfile.write(path, 16000, np.round(x * 20000.0).astype(np.int16))
    return path
