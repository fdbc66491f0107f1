"""Host-side data-format edges of generate_gesture (CPU): BVH parse / feature extraction / BVH write of this package against what
the reference's own functions returned for the same inputs (tests/golden/animation_io.npz and pose_post.npz, oracle/make_golden.py)."""
import os

import numpy as np

from oracle import make_golden as mg, pose_oracle as po
from tests import _fixtures as fx
from zeggs_b200 import animation, bvhio, generate


def test_pose_oracle_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "pose_post.npz"))
    for n in range(2):
        pos, eul = po.pose_to_bvh_channels(g["root_pos"][n], g["root_rot"][n], g["lpos"][n], g["ltxy"][n])
        assert np.abs(pos - g[f"positions{n}"]).max() <= 2e-5 * max(1.0, np.abs(g[f"positions{n}"]).max())
        assert np.abs(eul - g[f"rotations{n}"]).max() <= 2e-3          # degrees
        q = po.quat_from_xform(po.orthogonalize_from_xy(g["ltxy"][n]))
        assert np.abs(q - g[f"lrot{n}"]).max() <= 1e-5


def test_split_by_ratio():
    assert generate.split_by_ratio(240, [0.5, 0.5]) == [[0, 120], [120, 240]]
    assert generate.split_by_ratio(241, [0.25, 0.75]) == [[0, 60], [60, 241]]


def test_bvh_round_trip(tmp_path):
    p = fx.make_synthetic_bvh(str(tmp_path / "s.bvh"), frames=12)
    a = animation.load_bvh(p)
    assert a["rotations"].shape == (12, 75, 3) and a["order"] == "zyx" and abs(a["frametime"] - 0.016667) < 1e-9
    bvhio.save_bvh(str(tmp_path / "t.bvh"), a["positions"], a["rotations"], a["parents"], a["names"], a["order"], a["frametime"])
    b = animation.load_bvh(str(tmp_path / "t.bvh"))
    assert np.abs(a["rotations"] - b["rotations"]).max() <= 1e-5 and np.abs(a["positions"] - b["positions"]).max() <= 1e-5
    assert list(a["parents"]) == list(b["parents"]) and a["names"] == b["names"]


def test_bvh_writer_is_byte_identical_to_the_reference_writer(tmp_path, golden_dir):
    ref = np.load(os.path.join(golden_dir, "animation_io.npz"))["writer_bvh"].tobytes()
    d = fx.skeleton()
    rs = np.random.RandomState(0)
    pos = rs.randn(5, 75, 3).astype(np.float32); rot = (rs.randn(5, 75, 3) * 50).astype(np.float32)
    bvhio.save_bvh(str(tmp_path / "b.bvh"), pos, rot, d["parents"], d["bone_names"], "zyx", d["dt"])
    assert open(tmp_path / "b.bvh", "rb").read() == ref


def test_load_and_preprocess_animation_match_the_reference(tmp_path, golden_dir):
    g = np.load(os.path.join(golden_dir, "animation_io.npz"))
    p = fx.make_synthetic_bvh(str(tmp_path / "s.bvh"), frames=120)
    a = animation.load_bvh(p)
    for k in ("rotations", "positions", "offsets", "parents"):
        assert np.array_equal(fx.digest(np.asarray(a[k], dtype=np.float64)), g["load_" + k]), k
    for tag, cut in mg.ANIM_CUTS.items():
        O = animation.preprocess_animation(animation.trim(a, cut))
        assert set(O) <= set(mg.ANIM_KEYS)
        for k, v in O.items():
            assert v.shape == tuple(g[f"{tag}_{k}_shape"]), (tag, k)
            ref = g[f"{tag}_{k}_sample"].astype(np.float64)
            got = v.reshape(-1)[mg.anim_sample_index(v.size, k)]
            assert np.abs(ref - got).max() <= 1e-5 * max(1.0, float(g[f"{tag}_{k}_absmax"])), (tag, k)
