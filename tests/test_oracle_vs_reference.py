"""Pin the oracle against the reference: against the live reference with the shipped pretrained v1 weights (skipped where the
reference tree is absent), and against the reference's preprocess_audio output stored in tests/golden/mel_clip90.npz."""
import os

import numpy as np
import pytest
import torch

from oracle import model_oracle as mo
from oracle import ref_shim
from zeggs_b200 import synth

NAMES = ["root_pos", "root_rot", "root_vel", "root_vrt", "lpos", "ltxy", "lvel", "lvrt"]


@pytest.fixture(scope="module")
def pretrained():
    if not ref_shim.available():
        pytest.skip("reference tree not present")
    nets = ref_shim.load_pretrained("v1")
    P = {}
    for pre, key in (("speech_encoder.", "speech_encoder"), ("style_encoder.", "style_encoder"), ("decoder.", "decoder")):
        for k, v in nets[key].state_dict().items():
            P[pre + k] = v.clone()
    return nets, P


def test_pretrained_v1_forward(pretrained):
    nets, P = pretrained
    st = synth.load_stats()
    f = lambda k: torch.as_tensor(st[k], dtype=torch.float32)
    B, T, T_ex = 2, 24, 48
    win = {k: torch.from_numpy(v) for k, v in synth.make_pose_windows(B, T, seed=21).items()}
    audio = torch.from_numpy(synth.make_audio_features(B, T, seed=21))
    ex = torch.from_numpy(synth.make_style_example(B, T_ex, seed=21))
    with torch.no_grad():
        a = (audio - f("audio_input_mean")) / f("audio_input_std")
        sp_ref = nets["speech_encoder"](a)
        sp = mo.speech_encoder(P, a)
        assert torch.max(torch.abs(sp - sp_ref)) <= 2e-6
        e = (ex - f("anim_input_mean")) / f("anim_input_std")
        enc_ref = nets["style_encoder"].encoder(e)
        _, mu, logvar = mo.style_encoder(P, e)
        assert torch.max(torch.abs(torch.cat([mu, logvar], 1) - enc_ref)) <= 1e-5
        style = mu.unsqueeze(1).repeat(1, T, 1)
        args = [win[n][:, 0] for n in NAMES] + [win["gaze_pos"], sp_ref, style]
        O_ref = nets["decoder"](*args, torch.as_tensor(st["parents"]), f("anim_input_mean"), f("anim_input_std"),
                                f("anim_output_mean"), f("anim_output_std"), float(st["dt"]))
        O = mo.decoder_forward(P, *args, f("anim_input_mean"), f("anim_input_std"), f("anim_output_mean"),
                               f("anim_output_std"), float(st["dt"]))
        for n, o, r in zip(NAMES, O, O_ref):
            tol = 5e-5 * max(1.0, float(r.abs().max()))
            assert torch.max(torch.abs(o - r)) <= tol, n


def test_live_mel_matches(golden_dir):
    """preprocess_audio of a 1.5 s clip at 60 fps / 90 frames against the reference's output (oracle/make_golden.py mel_clip)."""
    from oracle import mel_oracle
    g = np.load(os.path.join(golden_dir, "mel_clip90.npz"))
    wav = synth.make_waveforms(1, int(g["n_samples"]), seed=int(g["wav_seed"]))[0]
    ref = g["feat"]
    assert ref.shape == (90, 81)
    got = mel_oracle.preprocess_audio(wav, 60, 90)
    assert np.max(np.abs(ref - got)) <= 1e-6
