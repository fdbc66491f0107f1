"""Streaming feature window rule (zeggs_b200.streaming.WindowRule), CPU only: speech features of a stream pushed in random pieces,
recomputed window by window and assembled from the kept rows, equal the whole-clip features (oracle mel front end + oracle
SpeechEncoder in float64)."""
import numpy as np
import pytest
import torch

from tests._util import ROOT  # noqa: F401  (puts the repository on sys.path)


def _speech_fn(hop):
    from oracle import mel_oracle, model_oracle as mo
    from zeggs_b200 import synth
    st = synth.load_stats()
    P = {k: torch.from_numpy(v).double() for k, v in synth.make_params(H=64, seed=61, with_style=False).items()
         if k.startswith("speech_encoder.")}
    mean = torch.as_tensor(st["audio_input_mean"], dtype=torch.float64)
    std = torch.as_tensor(st["audio_input_std"], dtype=torch.float64)

    def speech(x, T):
        feat = torch.from_numpy(mel_oracle.preprocess_audio(x, 60, T, hop=hop)).double()
        return mo.speech_encoder(P, ((feat - mean) / std)[None])[0]
    return speech


def _stream(x, rule, chunk, pieces, speech):
    """The generator's schedule: a step computes chunk + 1 rows from the last emitted frame (frame 0 on the first step) once the
    fixed-length window is there; close() computes the rest on the final window.  -> {global frame: speech row}."""
    W = rule.window_samples(chunk + 1)
    rows, frames_out, received = {}, 0, 0
    for n in pieces:
        received += n
        while True:
            w = rule.plan(received, max(frames_out - 1, 0), False, W)
            if w is None:
                break
            assert w.s1 - w.s0 == W and w.s0 % rule.grid == 0 and w.r1 - w.r0 >= chunk + 1
            sp = speech(x[w.s0:w.s1], w.anim_length)
            for r in range(w.r0, w.r0 + chunk + 1):
                rows[w.k0 + r] = sp[r]
            frames_out += chunk + 1 if frames_out == 0 else chunk
    w = rule.plan(received, max(frames_out - 1, 0), True)
    assert w is not None and w.s1 == len(x) and w.s0 % rule.grid == 0
    sp = speech(x[w.s0:w.s1], w.anim_length)
    for r in range(w.r0, w.r1):
        rows[w.k0 + r] = sp[r]
    assert w.k0 + w.r1 == rule.total_frames(len(x))
    return rows


@pytest.mark.parametrize("n_samples,hop", [(837, 200), (16123, 200), (53211, 200), (16123, 160)])
@pytest.mark.parametrize("chunk", [1, 7, 30])
def test_streamed_speech_features_equal_whole_clip(n_samples, hop, chunk):
    from zeggs_b200 import synth
    from zeggs_b200.streaming import WindowRule
    rule = WindowRule(hop=hop)
    x = synth.make_waveforms(1, n_samples, seed=n_samples)[0]
    rs = np.random.RandomState(n_samples + chunk)
    pieces, left = [], n_samples
    while left:
        pieces.append(min(left, int(rs.randint(1, 3000))))
        left -= pieces[-1]
    speech = _speech_fn(hop)
    T = int(round(60.0 * (n_samples / 16000)))
    ref = speech(x, T)
    rows = _stream(x, rule, chunk, pieces, speech)
    assert sorted(rows) == list(range(T))
    got = torch.stack([rows[k] for k in range(T)])
    err = float((got - ref).abs().max())
    print(f"  n={n_samples} hop={hop} chunk={chunk}: {T} frames, {len(pieces)} pieces, max-abs err {err:.3e}")
    assert err <= 1e-6


def test_window_length_covers_every_grid_phase():
    from zeggs_b200.streaming import WindowRule
    for hop in (200, 160):
        rule = WindowRule(hop=hop)
        for rows in (2, 8, 31):
            W = rule.window_samples(rows)
            for nf in range(0, 300):
                w = rule.plan(10 ** 7, nf, False, W)
                assert w is not None and w.r1 - w.r0 >= rows and w.k0 + w.r0 == nf


def test_lookahead():
    """Frame k needs mel frame floor((k + 15) * fpa) + 1 in full: 15 frames of the k31 convolution plus one hop and half an FFT."""
    from zeggs_b200.streaming import WindowRule
    assert WindowRule(hop=200).lookahead_samples() == 4600
    assert WindowRule(hop=200).lookahead_seconds() == 0.2875
    assert WindowRule(hop=160).lookahead_samples() == 4560
