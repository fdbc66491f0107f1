"""Streaming inference on the GPU: the resumable decoder window (zeggs_decoder_window_fwd_state) and the multi-session chunked
generator (zeggs_b200.streaming.StreamingGenerator).

Tolerances, per pose channel group, relative to max(1, max|ref|):
  fp32 engine chunked vs fp32 one-shot window         1e-5
  tc engine chunked vs the oracle's whole window       1e-2  (the tc-vs-oracle window bound)
  h_final vs the oracle's last state                   1e-4 fp32, 2e-2 tc
  streamed vs generate_motion per clip                 1e-4 fp32, 2e-2 tc (the T = 3600 drift bound)
"""
import numpy as np
import pytest
import torch

from tests._util import NAMES, ensure_built, make_decoder, report, stats_tensors, tt

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    ensure_built()
    return torch.device("cuda:0")


@pytest.fixture
def engine():
    from zeggs_b200 import ops
    yield ops.set_decoder_engine
    ops.set_decoder_engine("fp32")


def _st4(st, dev):
    return tuple(st[k].to(dev) for k in ("anim_input_mean", "anim_input_std", "anim_output_mean", "anim_output_std"))


def _groups(out, ref, tol, what):
    for n, o, r in zip(NAMES, out, ref):
        assert tuple(o.shape) == tuple(r.shape), n
        err, sc = report(f"{what} {n}", o, r)
        assert err <= tol * max(1.0, sc), n


def _window_case(H, B, T, seed):
    from zeggs_b200 import synth
    P = synth.make_params(H=H, seed=seed, with_style=False)
    win = tt(synth.make_pose_windows(B, T, seed=seed))
    rs = np.random.RandomState(seed)
    speech = torch.from_numpy((rs.randn(B, T, 64) * 0.5).astype(np.float32))
    style = torch.from_numpy(rs.randn(B, 1, 64).astype(np.float32)).repeat(1, T, 1)
    return P, win, speech, style


def _chunked(dec, st4, dt, pose0, rp0, rq0, gaze, speech, style, cuts):
    """Frames 0..sum(cuts) as consecutive resumable windows: each starts at the last frame of the previous one."""
    from zeggs_b200 import ops
    Ys, rps, rqs, h, a = [], [], [], None, 0
    pose, rp, rq = pose0, rp0, rq0
    for n in cuts:
        sl = slice(a, a + n + 1)
        Y, p, q, h = ops.decoder_window_forward_state(dec, rp, rq, pose, gaze[:, sl], speech[:, sl], style[:, sl], st4, dt, h_init=h)
        k = 0 if a == 0 else 1
        Ys.append(Y[:, k:]); rps.append(p[:, k:]); rqs.append(q[:, k:])
        pose, rp, rq = Y[:, -1], p[:, -1], q[:, -1]
        a += n
    return ops.split_pose(torch.cat(Ys, 1), torch.cat(rps, 1), torch.cat(rqs, 1)), h


@pytest.mark.parametrize("eng", ["fp32", "tc"])
@pytest.mark.parametrize("H,B", [(512, 7), (1024, 32), (1024, 40)])
def test_continuation_equals_one_shot(dev, engine, eng, H, B):
    from oracle import model_oracle as mo
    from zeggs_b200 import ops
    engine(eng)
    T, cuts = 97, [1, 16, 30, 49]
    st = stats_tensors()
    P, win, speech, style = _window_case(H, B, T, seed=900 + H + B)
    dec = make_decoder(P, H, device=dev)
    st4, dt = _st4(st, dev), st["dt"]
    pose0 = torch.cat([win[n][:, 0].reshape(B, -1) for n in NAMES[2:]], 1).to(dev)
    rp0, rq0, gaze = win["root_pos"][:, 0].to(dev), win["root_rot"][:, 0].to(dev), win["gaze_pos"].to(dev)
    with torch.no_grad():
        got, h = _chunked(dec, st4, dt, pose0, rp0, rq0, gaze, speech.to(dev), style.to(dev), cuts)
        ref, internals = mo.decoder_forward(tt(P), *[win[n][:, 0] for n in NAMES], win["gaze_pos"], speech, style,
                                            st["anim_input_mean"], st["anim_input_std"], st["anim_output_mean"],
                                            st["anim_output_std"], dt, return_internals=True)
        if eng == "fp32":
            Y, rp, rq = dec.forward_packed(rp0, rq0, pose0, gaze, speech.to(dev), style.to(dev), *st4, dt)
            _groups(got, ops.split_pose(Y, rp, rq), 1e-5, f"chunked vs one-shot fp32 H{H} B{B}")
        _groups(got, ref, 2e-4 if eng == "fp32" else 1e-2, f"chunked {eng} vs oracle H{H} B{B}")
    err, sc = report(f"h_final {eng} H{H} B{B}", h, internals["states"][-1])
    assert err <= (1e-4 if eng == "fp32" else 2e-2) * max(1.0, sc)


@pytest.mark.parametrize("eng", ["fp32", "tc"])
def test_state_entry_without_carry_is_the_plain_window(dev, engine, eng):
    """s = NULL and init_from_state all 0 are bit-identical to zeggs_decoder_window_fwd; in a mixed call the samples that start
    from the CellStateEncoder are bit-identical to the plain call; save_for_backward = 1 is refused."""
    from zeggs_b200 import _lib, ops
    engine(eng)
    H, B, T = 512, 9, 23
    st = stats_tensors()
    P, win, speech, style = _window_case(H, B, T, seed=31)
    dec = make_decoder(P, H, device=dev)
    st4, dt = _st4(st, dev), st["dt"]
    pose0 = torch.cat([win[n][:, 0].reshape(B, -1) for n in NAMES[2:]], 1).to(dev)
    args = (dec, win["root_pos"][:, 0].to(dev), win["root_rot"][:, 0].to(dev), pose0, win["gaze_pos"].to(dev), speech.to(dev),
            style.to(dev), st4, dt)
    l = _lib.lib()
    with torch.no_grad():
        plain = [t.clone() for t in ops.decoder_window_forward(*args)[:3]]
        Y, rp, rq, (a, keep, ws) = ops.decoder_window_forward(*args)
        Y.fill_(float("nan"))
        _lib.check(l.zeggs_decoder_window_fwd_state(a, None, _lib.stream_ptr()), "state entry, s = NULL")
        assert all(torch.equal(x, y) for x, y in zip((Y, rp, rq), plain))
        a.save_for_backward = 1
        assert l.zeggs_decoder_window_fwd_state(a, _lib.DecoderStateArgs(), _lib.stream_ptr()) != 0
        h = torch.randn(2, B, H, device=dev)
        got = ops.decoder_window_forward_state(*args, h_init=h, init_from_state=torch.zeros(B, dtype=torch.int32))
        assert all(torch.equal(x, y) for x, y in zip(got[:3], plain))
        flags = torch.tensor([b % 2 for b in range(B)], dtype=torch.int32)
        mixed = ops.decoder_window_forward_state(*args, h_init=h, init_from_state=flags)
        fresh = flags == 0
        assert all(torch.equal(x[fresh.to(dev)], y[fresh.to(dev)]) for x, y in zip(mixed[:3], plain))
        assert not torch.equal(mixed[0][~fresh.to(dev)], plain[0][~fresh.to(dev)])
        one = ops.decoder_window_forward_state(args[0], *[t[:, :1] if t.dim() == 3 else t for t in args[1:4]],
                                               args[4][:, :1], args[5][:, :1], args[6][:, :1], st4, dt, h_init=h)
        assert torch.equal(one[3], h)                                   # T == 1: h_final is the initial state


# ---------------------------------------------------------------------------------------------- the generator
def _nets(P, H, dev):
    from zeggs_b200 import modules

    def load(m, prefix):
        m.load_state_dict({k[len(prefix):]: torch.from_numpy(v) for k, v in P.items() if k.startswith(prefix)})
        return m.to(dev).eval()
    return dict(speech_encoder=load(modules.SpeechEncoder(81, 64, 64), "speech_encoder."),
                style_encoder=load(modules.StyleEncoder(1134, 512, 64, type="attn", use_vae=True), "style_encoder."),
                decoder=load(modules.Decoder(1134, 1131, 64, 64, H, 2), "decoder."))


def _clips(seconds, seed):
    from zeggs_b200 import synth
    return [synth.make_waveforms(1, int(round(16000 * s)), seed=seed + i)[0] for i, s in enumerate(seconds)]


def _drive(gen, sids, clips, seed):
    """Push every clip in seeded random pieces, round-robin, stepping after each round; then close.  sids[i] is the session of
    clips[i], or None for a clip whose pieces are drawn but not pushed (same piece sizes for the others).  -> {sid: 8-tuple}."""
    rs = np.random.RandomState(seed)
    pos = [0] * len(clips)
    outs = {sid: [] for sid in sids if sid is not None}
    while any(p < len(c) for p, c in zip(pos, clips)):
        for i, c in enumerate(clips):
            n = int(rs.randint(50, 4000))
            if pos[i] < len(c):
                if sids[i] is not None:
                    gen.push(sids[i], c[pos[i]:pos[i] + n])
                pos[i] += n
        for sid, o in gen.step().items():
            outs[sid].append(o)
    for sid in outs:
        outs[sid].append(gen.close(sid))
    return {sid: tuple(torch.cat([o[k] for o in outs[sid]], 1) for k in range(8)) for sid in outs}


def _setup(H, seed, dev):
    from zeggs_b200 import synth
    P = synth.make_params(H=H, seed=seed)
    st = synth.load_stats()
    ex = synth.make_style_example(1, 120, seed=seed)[0]
    win = synth.make_pose_windows(1, 2, seed=seed)
    fp = {k: win[k][0, 0] for k in NAMES}
    return _nets(P, H, dev), st, ex, fp, win["gaze_pos"][0, 0]


@pytest.mark.parametrize("eng", ["fp32", "tc"])
def test_streamed_sessions_equal_generate_motion(dev, engine, eng):
    from oracle.make_golden import audio_params
    from zeggs_b200 import generate, streaming
    engine(eng)
    nets, st, ex, fp, g0 = _setup(512, 71, dev)
    dt = float(st["dt"])
    clips = _clips([0.05, 1.0, 2.37, 3.0, 4.1], seed=40)
    pcm = [np.round(c * 20000.0).astype(np.int16) if i == 2 else c for i, c in enumerate(clips)]   # session 2 streams int16
    ref = []
    for i, c in enumerate(clips):
        x = pcm[i].astype(np.float32) / 32768.0 if i == 2 else c
        out, _ = generate.generate_motion(nets, st, audio_params(200), x, ex, fp, g0, dt, eps=torch.zeros(1, 64, device=dev), device=dev)
        ref.append(out)
    tol = 1e-4 if eng == "fp32" else 2e-2
    for chunk in (1, 15, 30):
        gen = streaming.StreamingGenerator(nets, st, audio_params(200), chunk_frames=chunk, device=dev)
        sids = [gen.open(ex, fp, g0, dt, eps=torch.zeros(1, 64, device=dev)) for _ in clips]
        got = _drive(gen, sids, pcm, seed=chunk)
        for i, sid in enumerate(sids):
            assert got[sid][0].shape[1] == ref[i][0].shape[1] == int(round(60 * len(clips[i]) / 16000))
            _groups(got[sid], ref[i], tol, f"stream[{eng}] chunk {chunk} clip {i}")


@pytest.mark.parametrize("eng", ["fp32", "tc"])
def test_session_is_independent_of_the_batch(dev, engine, eng):
    """A session's frames are bit-identical whether it is stepped alone or in a batch of 40."""
    from oracle.make_golden import audio_params
    from zeggs_b200 import streaming
    engine(eng)
    nets, st, ex, fp, g0 = _setup(512, 72, dev)
    dt = float(st["dt"])
    rs = np.random.RandomState(5)
    clips = _clips(list(rs.uniform(0.6, 2.0, 40)), seed=100)
    runs = []
    for batch in (False, True):
        gen = streaming.StreamingGenerator(nets, st, audio_params(200), chunk_frames=15, device=dev)
        sids = [gen.open(ex, fp, g0, dt, eps=torch.zeros(1, 64, device=dev)) if batch or i == 0 else None for i in range(len(clips))]
        runs.append(_drive(gen, sids, clips, seed=9)[sids[0]])
    for k, (a, b) in enumerate(zip(*runs)):
        assert torch.equal(a, b), NAMES[k]


def test_loudness(dev):
    """normalize_loudness without a fixed gain cannot stream; with a fixed gain the stream matches the whole clip's features
    (MelFrontEnd.forward(..., gain=)) through the SpeechEncoder and the decoder."""
    from oracle.make_golden import audio_params
    from zeggs_b200 import _lib, audio, streaming
    nets, st, ex, fp, g0 = _setup(64, 73, dev)
    dt = float(st["dt"])
    conf = audio_params(200)
    conf.normalize_loudness = True
    gen = streaming.StreamingGenerator(nets, st, conf, chunk_frames=15, device=dev)
    with pytest.raises(_lib.ZeggsError, match="normalize_loudness"):
        gen.open(ex, fp, g0, dt)
    gain = 1.7
    x = _clips([2.5], seed=7)[0]
    sid = gen.open(ex, fp, g0, dt, eps=torch.zeros(1, 64, device=dev), gain=gain)
    got = _drive(gen, [sid], [x], seed=3)[sid]
    f = lambda k: torch.as_tensor(st[k], dtype=torch.float32, device=dev)
    T = int(round(60 * len(x) / 16000))
    with torch.no_grad():
        _, feat = audio.MelFrontEnd(dev).forward(torch.from_numpy(x).to(dev), 60, T, gain=torch.tensor([gain], device=dev))
        sp = nets["speech_encoder"]((feat - f("audio_input_mean")) / f("audio_input_std"))
        ex_n = (torch.as_tensor(ex, device=dev)[None] - f("anim_input_mean")) / f("anim_input_std")
        z, _, _ = nets["style_encoder"](ex_n, 1.0, eps=torch.zeros(1, 64, device=dev))
        t = lambda k: torch.as_tensor(fp[k], dtype=torch.float32, device=dev)[None]
        ref = nets["decoder"](*[t(k) for k in NAMES], torch.as_tensor(g0, device=dev).reshape(1, 1, 3).repeat(1, T, 1), sp,
                              z[:, None].repeat(1, T, 1), None, *_st4({k: f(k) for k in st if k.startswith("anim")}, dev), dt)
    _groups(got, ref, 1e-4, "stream with fixed gain")
