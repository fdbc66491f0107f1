"""Streaming gesture generation: poses while the speaker is still talking, for many live sessions at once.

The decoder is causal in speech; the audio features are not.  The SpeechEncoder's k31 replicate-padded convolution looks
SPEECH_RF frames ahead, and the mel front end reflects at the clip edges and resamples 80 -> 60 fps.  So the features of a
stream are recomputed over a sliding sample window with the existing kernels (zeggs_mel_forward, zeggs_speech_enc_fwd), and
only the rows that depend on neither edge of the window are kept (WindowRule).  The decoder carries its GRU state from one
chunk to the next through zeggs_decoder_window_fwd_state; every session of a step shares one mel call, one SpeechEncoder call
and one decoder call per 32-session tile.

Loudness normalisation measures the whole clip (BS.1770 integrated loudness), so it cannot run on a stream: a caller that
wants it passes a fixed gain.
"""
import math
from collections import namedtuple

import numpy as np
import torch

from . import _lib, audio, ops
from .generate import POSE_KEYS
from .modules import P_IN

SPEECH_RF = 15          # SpeechEncoder layer1: kernel 31, padding 'same' -> 15 frames of context on each side

Window = namedtuple("Window", "s0 s1 anim_length r0 r1 k0")
Window.__doc__ = """Feature window of a stream: samples [s0, s1) are featurised as one clip of `anim_length` 60 fps frames; local
rows [r0, r1) are the kept ones, equal to global frames [k0 + r0, k0 + r1) of the whole-clip features."""


class WindowRule:
    """Index arithmetic of the sliding feature window (pure host code).

    - Windows start on multiples of `grid` = lcm(samples per whole number of frames, hop) samples (800 at 16 kHz / 60 fps,
      hop 200 or 160), so the window's local 60 fps and mel frame grids coincide with the global ones.
    - A window that does not start at sample 0 keeps no row whose receptive field reaches its left edge: the first `left`
      local frames touch mel frames that see the reflect padding (one mel frame of margin covers the floor of the
      resampler's double-precision position), the next SPEECH_RF frames see them through the k31 convolution.
    - A window that does not end at the end of the stream keeps no row whose receptive field reaches a mel frame that
      sees the right reflect padding or the L-2 clamp of the resampler.
    - The final window (close of the stream) ends at the true end: its frame count is the offline one, round(60 N / fs).
    """

    def __init__(self, fs=16000, hop=200, n_fft=800, anim_fs=60):
        self.fs, self.hop, self.n_fft, self.anim_fs = int(fs), int(hop), int(n_fft), int(anim_fs)
        per = self.fs // math.gcd(self.fs, self.anim_fs)
        self.grid = per * self.hop // math.gcd(per, self.hop)
        self.grid_frames = self.grid * self.anim_fs // self.fs
        half_frames = -(-(self.n_fft // 2) // self.hop)
        self.left = next(j for j in range(1 << 20) if self._mel(j) - 1 >= half_frames)

    def _mel(self, j):
        """Lower mel frame of the linear resample at 60 fps frame j: floor(j * fs / hop / anim_fs), exact."""
        return (j * self.fs) // (self.hop * self.anim_fs)

    def mel_num_frames(self, n):
        """zeggs_mel_num_frames for n >= n_fft (centered STFT)."""
        m = n + 2 * (self.n_fft // 2)
        return (m - self.n_fft) // self.hop + (1 if m % self.hop else 0)

    def total_frames(self, n_samples):
        """Frame count of the offline path for a clip of n_samples (generate_motion)."""
        return int(round(self.anim_fs * (n_samples / self.fs)))

    def start(self, next_frame):
        """First sample of the window whose first kept row is global frame next_frame."""
        return self.grid * max(0, (next_frame - SPEECH_RF - self.left) // self.grid_frames)

    def plan(self, received, next_frame, final, n_window=None):
        """(samples received, next frame, final) -> Window, or None when no row from next_frame on can be computed yet.
        Non-final windows end at `received`, or span exactly n_window samples (None if the stream has not reached that)."""
        s0 = self.start(next_frame)
        k0 = s0 * self.anim_fs // self.fs
        r0 = next_frame - k0
        if final:
            s1 = received
            T = self.total_frames(received) - k0
            r1 = T
        else:
            s1 = received if n_window is None else s0 + n_window
            if s1 > received or s1 - s0 < self.n_fft:
                return None
            n = s1 - s0
            i_r = min(self.mel_num_frames(n) - 1, (n - self.n_fft // 2) // self.hop)   # last mel frame clear of the right edge
            T = (i_r * self.hop * self.anim_fs - 1) // self.fs + 1                       # frames j with _mel(j) + 1 <= i_r
            r1 = T - SPEECH_RF
        if r1 <= r0:
            return None
        return Window(s0, s1, T, r0, r1, k0)

    def window_samples(self, rows):
        """Window length that yields `rows` kept rows from any next_frame (the worst grid phase)."""
        r0 = SPEECH_RF + self.left + self.grid_frames - 1
        return (self._mel(r0 + rows - 1 + SPEECH_RF) + 1) * self.hop + self.n_fft // 2

    def lookahead_samples(self):
        """Algorithmic lookahead: the most audio past frame k's timestamp (k fs / anim_fs) that frame k's features need."""
        from fractions import Fraction
        need = lambda k: (self._mel(k + SPEECH_RF) + 1) * self.hop + self.n_fft // 2 - Fraction(k * self.fs, self.anim_fs)
        return max(need(self.grid_frames * 64 + k) for k in range(self.grid_frames))

    def lookahead_seconds(self):
        return float(self.lookahead_samples() / self.fs)


class _Session:
    def __init__(self, sid, slot, dt):
        self.sid, self.slot, self.dt = sid, slot, float(dt)
        self.buf = np.zeros(0, np.float32)     # samples [base, received)
        self.base = 0
        self.received = 0
        self.frames_out = 0


def _pcm_to_f32(samples):
    x = np.asarray(samples)
    if x.dtype == np.int16:
        return x.astype(np.float32) / np.float32(32768.0)      # audio_files.py:211-236; exact (power-of-two scale)
    return x.astype(np.float32, copy=False)


class StreamingGenerator:
    """Multi-session chunked generator.

        gen = StreamingGenerator(nets, stats, audio_conf, chunk_frames=30)
        sid = gen.open(style, first_pose, gaze_pos0, dt)     # style: raw example [T_ex,1134] or an embedding [Z]
        gen.push(sid, samples)                               # float32 or int16 @ fs, any length
        out = gen.step()                                     # {sid: 8-tuple [1, n, ...]} per session with a full chunk
        tail = gen.close(sid)                                # the remaining frames, end-of-clip semantics; frees the slot

    A session's first chunk starts with frame 0 (the first pose), so it holds chunk_frames + 1 frames; later chunks hold
    chunk_frames.  All chunks and the close tail together are generate_motion's frames for the same audio."""

    def __init__(self, nets, stats, audio_conf, chunk_frames=30, device="cuda"):
        if chunk_frames < 1:
            raise _lib.ZeggsError("chunk_frames must be >= 1")
        self.dev = torch.device(device)
        self.nets = nets
        self.chunk = int(chunk_frames)
        f = lambda k: torch.as_tensor(stats[k], dtype=torch.float32, device=self.dev)
        self.audio_mean, self.audio_std = f("audio_input_mean"), f("audio_input_std")
        self.anim_in = (f("anim_input_mean"), f("anim_input_std"))
        self.stats = (f("anim_input_mean"), f("anim_input_std"), f("anim_output_mean"), f("anim_output_std"))
        kw = audio._conf_kwargs(audio_conf)
        get = (lambda k: audio_conf.get(k, False)) if isinstance(audio_conf, dict) else (lambda k: getattr(audio_conf, k, False))
        self.normalize_loudness = bool(get("normalize_loudness"))
        self.fe = audio._front_end(self.dev, **kw)
        self.rule = WindowRule(kw["sampling_rate"], kw["hop_length"], kw["filter_length"], 60)
        # every step's decoder window is chunk + 1 frames: the last frame already emitted (or the first pose), then the chunk
        self.n_window = self.rule.window_samples(self.chunk + 1)
        self.window_frames = self.rule.plan(self.n_window, 0, False, self.n_window).anim_length
        dec = nets["decoder"]
        self.H, self.S, self.Z = dec.hidden_size, dec.speech_encoding_size, dec.style_encoding_size
        self.sessions = {}
        self._next_sid = 0
        self._free = []
        self._cap = 0
        self._h = torch.zeros((2, 0, self.H), device=self.dev)                    # per slot: GRU state after the last frame
        self._pose = torch.zeros((0, ops.P_OUT), device=self.dev)                 # pose vector, root position / rotation of it
        self._rp = torch.zeros((0, 3), device=self.dev)
        self._rq = torch.zeros((0, 4), device=self.dev)
        self._z = torch.zeros((0, self.Z), device=self.dev)                       # style encoding
        self._gaze = torch.zeros((0, 3), device=self.dev)                         # constant gaze target (generate.py:374-376)
        self._gain = torch.ones(0, device=self.dev)

    # ------------------------------------------------------------------------------------------ sessions
    @property
    def lookahead_seconds(self):
        return self.rule.lookahead_seconds()

    @property
    def recompute_factor(self):
        """Feature frames computed per emitted frame: (context + chunk) / chunk."""
        return self.window_frames / self.chunk

    def _slot(self):
        if self._free:
            return self._free.pop()
        slot = self._cap
        grow = max(8, self._cap)
        z = lambda t, *shape: torch.cat([t, torch.zeros(shape, dtype=t.dtype, device=self.dev)], dim=0)
        self._h = torch.cat([self._h, torch.zeros((2, grow, self.H), device=self.dev)], dim=1)
        self._pose, self._rp, self._rq = z(self._pose, grow, ops.P_OUT), z(self._rp, grow, 3), z(self._rq, grow, 4)
        self._z, self._gaze = z(self._z, grow, self.Z), z(self._gaze, grow, 3)
        self._gain = torch.cat([self._gain, torch.ones(grow, device=self.dev)])
        self._cap += grow
        self._free = list(range(self._cap - 1, slot, -1))
        return slot

    @torch.no_grad()
    def open(self, style, first_pose, gaze_pos0, dt, temperature=1.0, eps=None, gain=None):
        """Start a session -> its id.  style: raw example [T_ex,1134] (encoded here once, as generate_motion does) or an
        embedding [Z]; first_pose: dict of the 8 first-frame tensors; gain: fixed factor on every sample (loudness)."""
        if self.normalize_loudness and gain is None:
            raise _lib.ZeggsError("normalize_loudness needs the whole clip (BS.1770 integrated loudness): a stream cannot measure "
                                  "it.  Pass a fixed gain= to open(), or turn normalize_loudness off in the audio configuration")
        style = torch.as_tensor(style, dtype=torch.float32, device=self.dev)
        if style.dim() == 2 and style.shape[-1] == P_IN:
            ex = (style[None] - self.anim_in[0]) / self.anim_in[1]
            z, _, _ = self.nets["style_encoder"](ex, temperature, eps=eps)
        else:
            z = style.reshape(1, -1)
        if z.shape[1] != self.Z:
            raise _lib.ZeggsError(f"style encoding must have {self.Z} values, got {z.shape[1]}")
        fp = {k: torch.as_tensor(first_pose[k], dtype=torch.float32, device=self.dev) for k in POSE_KEYS}
        slot = self._slot()
        self._pose[slot] = torch.cat([fp[k].reshape(-1) for k in POSE_KEYS[2:]])
        self._rp[slot] = fp["root_pos"].reshape(3)
        self._rq[slot] = fp["root_rot"].reshape(4)
        self._z[slot] = z[0]
        self._gaze[slot] = torch.as_tensor(gaze_pos0, dtype=torch.float32, device=self.dev).reshape(3)
        self._gain[slot] = 1.0 if gain is None else float(gain)
        self._h[:, slot] = 0.0
        sid = self._next_sid
        self._next_sid += 1
        self.sessions[sid] = _Session(sid, slot, dt)
        return sid

    def _session(self, sid):
        s = self.sessions.get(sid)
        if s is None:
            raise _lib.ZeggsError(f"no open streaming session {sid}")
        return s

    def push(self, sid, samples):
        """Append audio (float32, or int16 PCM decoded as x / 32768) to a session."""
        s = self._session(sid)
        x = _pcm_to_f32(samples).reshape(-1)
        s.buf = np.concatenate([s.buf, x])
        s.received += x.size

    def _window(self, s, final):
        a = max(s.frames_out - 1, 0)                       # the decoder window starts at the last emitted frame
        return self.rule.plan(s.received, a, final, None if final else self.n_window)

    # ------------------------------------------------------------------------------------------ compute
    # Rows are independent in every kernel on the path, but the GEMM front end picks its algorithm from the product's size
    # (fp32 SIMT below 4e6 multiply-adds, tcgen05 split-bf16 above, split-K by tile count).  The SpeechEncoder and the
    # CellStateEncoder multiply over the batch rows, so their calls run on tiles padded to TILE sessions: a session's frames are
    # then bit-identical whether it is stepped alone or with others.
    TILE = 32

    def _pad(self, t, dim=0):
        m = t.shape[dim]
        if m == self.TILE:
            return t
        rep = t.narrow(dim, 0, 1).expand(*[self.TILE - m if d == dim else -1 for d in range(t.dim())])
        return torch.cat([t, rep], dim)

    def _run(self, sess, wins, wav, rows):
        """Sessions with equal-length windows wav [n, samples] (one mel call) -> {session: 8-tuple}; one SpeechEncoder call and
        one decoder window per tile of sessions with the same dt.  The decoder window of a session runs from its last emitted
        frame (or the first pose) over `rows` kept rows."""
        slots = torch.tensor([s.slot for s in sess], device=self.dev)
        _, feat = self.fe.forward(wav, 60, wins[0].anim_length, want_mel=False, want_feat=True, gain=self._gain[slots])
        x = (feat - self.audio_mean) / self.audio_std
        out = {}
        for dt in sorted({s.dt for s in sess}):                     # dt is a scalar of the decoder call
            pick = [i for i, s in enumerate(sess) if s.dt == dt]
            for t0 in range(0, len(pick), self.TILE):
                tile = pick[t0:t0 + self.TILE]
                sp = self.nets["speech_encoder"](self._pad(x[tile]))[:len(tile)]
                idx = torch.tensor([wins[i].r0 for i in tile], device=self.dev)[:, None] + torch.arange(rows, device=self.dev)
                out.update(self._decode([sess[i] for i in tile], sp[torch.arange(len(tile), device=self.dev)[:, None], idx]))
        return out

    def _decode(self, sess, speech):
        m, T = speech.shape[0], speech.shape[1]
        slots = torch.tensor([s.slot for s in sess], device=self.dev)
        carry = torch.tensor([1 if s.frames_out > 0 else 0 for s in sess], dtype=torch.int32, device=self.dev)
        p = self._pad
        Y, rp, rq, hf = ops.decoder_window_forward_state(
            self.nets["decoder"], p(self._rp[slots]), p(self._rq[slots]), p(self._pose[slots]),
            p(self._gaze[slots])[:, None].expand(self.TILE, T, 3), p(speech), p(self._z[slots])[:, None].expand(self.TILE, T, self.Z),
            self.stats, sess[0].dt, h_init=p(self._h[:, slots], 1), init_from_state=p(carry))
        self._h[:, slots] = hf[:, :m]
        self._pose[slots], self._rp[slots], self._rq[slots] = Y[:m, -1], rp[:m, -1], rq[:m, -1]
        out = {}
        for i, s in enumerate(sess):
            first = 0 if s.frames_out == 0 else 1
            out[s] = ops.split_pose(Y[i:i + 1, first:], rp[i:i + 1, first:], rq[i:i + 1, first:])
            s.frames_out += T - first
        return out

    def _trim(self, s):
        keep = self.rule.start(max(s.frames_out - 1, 0))
        if keep > s.base:
            s.buf = s.buf[keep - s.base:]
            s.base = keep

    @torch.no_grad()
    def step(self):
        """Advance every session that has a full chunk of final frames -> {sid: 8-tuple [1, n, ...]}."""
        ready = [(s, w) for s in self.sessions.values() for w in [self._window(s, False)] if w is not None]
        if not ready:
            return {}
        wav = np.stack([s.buf[w.s0 - s.base:w.s1 - s.base] for s, w in ready])
        wav = torch.from_numpy(wav).pin_memory().to(self.dev, non_blocking=True)
        out = self._run([s for s, _ in ready], [w for _, w in ready], wav, self.chunk + 1)
        for s, _ in ready:
            self._trim(s)
        return {s.sid: o for s, o in out.items()}

    @torch.no_grad()
    def close(self, sid):
        """End of the stream: the remaining frames with the offline path's end-of-clip semantics; frees the session's slot."""
        s = self._session(sid)
        w = self._window(s, True)
        if w is not None:
            wav = torch.from_numpy(np.ascontiguousarray(s.buf[w.s0 - s.base:w.s1 - s.base])[None]).to(self.dev)
            out = self._run([s], [w], wav, w.r1 - w.r0)[s]
        else:
            z = lambda c: torch.zeros((1, 0, c), device=self.dev)
            out = ops.split_pose(z(ops.P_OUT), z(3), z(4))
        del self.sessions[sid]
        self._free.append(s.slot)
        return out
