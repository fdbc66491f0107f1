"""Launchers: torch tensors -> C-ABI calls (libzeggs_b200.so).  Plumbing only (buffers, streams,
autograd wiring); all arithmetic is in csrc/*.cu."""
import ctypes as C

import torch

from . import _lib

NJ, P_IN, P_OUT = 75, 1134, 1131


def _f32c(t, device=None):
    t = t.detach() if t.requires_grad else t
    if device is not None and t.device != device:
        t = t.to(device)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class _Workspace:
    """Grow-only per-device scratch buffers owned by the caller side (the library allocates nothing)."""

    def __init__(self):
        self.bufs = {}

    def get(self, key, nbytes, device):
        b = self.bufs.get((key, str(device)))
        if b is None or b.numel() < nbytes:
            b = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
            self.bufs[(key, str(device))] = b
        return b


WS = _Workspace()

_scratch = {}
_ctx = {}
GEMM_MODE = 1          # 0: fp32 SIMT everywhere, 1: tcgen05 split-bf16 (~fp32 accuracy), 2: tcgen05 plain bf16
# experiment knob: with the tensor-core recurrence engine selected, run the batched GEMMs (encoders, hoisted terms, fold matrix) as ONE
# bf16 pass instead of the 3-pass split-bf16 scheme
TC_GEMM_BF16 = __import__("os").environ.get("ZEGGS_TC_GEMM_BF16", "0") == "1"


def _effective_gemm_mode():
    return 2 if (TC_GEMM_BF16 and GEMM_MODE == 1 and DECODER_ENGINE != "fp32") else GEMM_MODE


def set_gemm_mode(mode):
    """GEMM engine of the batched (non-recurrent) products for subsequent calls from this process."""
    global GEMM_MODE
    if mode not in (0, 1, 2):
        raise _lib.ZeggsError("gemm mode must be 0 (fp32 SIMT), 1 (tcgen05 bf16x3) or 2 (tcgen05 bf16)")
    GEMM_MODE = mode
    for c in _ctx.values():
        c.gemm_mode = _effective_gemm_mode()


# Lanes: calls that run CONCURRENTLY on different CUDA streams (the two encoders next to each other, the encoders' backward next to the
# decoder's weight-gradient GEMMs) must not share the GEMM front end's scratch buffer.  `with ops.lane("speech"):` makes every call issued
# inside the block travel with that lane's own zeggs_ctx (own scratch); the default lane is "main".
_lane_local = __import__("threading").local()


def current_lane():
    return getattr(_lane_local, "name", "main")


class lane:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        self.prev = current_lane()
        _lane_local.name = self.name
        return self

    def __exit__(self, *exc):
        _lane_local.name = self.prev
        return False


def ensure_scratch(dev):
    """Caller-owned scratch for the tcgen05 GEMM front end (bf16 operand copies); ZEGGS_SCRATCH_MB (main lane) / ZEGGS_LANE_SCRATCH_MB
    (side lanes) override the size.  The buffer, the GEMM mode and the weight-gradient mode travel to the library in a per-(device, lane)
    zeggs_ctx passed with every call (ctx_ptr): the library keeps no mutable global state for them."""
    import os
    ln = current_lane()
    key = (str(dev), ln)
    if key not in _scratch:
        mb = int(os.environ.get("ZEGGS_SCRATCH_MB", "1536")) if ln == "main" else int(os.environ.get("ZEGGS_LANE_SCRATCH_MB", "768"))
        buf = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
        _scratch[key] = buf
        _ctx[key] = _lib.Ctx(scratch=buf.data_ptr(), scratch_bytes=buf.numel(), gemm_mode=_effective_gemm_mode(),
                             fast_wgrad=0 if DECODER_ENGINE == "fp32" else 1)
    return _scratch[key]


def ctx_ptr(dev):
    """Address of the current lane's zeggs_ctx on this device (for the `ctx` field of the args structs)."""
    ensure_scratch(dev)
    return C.addressof(_ctx[(str(dev), current_lane())])


_weights_epoch = 0

# decoder recurrence engine: "fp32" (SIMT, parity grade), "tc" (tcgen05, bf16 operands / fp32 state) or "auto" (tc where the
# geometry is eligible, fp32 otherwise).  An explicit "tc" request on an ineligible geometry RAISES (it never silently
# runs the other engine).
DECODER_ENGINE = __import__("os").environ.get("ZEGGS_DECODER_ENGINE", "fp32")
TC_MIN_HIDDEN = 288


def tc_eligible(H, S, Z):
    """The tensor-core recurrence (forward AND BPTT kernels) covers H % 128 == 0, 384 <= H <= 1024: the library's
    zeggs_decoder_packed_tc_bytes / _bwd_tc_bytes report 0 for anything else."""
    l = _lib.lib()
    return H >= TC_MIN_HIDDEN and l.zeggs_decoder_packed_tc_bytes(H, S, Z) > 0 and l.zeggs_decoder_packed_bwd_tc_bytes(H, S, Z) > 0


def set_decoder_engine(name):
    global DECODER_ENGINE
    if name not in ("fp32", "tc", "auto"):
        raise _lib.ZeggsError("decoder engine must be 'fp32', 'tc' or 'auto'")
    DECODER_ENGINE = name
    # the tensor-core engine's weight gradients are single-pass bf16: the encoders' weight-gradient GEMMs follow it
    for c in _ctx.values():
        c.fast_wgrad = 0 if name == "fp32" else 1
        c.gemm_mode = _effective_gemm_mode()


def resolve_engine(H, S, Z):
    """-> True when the tensor-core engine runs this geometry under the current setting."""
    if DECODER_ENGINE == "fp32":
        return False
    ok = tc_eligible(H, S, Z)
    if DECODER_ENGINE == "tc" and not ok:
        raise _lib.ZeggsError(f"decoder engine 'tc' requested but hidden size {H} is not eligible (needs H % 128 == 0 and "
                              f"384 <= H <= 1024); use 'fp32' or 'auto'")
    return ok


def bump_weights_epoch():
    """Called by anything that rewrites parameters without going through torch (the fused optimizer)."""
    global _weights_epoch
    _weights_epoch += 1


def weights_key(params):
    return (_weights_epoch,) + tuple(p._version for p in params) + tuple(p.data_ptr() for p in params)


def normalize_rows(x, mean, std):
    """(x - mean) / std over the last dimension in one pass (zeggs_normalize_rows); same arithmetic as the two torch ops."""
    if x.device.type != "cuda":
        raise _lib.ZeggsError("zeggs_b200.ops.normalize_rows runs on CUDA tensors only")
    x = _f32c(x)
    Cn = x.shape[-1]
    try:                                    # statistics broadcast over the channel dimension (the audio std is a scalar)
        mean = _f32c(mean, x.device).reshape(-1).expand(Cn).contiguous() if mean.numel() in (1, Cn) else None
        std = _f32c(std, x.device).reshape(-1).expand(Cn).contiguous() if std.numel() in (1, Cn) else None
    except RuntimeError:
        mean = std = None
    if mean is None or std is None:
        raise _lib.ZeggsError("normalize_rows: mean / std must be scalars or have the size of the last dimension")
    out = torch.empty_like(x)
    _lib.check(_lib.lib().zeggs_normalize_rows(x.data_ptr(), mean.data_ptr(), std.data_ptr(), out.data_ptr(), x.numel() // Cn, Cn,
                                               _lib.stream_ptr()), "zeggs_normalize_rows")
    return out


def split_pose(Y, root_pos, root_rot):
    """[B,T,1131] pose vectors -> the reference's 8-tuple (modules.py:153-162, 731-736)."""
    B, T = Y.shape[0], Y.shape[1]
    o = 6
    return (root_pos, root_rot, Y[..., 0:3], Y[..., 3:6],
            Y[..., o:o + NJ * 3].reshape(B, T, NJ, 3),
            Y[..., o + NJ * 3:o + NJ * 9].reshape(B, T, NJ, 2, 3),
            Y[..., o + NJ * 9:o + NJ * 12].reshape(B, T, NJ, 3),
            Y[..., o + NJ * 12:o + NJ * 15].reshape(B, T, NJ, 3))


def _decoder_args(dec, B, T, dev, tensors, stats, dt, save, pack_only=False):
    """Fill a DecoderFwdArgs; returns (args, keepalive list).  pack_only: stop after the weight packs (decoder_prepack)."""
    H, S, Z = dec.hidden_size, dec.speech_encoding_size, dec.style_encoding_size
    l = _lib.lib()
    w = [_f32c(p, dev) for p in dec._weights()]
    names = ["W0", "b0", "W_ih0", "b_ih0", "W_hh0", "b_hh0", "W_ih1", "b_ih1", "W_hh1", "b_hh1", "W2", "b2",
             "Wc0", "bc0", "Wc1", "bc1", "Wc2", "bc2"]
    a = _lib.DecoderFwdArgs(B=B, T=T, H=H, S=S, Z=Z, dt=dt, ctx=ctx_ptr(dev))
    for n, t in zip(names, w):
        setattr(a, n, _lib.ptr(t))
    keep = list(w)
    st = [_f32c(s, dev).reshape(-1) for s in stats]
    for n, t in zip(["in_mean", "in_std", "out_mean", "out_std"], st):
        setattr(a, n, _lib.ptr(t))
    keep += st
    for n, t in tensors.items():
        setattr(a, n, _lib.ptr(t))
        keep.append(t)
    # packed weights: re-packed whenever any parameter's version counter moved (each engine packs only its own slices)
    ver = weights_key(dec._weights())
    use_tc = resolve_engine(H, S, Z)
    if use_tc and B > 32:
        raise _lib.ZeggsError("tensor-core decoder engine: one call covers one 32-sample batch tile (decoder_window splits larger batches)")
    if not use_tc:
        cache = getattr(dec, "_zeggs_packed", None)
        if cache is None or cache[0] != ver or cache[1].device != dev:
            nbytes = l.zeggs_decoder_packed_bytes(H, S, Z)
            if nbytes == 0:
                raise _lib.ZeggsError(f"decoder hidden size {H} unsupported")
            packed = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
            _lib.check(l.zeggs_decoder_pack_weights(a, packed.data_ptr(), _lib.stream_ptr()), "zeggs_decoder_pack_weights")
            dec.__dict__["_zeggs_packed"] = (ver, packed)
            cache = dec.__dict__["_zeggs_packed"]
        a.packed = cache[1].data_ptr()
        keep.append(cache[1])
    if use_tc:
        tcc = dec.__dict__.get("_zeggs_packed_tc")
        if tcc is None or tcc[0] != ver or tcc[1].device != dev:
            nb = l.zeggs_decoder_packed_tc_bytes(H, S, Z)
            ptc = torch.empty(nb, dtype=torch.uint8, device=dev)
            _lib.check(l.zeggs_decoder_pack_weights_tc(a, ptc.data_ptr(), _lib.stream_ptr()), "zeggs_decoder_pack_weights_tc")
            dec.__dict__["_zeggs_packed_tc"] = (ver, ptc)
            tcc = dec.__dict__["_zeggs_packed_tc"]
        wtc = WS.get("dec_tc", l.zeggs_decoder_tc_workspace_bytes(H, S, Z), dev)
        a.engine, a.packed_tc, a.workspace_tc = 1, tcc[1].data_ptr(), wtc.data_ptr()
        keep += [tcc[1], wtc]
    if pack_only:
        return a, keep, None
    wsb = l.zeggs_decoder_workspace_bytes(B, T, H, S, Z, int(save))
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev) if save else WS.get("dec_fwd", wsb, dev)
    a.workspace = ws.data_ptr()
    a.workspace_bytes = wsb
    a.save_for_backward = int(save)
    keep.append(ws)
    return a, keep, ws


def decoder_prepack(dec, B, T, dev, stats, dt, backward=True):
    """Everything the decoder derives from its WEIGHTS alone -- the engine's packed / bf16 weight images, the folded layer-2 matrix and
    (backward=True) the transposed images of the BPTT kernel -- issued on the current stream and lane.  The window calls find the caches
    fresh and skip the work, so a training step can run this next to the encoders' forward instead of in front of the recurrence."""
    l = _lib.lib()
    a, keep, _ = _decoder_args(dec, B, T, dev, {}, stats, dt, False, pack_only=True)
    if backward and a.engine == 1:
        _pack_bwd_tc(dec, a, dev)
    return keep


def _pack_bwd_tc(dec, a, dev):
    l = _lib.lib()
    H, S, Z = a.H, a.S, a.Z
    ver = weights_key(dec._weights())
    tcc = dec.__dict__.get("_zeggs_packed_bwd_tc")
    if tcc is None or tcc[0] != ver or tcc[1].device != dev:
        ptc = torch.empty(l.zeggs_decoder_packed_bwd_tc_bytes(H, S, Z), dtype=torch.uint8, device=dev)
        _lib.check(l.zeggs_decoder_pack_weights_bwd_tc(a, ptc.data_ptr(), _lib.stream_ptr()), "zeggs_decoder_pack_weights_bwd_tc")
        dec.__dict__["_zeggs_packed_bwd_tc"] = (ver, ptc)
        tcc = dec.__dict__["_zeggs_packed_bwd_tc"]
    return tcc


def decoder_window_forward(dec, root_pos0, root_rot0, pose0, gaze_pos, speech, style, stats, dt, save=False):
    dev = speech.device
    if dev.type != "cuda":
        raise _lib.ZeggsError("zeggs_b200.Decoder runs on CUDA tensors only (no CPU fallback)")
    ensure_scratch(dev)
    B, T = speech.shape[0], speech.shape[1]
    tensors = dict(root_pos0=_f32c(root_pos0, dev).reshape(B, 3), root_rot0=_f32c(root_rot0, dev).reshape(B, 4),
                   pose0=_f32c(pose0, dev).reshape(B, P_OUT), gaze_pos=_f32c(gaze_pos, dev).reshape(B, T, 3),
                   speech=_f32c(speech, dev), style=_f32c(style, dev))
    if tensors["style"].shape[:2] != (B, T):
        raise _lib.ZeggsError("style_encoding must be [B,T,Z] (modules.py:119)")
    Y = torch.empty((B, T, P_OUT), dtype=torch.float32, device=dev)
    rp = torch.empty((B, T, 3), dtype=torch.float32, device=dev)
    rq = torch.empty((B, T, 4), dtype=torch.float32, device=dev)
    tensors.update(Y=Y, root_pos=rp, root_rot=rq)
    a, keep, ws = _decoder_args(dec, B, T, dev, tensors, stats, dt, save)
    _lib.check(_lib.lib().zeggs_decoder_window_fwd(a, _lib.stream_ptr()), "zeggs_decoder_window_fwd")
    return Y, rp, rq, (a, keep, ws)


def decoder_window_forward_state(dec, root_pos0, root_rot0, pose0, gaze_pos, speech, style, stats, dt, h_init=None,
                                 init_from_state=None):
    """Resumable inference window (zeggs_decoder_window_fwd_state) -> (Y [B,T,1131], root_pos, root_rot, h_final [2,B,H]).
    h_init [2,B,H]: GRU state frame 1 starts from (None: the CellStateEncoder); init_from_state [B] int32: per-sample choice between
    h_init (1) and the CellStateEncoder (0), None = all h_init.  On the tensor-core engine batches above 32 run as 32-sample tiles."""
    dev = speech.device
    if dev.type != "cuda":
        raise _lib.ZeggsError("zeggs_b200.Decoder runs on CUDA tensors only (no CPU fallback)")
    ensure_scratch(dev)
    B, T = speech.shape[0], speech.shape[1]
    if init_from_state is not None and h_init is None:
        raise _lib.ZeggsError("init_from_state needs h_init")
    if B > 32 and resolve_engine(dec.hidden_size, dec.speech_encoding_size, dec.style_encoding_size):
        outs = [decoder_window_forward_state(
            dec, root_pos0[i:i + 32], root_rot0[i:i + 32], pose0[i:i + 32], gaze_pos[i:i + 32], speech[i:i + 32], style[i:i + 32],
            stats, dt, None if h_init is None else h_init[:, i:i + 32],
            None if init_from_state is None else init_from_state[i:i + 32]) for i in range(0, B, 32)]
        Y, rp, rq, hf = zip(*outs)
        return torch.cat(Y, 0), torch.cat(rp, 0), torch.cat(rq, 0), torch.cat(hf, 1)
    H = dec.hidden_size
    tensors = dict(root_pos0=_f32c(root_pos0, dev).reshape(B, 3), root_rot0=_f32c(root_rot0, dev).reshape(B, 4),
                   pose0=_f32c(pose0, dev).reshape(B, P_OUT), gaze_pos=_f32c(gaze_pos, dev).reshape(B, T, 3),
                   speech=_f32c(speech, dev), style=_f32c(style, dev))
    if tensors["style"].shape[:2] != (B, T):
        raise _lib.ZeggsError("style_encoding must be [B,T,Z] (modules.py:119)")
    Y = torch.empty((B, T, P_OUT), dtype=torch.float32, device=dev)
    rp = torch.empty((B, T, 3), dtype=torch.float32, device=dev)
    rq = torch.empty((B, T, 4), dtype=torch.float32, device=dev)
    h_final = torch.empty((2, B, H), dtype=torch.float32, device=dev)
    tensors.update(Y=Y, root_pos=rp, root_rot=rq)
    a, keep, ws = _decoder_args(dec, B, T, dev, tensors, stats, dt, False)
    s = _lib.DecoderStateArgs(h_final=h_final.data_ptr())
    if h_init is not None:
        h_init = _f32c(h_init, dev)
        if tuple(h_init.shape) != (2, B, H):
            raise _lib.ZeggsError(f"h_init must be [2,B,H] = [2,{B},{H}], got {tuple(h_init.shape)}")
        s.h_init = h_init.data_ptr()
    if init_from_state is not None:
        init_from_state = init_from_state.to(device=dev, dtype=torch.int32).contiguous()
        if tuple(init_from_state.shape) != (B,):
            raise _lib.ZeggsError(f"init_from_state must be [B] = [{B}]")
        s.init_from_state = init_from_state.data_ptr()
    _lib.check(_lib.lib().zeggs_decoder_window_fwd_state(a, s, _lib.stream_ptr()), "zeggs_decoder_window_fwd_state")
    return Y, rp, rq, h_final


_DEC_GRAD_NAMES = ["dW0", "db0", "dW_ih0", "db_ih0", "dW_hh0", "db_hh0", "dW_ih1", "db_ih1", "dW_hh1", "db_hh1",
                   "dW2", "db2", "dWc0", "dbc0", "dWc1", "dbc1", "dWc2", "dbc2"]


def _grad_targets(weights, grads_out):
    """Gradient buffers for `weights`: fresh tensors, or the caller's (e.g. the views of the optimizer's flat gradient buffer:
    the kernels then write every parameter gradient straight to its final place -- no autograd accumulation pass)."""
    if grads_out is None:
        return [torch.empty_like(w, dtype=torch.float32, memory_format=torch.contiguous_format) for w in weights]
    for w, g in zip(weights, grads_out):
        if g.shape != w.shape or not g.is_contiguous() or g.dtype != torch.float32:
            raise _lib.ZeggsError("gradient target must be a contiguous fp32 tensor of the parameter's shape")
    return list(grads_out)


def decoder_window_backward(dec, state, dY, dRp, dRq, grads_out=None, split=False):
    """BPTT of one decoder window (zeggs_decoder_window_bwd).  state = the 4th result of decoder_window_forward(save=True).
    Returns (weight gradients in dec._weights() order, dSpeech [B,T,S], dStyle [B,T,Z]).
    split=True: run phase 1 only (recurrence, CellStateEncoder gradients, dSpeech / dStyle) and return a 4th value `finish`;
    calling it issues phase 2 (all remaining parameter gradients) on the then-current stream of the same lane -- the caller may run the
    encoders' backward passes on other streams / lanes in between."""
    l = _lib.lib()
    a, keep, ws = state
    dev = ws.device
    B, T, H, S, Z = a.B, a.T, a.H, a.S, a.Z
    b = _lib.DecoderBwdArgs()
    hold = []
    for name, g in (("dY", dY), ("dRootPos", dRp), ("dRootRot", dRq)):
        if g is not None:
            g = g.contiguous().float()
            hold.append(g)
            setattr(b, name, g.data_ptr())
    # transposed weight slices for the backward recurrence (cached on the module like the forward pack)
    ver = weights_key(dec._weights())
    use_tc = a.engine == 1
    if use_tc and l.zeggs_decoder_packed_bwd_tc_bytes(H, S, Z) == 0:
        raise _lib.ZeggsError(f"tensor-core decoder backward unavailable for hidden size {H}")
    if not use_tc:
        cache = dec.__dict__.get("_zeggs_packed_bwd")
        if cache is None or cache[0] != ver or cache[1].device != dev:
            nb = l.zeggs_decoder_packed_bwd_bytes(H, S, Z)
            packed = torch.empty(nb // 4, dtype=torch.float32, device=dev)
            _lib.check(l.zeggs_decoder_pack_weights_bwd(a, packed.data_ptr(), _lib.stream_ptr()), "zeggs_decoder_pack_weights_bwd")
            dec.__dict__["_zeggs_packed_bwd"] = (ver, packed)
            cache = dec.__dict__["_zeggs_packed_bwd"]
        b.packed_bwd = cache[1].data_ptr()
        hold.append(cache[1])
    else:
        tcc = _pack_bwd_tc(dec, a, dev)
        wtc = WS.get("dec_bwd_tc", l.zeggs_decoder_bwd_tc_workspace_bytes(H, S, Z), dev)
        b.packed_bwd_tc, b.workspace_tc = tcc[1].data_ptr(), wtc.data_ptr()
        hold += [tcc[1], wtc]
    grads = _grad_targets(dec._weights(), grads_out)
    for n, g in zip(_DEC_GRAD_NAMES, grads):
        setattr(b, n, g.data_ptr())
    dSpeech = torch.empty((B, T, S), dtype=torch.float32, device=dev)
    dStyle = torch.empty((B, T, Z), dtype=torch.float32, device=dev)
    b.dSpeech, b.dStyle = dSpeech.data_ptr(), dStyle.data_ptr()
    wsb = l.zeggs_decoder_bwd_workspace_bytes(B, T, H, S, Z)
    bws = WS.get("dec_bwd", wsb, dev)
    b.workspace, b.workspace_bytes = bws.data_ptr(), wsb
    if not split:
        _lib.check(l.zeggs_decoder_window_bwd(a, b, _lib.stream_ptr()), "zeggs_decoder_window_bwd")
        return grads, dSpeech, dStyle
    b.phase = 1
    _lib.check(l.zeggs_decoder_window_bwd(a, b, _lib.stream_ptr()), "zeggs_decoder_window_bwd (phase 1)")

    def finish():
        b.phase = 2
        _lib.check(l.zeggs_decoder_window_bwd(a, b, _lib.stream_ptr()), "zeggs_decoder_window_bwd (phase 2)")
        return hold, bws, grads, state        # everything phase 2 reads stays referenced until it has been issued
    return grads, dSpeech, dStyle, finish


def loss_fwd_bwd(Y, rp, rq, WY, Wrp, Wrq, gaze, parents_i32, dt, mu, logvar, kl_weight, terms_out=None, kl_weight_dev=None):
    """train.py:277-421 forward and gradient in one call (zeggs_loss_fwd_bwd) -> (loss = terms[0], (dY, dRp, dRq, dmu, dlogvar))."""
    l = _lib.lib()
    dev = Y.device
    B, T = Y.shape[0], Y.shape[1]
    f = _f32c
    Y, rp, rq, WY, Wrp, Wrq, gaze = f(Y), f(rp), f(rq), f(WY), f(Wrp), f(Wrq), f(gaze)
    losses = terms_out if terms_out is not None else torch.empty(19, dtype=torch.float32, device=dev)
    dY, dRp, dRq = torch.empty_like(Y), torch.empty_like(rp), torch.empty_like(rq)
    a = _lib.LossArgs(B=B, T=T, Z=(mu.shape[1] if mu is not None else 0), dt=dt, kl_weight=kl_weight)
    if kl_weight_dev is not None:          # device scalar (graph-replayable): overrides the by-value weight
        a.kl_weight_dev = kl_weight_dev.data_ptr()
    a.Y, a.root_pos, a.root_rot = Y.data_ptr(), rp.data_ptr(), rq.data_ptr()
    a.WY, a.W_root_pos, a.W_root_rot = WY.data_ptr(), Wrp.data_ptr(), Wrq.data_ptr()
    a.gaze_pos, a.parents, a.losses = gaze.data_ptr(), parents_i32.data_ptr(), losses.data_ptr()
    a.dY, a.dRootPos, a.dRootRot = dY.data_ptr(), dRp.data_ptr(), dRq.data_ptr()
    dmu = dlv = None
    if mu is not None:
        mu, logvar = f(mu), f(logvar)
        dmu, dlv = torch.empty_like(mu), torch.empty_like(logvar)
        a.mu, a.logvar, a.dmu, a.dlogvar = mu.data_ptr(), logvar.data_ptr(), dmu.data_ptr(), dlv.data_ptr()
    wsb = l.zeggs_loss_workspace_bytes(B, T)
    ws = WS.get("loss", wsb, dev)
    a.workspace, a.workspace_bytes = ws.data_ptr(), wsb
    _lib.check(l.zeggs_loss_fwd_bwd(a, _lib.stream_ptr()), "zeggs_loss_fwd_bwd")
    return losses[0], (dY, dRp, dRq, dmu, dlv)


def decoder_window(dec, root_pos0, root_rot0, pose0, gaze_pos, speech, style,
                   in_mean, in_std, out_mean, out_std, dt):
    if speech.device.type != "cuda":
        raise _lib.ZeggsError("zeggs_b200.Decoder runs on CUDA tensors only (no CPU fallback)")
    B = speech.shape[0]
    if B > 32 and resolve_engine(dec.hidden_size, dec.speech_encoding_size, dec.style_encoding_size):
        # the tensor-core recurrence works on one 32-sample batch tile: independent windows -> run the tiles back to back
        outs = [decoder_window(dec, root_pos0[i:i + 32], root_rot0[i:i + 32], pose0[i:i + 32], gaze_pos[i:i + 32],
                               speech[i:i + 32], style[i:i + 32], in_mean, in_std, out_mean, out_std, dt)
                for i in range(0, B, 32)]
        return tuple(torch.cat(o, 0) for o in zip(*outs))
    needs_grad = torch.is_grad_enabled() and (
        any(p.requires_grad for p in dec.parameters()) or speech.requires_grad or style.requires_grad)
    if needs_grad:
        from .autograd import DecoderWindowFn
        return DecoderWindowFn.apply(dec, root_pos0, root_rot0, pose0, gaze_pos, speech, style,
                                     in_mean, in_std, out_mean, out_std, dt, *dec._weights())
    Y, rp, rq, _ = decoder_window_forward(dec, root_pos0, root_rot0, pose0, gaze_pos, speech, style,
                                          (in_mean, in_std, out_mean, out_std), dt, save=False)
    return Y, rp, rq


def sgemm(A, B, bias=None, act=0, trans_a=False, out=None, accumulate=False):
    """trans_a False: act(A[M,K] @ B[N,K]^T + bias);  True: A[K,M]^T @ B[K,N]."""
    if trans_a:
        K, M = A.shape
        N = B.shape[1]
    else:
        M, K = A.shape
        N = B.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    _lib.check(_lib.lib().zeggs_sgemm(int(trans_a), M, N, K, _lib.ptr(A), A.stride(0), _lib.ptr(B), B.stride(0),
                                     _lib.ptr(bias) if bias is not None else None, _lib.ptr(out), out.stride(0),
                                     act, int(accumulate), _lib.stream_ptr()), "zeggs_sgemm")
    return out


def split_bf16(x, want_lo=True, pad_to=8):
    """fp32 [rows, cols] -> (hi, lo) bf16 [rows, ld] with ld = cols rounded up to `pad_to` (zero padded)."""
    rows, cols = x.shape
    ld = (cols + pad_to - 1) // pad_to * pad_to
    hi = torch.empty((rows, ld), dtype=torch.bfloat16, device=x.device)
    lo = torch.empty((rows, ld), dtype=torch.bfloat16, device=x.device) if want_lo else None
    _lib.check(_lib.lib().zeggs_split_bf16(_lib.ptr(x), rows, cols, x.stride(0), hi.data_ptr(),
                                          lo.data_ptr() if want_lo else None, ld, _lib.stream_ptr()), "zeggs_split_bf16")
    return hi, lo


def tc_gemm(A_hi, B_hi, A_lo=None, B_lo=None, K=None, bias=None, act=0, out=None, accumulate=False):
    """tcgen05 GEMM: act(A[M,K] @ B[N,K]^T + bias); bf16 operands (optionally split hi/lo), fp32 result."""
    M, N = A_hi.shape[0], B_hi.shape[0]
    K = K or A_hi.shape[1]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=A_hi.device)
    _lib.check(_lib.lib().zeggs_tc_gemm_bf16(
        M, N, K, A_hi.data_ptr(), A_lo.data_ptr() if A_lo is not None else None, A_hi.stride(0),
        B_hi.data_ptr(), B_lo.data_ptr() if B_lo is not None else None, B_hi.stride(0),
        _lib.ptr(bias) if bias is not None else None, _lib.ptr(out), out.stride(0), act, int(accumulate),
        _lib.stream_ptr()), "zeggs_tc_gemm_bf16")
    return out


# ---------------------------------------------------------------------------------------------- encoders
class DeviceSeed:
    """Dropout seed in DEVICE memory (zeggs_dropout_mask_dev): a captured CUDA graph of the train step draws fresh masks on every
    replay because `advance()` -- one in-graph increment -- is part of the step.  `salt` separates the masks within a step."""

    def __init__(self, device):
        self.t = torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).to(device)      # torch.manual_seed() -> reproducible runs
        self.salt = 0

    def advance(self):
        self.t.add_(1)
        self.salt = 0


_dev_seed = None


class device_seed:
    """Context: dropout masks drawn inside it use `seed` (a DeviceSeed) instead of the host generator."""

    def __init__(self, seed):
        self.seed = seed

    def __enter__(self):
        global _dev_seed
        self.prev, _dev_seed = _dev_seed, self.seed

    def __exit__(self, *exc):
        global _dev_seed
        _dev_seed = self.prev


def _drop_mask(shape, p, device):
    """Dropout mask (u >= p) / (1 - p) in one kernel; the seed comes from torch's CPU generator, so torch.manual_seed()
    makes training runs reproducible (and no device synchronisation is involved) -- or from a DeviceSeed inside a
    `device_seed` context (graph-replayable)."""
    out = torch.empty(shape, dtype=torch.float32, device=device)
    if _dev_seed is not None:
        _dev_seed.salt += 1
        _lib.check(_lib.lib().zeggs_dropout_mask_dev(out.data_ptr(), out.numel(), float(p), _dev_seed.t.data_ptr(), _dev_seed.salt,
                                                    _lib.stream_ptr()), "zeggs_dropout_mask_dev")
        return out
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    _lib.check(_lib.lib().zeggs_dropout_mask(out.data_ptr(), out.numel(), float(p), seed, _lib.stream_ptr()), "zeggs_dropout_mask")
    return out


def speech_enc_args(enc, x, masks, y, ws):
    w = [_f32c(p, x.device) for p in enc._weights()]
    H, Cin = w[0].shape[0], w[0].shape[1]
    O = w[2].shape[0]
    B, T = x.shape[0], x.shape[1]
    a = _lib.SpeechEncArgs(B=B, T=T, C_in=Cin, H=H, O=O, ctx=ctx_ptr(x.device))
    for n, t in zip(("W0", "b0", "W1", "b1", "W2", "b2"), w):
        setattr(a, n, t.data_ptr())
    a.x, a.y = x.data_ptr(), y.data_ptr()
    if masks is not None:
        a.mask0, a.mask1 = masks[0].data_ptr(), masks[1].data_ptr()
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    return a, w


def speech_encoder_masks(enc, x, masks=None):
    """Dropout multipliers of modules.py:263-270 (sampled in train mode unless injected)."""
    B, T = x.shape[0], x.shape[1]
    H, O = enc.layer0.weight.shape[0], enc.layer1.weight.shape[0]
    if masks is None and enc.training:
        masks = (_drop_mask((B, T, H), 0.2, x.device), _drop_mask((B, T, O), 0.2, x.device))
    if masks is not None:
        masks = tuple(_f32c(m, x.device) for m in masks)
    return masks


def speech_encoder_fwd(enc, x, masks):
    """zeggs_speech_enc_fwd -> (y [B,T,O], state for speech_encoder_bwd)."""
    if x.device.type != "cuda":
        raise _lib.ZeggsError("zeggs_b200.SpeechEncoder runs on CUDA tensors only (no CPU fallback)")
    l = _lib.lib()
    ensure_scratch(x.device)
    x = _f32c(x)
    weights = enc._weights()
    B, T = x.shape[0], x.shape[1]
    Cin, H, O = weights[0].shape[1], weights[0].shape[0], weights[2].shape[0]
    y = torch.empty((B, T, O), dtype=torch.float32, device=x.device)
    ws = torch.empty(l.zeggs_speech_enc_workspace_bytes(B, T, Cin, H, O), dtype=torch.uint8, device=x.device)
    a, keep = speech_enc_args(enc, x, masks, y, ws)
    _lib.check(l.zeggs_speech_enc_fwd(a, _lib.stream_ptr()), "zeggs_speech_enc_fwd")
    return y, (a, keep, x, masks, y, ws, weights)


def speech_encoder_bwd(state, dy, grads_out=None):
    a, keep, x, masks, y, ws, weights = state
    a.ctx = ctx_ptr(x.device)              # the lane this call is issued from (may differ from the forward's)
    dy = dy.contiguous().float()
    grads = _grad_targets(weights, grads_out)
    g = _lib.SpeechEncGrads(dy=dy.data_ptr())
    for n, t in zip(("dW0", "db0", "dW1", "db1", "dW2", "db2"), grads):
        setattr(g, n, t.data_ptr())
    _lib.check(_lib.lib().zeggs_speech_enc_bwd(a, g, _lib.stream_ptr()), "zeggs_speech_enc_bwd")
    return grads


def speech_encoder(enc, x, masks=None):
    if x.device.type != "cuda":
        raise _lib.ZeggsError("zeggs_b200.SpeechEncoder runs on CUDA tensors only (no CPU fallback)")
    from .autograd import SpeechEncoderFn
    return SpeechEncoderFn.apply(enc, x, speech_encoder_masks(enc, x, masks), *enc._weights())


_pe_cache = {}


def style_enc_args(enc, x, eps, masks, temperature, outs, ws):
    dev = x.device
    w = [_f32c(p, dev) for p in enc._weights()]
    B, T, Cin = x.shape
    Hs, E = w[0].shape[0], w[4].shape[0]
    nh = enc.encoder.blocks[0].attention.multi_head_attention.num_heads
    a = _lib.StyleEncArgs(B=B, T=T, C_in=Cin, H=Hs, E=E, nheads=nh, temperature=temperature, ctx=ctx_ptr(dev))
    for n, t in zip(_lib.STYLE_W, w):
        setattr(a, n, t.data_ptr())
    key = (T, E, str(dev))
    if key not in _pe_cache:
        _pe_cache[key] = enc.encoder.pos_enc.table(T).to(dev).contiguous()
    pe = _pe_cache[key]
    a.x, a.pe = x.data_ptr(), pe.data_ptr()
    if eps is not None:
        a.eps = eps.data_ptr()
    if masks is not None:
        for n in ("c1", "c2", "attn", "ao", "ff"):
            setattr(a, "mask_" + n, masks[n].data_ptr())
    a.z, a.mu, a.logvar = (o.data_ptr() for o in outs)
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    return a, w + [pe]


def style_encoder_fwd(enc, x, eps, masks, temperature):
    """zeggs_style_enc_fwd -> ([z, mu, logvar], state for style_encoder_bwd)."""
    l = _lib.lib()
    x = _f32c(x)
    weights = enc._weights()
    B, T, Cin = x.shape
    Hs, E = weights[0].shape[0], weights[4].shape[0]
    nh = enc.encoder.blocks[0].attention.multi_head_attention.num_heads
    outs = [torch.empty((B, E // 2), dtype=torch.float32, device=x.device) for _ in range(3)]
    ws = torch.empty(l.zeggs_style_enc_workspace_bytes(B, T, Cin, Hs, E, nh), dtype=torch.uint8, device=x.device)
    a, keep = style_enc_args(enc, x, eps, masks, temperature, outs, ws)
    _lib.check(l.zeggs_style_enc_fwd(a, _lib.stream_ptr()), "zeggs_style_enc_fwd")
    return outs, (a, keep, x, eps, masks, outs, ws, weights)


def style_encoder_bwd(state, dz, dmu, dlv, grads_out=None):
    a, keep, x, eps, masks, outs, ws, weights = state
    a.ctx = ctx_ptr(x.device)              # the lane this call is issued from (may differ from the forward's)
    g = _lib.StyleEncGrads()
    hold = []
    for n, t in (("dz", dz), ("dmu", dmu), ("dlogvar", dlv)):
        if t is not None:
            t = t.contiguous().float()
            hold.append(t)
            setattr(g, n, t.data_ptr())
    grads = _grad_targets(weights, grads_out)
    for n, t in zip(_lib.STYLE_W, grads):
        setattr(g, "d" + n, t.data_ptr())
    _lib.check(_lib.lib().zeggs_style_enc_bwd(a, g, _lib.stream_ptr()), "zeggs_style_enc_bwd")
    return grads


def style_encoder_prepare(enc, x, eps=None, masks=None):
    """VAE noise (modules.py:299) and dropout multipliers (sampled in train mode unless injected) -> (eps, masks)."""
    dev = x.device
    ensure_scratch(dev)
    B, T = x.shape[0], x.shape[1]
    Hs = enc.encoder.convs[0].conv.weight.shape[0]
    E = enc.encoder.convs[4].conv.weight.shape[0]
    nh = enc.encoder.blocks[0].attention.multi_head_attention.num_heads
    if eps is None:
        if _dev_seed is not None:                           # device-seeded draw (replayable graph), else torch's generator
            eps = torch.empty((B, E // 2), dtype=torch.float32, device=dev)
            _dev_seed.salt += 1
            _lib.check(_lib.lib().zeggs_randn_dev(eps.data_ptr(), eps.numel(), _dev_seed.t.data_ptr(), _dev_seed.salt, _lib.stream_ptr()),
                       "zeggs_randn_dev")
        else:
            eps = torch.randn((B, E // 2), device=dev)      # modules.py:299
    if masks is None and enc.training:
        masks = dict(c1=_drop_mask((B, T, Hs), 0.2, dev), c2=_drop_mask((B, T, E), 0.2, dev),
                     attn=_drop_mask((B, nh, T, T), 0.1, dev), ao=_drop_mask((B, T, E), 0.1, dev),
                     ff=_drop_mask((B, T, E), 0.1, dev))
    if masks is not None:
        masks = {k: _f32c(v, dev) for k, v in masks.items()}
    return _f32c(eps, dev), masks


def style_encoder(enc, x, temperature=1.0, eps=None, masks=None):
    if x.device.type != "cuda":
        raise _lib.ZeggsError("zeggs_b200.StyleEncoder runs on CUDA tensors only (no CPU fallback)")
    from .autograd import StyleEncoderFn
    eps, masks = style_encoder_prepare(enc, x, eps, masks)
    return StyleEncoderFn.apply(enc, x, eps, masks, temperature, *enc._weights())


# ---------------------------------------------------------------------------------------------- pose -> BVH channel values
def pose_to_bvh_channels(root_pos, root_rot, lpos, ltxy, start_position=(0.0, 0.0, 0.0), start_rotation=(1.0, 0.0, 0.0, 0.0),
                         rebase=True, want_lrot=False):
    """Device post-step of generate.py:389-406 / utils.py:47-87: [N,T,...] pose tensors -> (positions [N,T,J,3], euler degrees
    [N,T,J,3] in 'zyx' channel order[, local rotations [N,T,J,4]]).  rebase: move the root's first frame to start_position /
    start_rotation, as write_bvh does when both are given."""
    if root_pos.device.type != "cuda":
        raise _lib.ZeggsError("pose_to_bvh_channels runs on CUDA tensors only (no CPU fallback)")
    rp, rq, lp, xy = _f32c(root_pos), _f32c(root_rot), _f32c(lpos), _f32c(ltxy)
    if rp.dim() == 2:
        rp, rq, lp, xy = rp[None], rq[None], lp[None], xy[None]
    N, T, J = lp.shape[0], lp.shape[1], lp.shape[2]
    pos = torch.empty((N, T, J, 3), dtype=torch.float32, device=lp.device)
    eul = torch.empty((N, T, J, 3), dtype=torch.float32, device=lp.device)
    lrot = torch.empty((N, T, J, 4), dtype=torch.float32, device=lp.device) if want_lrot else None
    a = _lib.PosePostArgs(N=N, T=T, J=J, rebase=int(bool(rebase)), root_pos=rp.data_ptr(), root_rot=rq.data_ptr(), lpos=lp.data_ptr(),
                          ltxy=xy.data_ptr(), positions=pos.data_ptr(), euler_deg=eul.data_ptr(),
                          lrot=lrot.data_ptr() if want_lrot else None)
    for i in range(3):
        a.start_pos[i] = float(start_position[i])
    for i in range(4):
        a.start_rot[i] = float(start_rotation[i])
    _lib.check(_lib.lib().zeggs_pose_to_bvh_channels(a, _lib.stream_ptr()), "zeggs_pose_to_bvh_channels")
    return (pos, eul, lrot) if want_lrot else (pos, eul)


# ---------------------------------------------------------------------------------------------- single decoder step
def decoder_step(dec, pose, speech, style, state):
    """RecurrentDecoderNormal.forward (modules.py:179-185) for one frame, fp32: pose [B,1134] normalised input vector, speech [B,S],
    style [B,Z], state [2,B,H] -> (y [B,1131] normalised, new state [2,B,H])."""
    if pose.device.type != "cuda":
        raise _lib.ZeggsError("decoder_step runs on CUDA tensors only (no CPU fallback)")
    l = _lib.lib()
    dev = pose.device
    w = [_f32c(p, dev) for p in dec._weights()[:12]]
    pose, speech, style, state = _f32c(pose), _f32c(speech), _f32c(style), _f32c(state)
    B, H, S, Z = pose.shape[0], dec.hidden_size, speech.shape[1], style.shape[1]
    y = torch.empty((B, P_OUT), dtype=torch.float32, device=dev)
    h_out = torch.empty((2, B, H), dtype=torch.float32, device=dev)
    wsb = l.zeggs_decoder_step_workspace_bytes(B, H, S, Z)
    ws = WS.get("dec_step", wsb, dev)
    a = _lib.DecoderStepArgs(B=B, H=H, S=S, Z=Z, pose=pose.data_ptr(), speech=speech.data_ptr(), style=style.data_ptr(),
                             h_in=state.data_ptr(), y=y.data_ptr(), h_out=h_out.data_ptr(), workspace=ws.data_ptr(), workspace_bytes=wsb)
    for n, t in zip(("W0", "b0", "W_ih0", "b_ih0", "W_hh0", "b_hh0", "W_ih1", "b_ih1", "W_hh1", "b_hh1", "W2", "b2"), w):
        setattr(a, n, t.data_ptr())
    _lib.check(l.zeggs_decoder_step_fwd(a, _lib.stream_ptr()), "zeggs_decoder_step_fwd")
    return y, h_out
