"""ctypes binding of libzeggs_b200.so (include/zeggs_b200.h).  Fails loudly when the library is
missing: there is no CPU or PyTorch fallback for the compute path."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libzeggs_b200.so")

c_float_p = C.c_void_p  # raw device pointers are passed as integers (tensor.data_ptr())


class MelArgs(C.Structure):
    _fields_ = [("n_clips", C.c_int), ("n_samples", C.c_int), ("n_fft", C.c_int), ("hop", C.c_int),
                ("n_mels", C.c_int), ("anim_length", C.c_int), ("min_amp", C.c_float),
                ("frames_per_anim", C.c_double),
                ("wav", C.c_void_p), ("window", C.c_void_p), ("twiddle", C.c_void_p),
                ("fb_start", C.c_void_p), ("fb_len", C.c_void_p), ("fb_off", C.c_void_p), ("fb_w", C.c_void_p),
                ("mel_out", C.c_void_p), ("feat_out", C.c_void_p), ("fb_total", C.c_int),
                ("gain", C.c_void_p), ("wav_i16", C.c_void_p)]


GATHER_MAX = 12


class GatherArgs(C.Structure):
    _fields_ = [("B", C.c_int), ("T", C.c_int), ("n_arrays", C.c_int), ("src", C.c_void_p * GATHER_MAX), ("dst", C.c_void_p * GATHER_MAX),
                ("width", C.c_int * GATHER_MAX), ("start", C.c_void_p), ("ex_out", C.c_void_p), ("L", C.c_int), ("ex_width", C.c_int),
                ("n_ex", C.c_int), ("ex_src", C.c_int * GATHER_MAX), ("ex_start", C.c_void_p), ("ex_n", C.c_void_p)]


class PosePostArgs(C.Structure):
    _fields_ = [("N", C.c_int), ("T", C.c_int), ("J", C.c_int), ("rebase", C.c_int), ("start_pos", C.c_float * 3),
                ("start_rot", C.c_float * 4), ("root_pos", C.c_void_p), ("root_rot", C.c_void_p), ("lpos", C.c_void_p),
                ("ltxy", C.c_void_p), ("positions", C.c_void_p), ("euler_deg", C.c_void_p), ("lrot", C.c_void_p)]


class LoudnessArgs(C.Structure):
    _fields_ = [("n_clips", C.c_int), ("n_samples", C.c_int), ("n_seg", C.c_int), ("n_blocks", C.c_int), ("warm", C.c_int),
                ("coef", C.c_double * 10), ("inv_block_len", C.c_double), ("target_lufs", C.c_double),
                ("wav", C.c_void_p), ("wav_i16", C.c_void_p), ("seg_bounds", C.c_void_p), ("blk_seg_lo", C.c_void_p),
                ("blk_seg_hi", C.c_void_p), ("gain_out", C.c_void_p), ("lufs_out", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class Ctx(C.Structure):
    """zeggs_ctx: per-call GEMM context (scratch buffer, GEMM mode, single-pass weight gradients)."""
    _fields_ = [("scratch", C.c_void_p), ("scratch_bytes", C.c_size_t), ("gemm_mode", C.c_int), ("fast_wgrad", C.c_int)]


class DecoderFwdArgs(C.Structure):
    _fields_ = ([("B", C.c_int), ("T", C.c_int), ("H", C.c_int), ("S", C.c_int), ("Z", C.c_int), ("dt", C.c_float)] +
                [(n, C.c_void_p) for n in (
                    "W0", "b0", "W_ih0", "b_ih0", "W_hh0", "b_hh0", "W_ih1", "b_ih1", "W_hh1", "b_hh1", "W2", "b2",
                    "Wc0", "bc0", "Wc1", "bc1", "Wc2", "bc2", "packed",
                    "in_mean", "in_std", "out_mean", "out_std",
                    "root_pos0", "root_rot0", "pose0", "gaze_pos", "speech", "style",
                    "Y", "root_pos", "root_rot", "workspace")] +
                [("workspace_bytes", C.c_size_t), ("save_for_backward", C.c_int), ("engine", C.c_int),
                 ("packed_tc", C.c_void_p), ("workspace_tc", C.c_void_p), ("ctx", C.c_void_p)])


class DecoderBwdArgs(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in (
        "dY", "dRootPos", "dRootRot", "packed_bwd",
        "dW0", "db0", "dW_ih0", "db_ih0", "dW_hh0", "db_hh0", "dW_ih1", "db_ih1", "dW_hh1", "db_hh1", "dW2", "db2",
        "dWc0", "dbc0", "dWc1", "dbc1", "dWc2", "dbc2", "dSpeech", "dStyle", "workspace")] +
        [("workspace_bytes", C.c_size_t), ("packed_bwd_tc", C.c_void_p), ("workspace_tc", C.c_void_p), ("phase", C.c_int)])


class DecoderStateArgs(C.Structure):
    """zeggs_decoder_state_args: GRU state in ([2,B,H], per-sample int32 selector) and out ([2,B,H]) of a resumable window."""
    _fields_ = [("h_init", C.c_void_p), ("init_from_state", C.c_void_p), ("h_final", C.c_void_p)]


def _struct(name, ints=(), floats=(), ptrs=(), tail=()):
    fields = [(n, C.c_int) for n in ints] + [(n, C.c_float) for n in floats] + [(n, C.c_void_p) for n in ptrs] + list(tail)
    return type(name, (C.Structure,), {"_fields_": fields})


SpeechEncArgs = _struct("SpeechEncArgs", ints=("B", "T", "C_in", "H", "O"),
                        ptrs=("W0", "b0", "W1", "b1", "W2", "b2", "x", "mask0", "mask1", "y", "workspace"),
                        tail=[("workspace_bytes", C.c_size_t), ("ctx", C.c_void_p)])
SpeechEncGrads = _struct("SpeechEncGrads", ptrs=("dy", "dW0", "db0", "dW1", "db1", "dW2", "db2"))
STYLE_W = ("Wc1", "bc1", "ln1_g", "ln1_b", "Wc2", "bc2", "ln2_g", "ln2_b", "Win", "bin", "Wout", "bout", "ln3_g", "ln3_b",
           "Wf1", "bf1", "Wf2", "bf2", "ln4_g", "ln4_b")
StyleEncArgs = _struct("StyleEncArgs", ints=("B", "T", "C_in", "H", "E", "nheads"), floats=("temperature",),
                       ptrs=STYLE_W + ("x", "eps", "pe", "mask_c1", "mask_c2", "mask_attn", "mask_ao", "mask_ff",
                                       "z", "mu", "logvar", "workspace"),
                       tail=[("workspace_bytes", C.c_size_t), ("ctx", C.c_void_p)])
StyleEncGrads = _struct("StyleEncGrads", ptrs=("dz", "dmu", "dlogvar") + tuple("d" + n for n in STYLE_W))


DecoderStepArgs = _struct("DecoderStepArgs", ints=("B", "H", "S", "Z"),
                          ptrs=("W0", "b0", "W_ih0", "b_ih0", "W_hh0", "b_hh0", "W_ih1", "b_ih1", "W_hh1", "b_hh1", "W2", "b2",
                                "pose", "speech", "style", "h_in", "y", "h_out", "workspace"),
                          tail=[("workspace_bytes", C.c_size_t)])
LossArgs = _struct("LossArgs", ints=("B", "T", "Z"), floats=("dt", "kl_weight"),
                   ptrs=("Y", "root_pos", "root_rot", "WY", "W_root_pos", "W_root_rot", "gaze_pos", "parents", "mu", "logvar",
                         "losses", "dY", "dRootPos", "dRootRot", "dmu", "dlogvar", "workspace"),
                   tail=[("workspace_bytes", C.c_size_t), ("kl_weight_dev", C.c_void_p)])


# every symbol include/zeggs_b200.h declares: (name, restype, argtypes)
# C struct name -> ctypes mirror (checked against the library's sizeof at test time: tests/test_abi_cpu.py)
def struct_mirrors():
    return {"zeggs_ctx": Ctx, "zeggs_mel_args": MelArgs, "zeggs_loudness_args": LoudnessArgs, "zeggs_decoder_fwd_args": DecoderFwdArgs,
            "zeggs_decoder_bwd_args": DecoderBwdArgs, "zeggs_speech_enc_args": SpeechEncArgs, "zeggs_speech_enc_grads": SpeechEncGrads,
            "zeggs_style_enc_args": StyleEncArgs, "zeggs_style_enc_grads": StyleEncGrads, "zeggs_decoder_step_args": DecoderStepArgs,
            "zeggs_loss_args": LossArgs, "zeggs_pose_post_args": PosePostArgs, "zeggs_gather_args": GatherArgs,
            "zeggs_decoder_state_args": DecoderStateArgs}


SYMBOLS = [
    ("zeggs_last_error", C.c_char_p, []),
    ("zeggs_version", C.c_int, []),
    ("zeggs_struct_size", C.c_size_t, [C.c_char_p]),
    ("zeggs_launch_count", C.c_longlong, []),
    ("zeggs_timing_enable", None, [C.c_int]),
    ("zeggs_timing_reset", None, []),
    ("zeggs_timing_read", C.c_int, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    ("zeggs_mel_num_frames", C.c_int, [C.c_int, C.c_int, C.c_int]),
    ("zeggs_mel_forward", C.c_int, [C.POINTER(MelArgs), C.c_void_p]),
    ("zeggs_decoder_step_workspace_bytes", C.c_size_t, [C.c_int] * 4),
    ("zeggs_decoder_step_fwd", C.c_int, [C.POINTER(DecoderStepArgs), C.c_void_p]),
    ("zeggs_window_gather", C.c_int, [C.POINTER(GatherArgs), C.c_void_p]),
    ("zeggs_normalize_rows", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    ("zeggs_pose_to_bvh_channels", C.c_int, [C.POINTER(PosePostArgs), C.c_void_p]),
    ("zeggs_loudness_workspace_bytes", C.c_size_t, [C.c_int, C.c_int]),
    ("zeggs_loudness_gain", C.c_int, [C.POINTER(LoudnessArgs), C.c_void_p]),
    ("zeggs_decoder_packed_bytes", C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    ("zeggs_decoder_pack_weights", C.c_int, [C.POINTER(DecoderFwdArgs), C.c_void_p, C.c_void_p]),
    ("zeggs_decoder_workspace_bytes", C.c_size_t, [C.c_int] * 6),
    ("zeggs_decoder_window_fwd", C.c_int, [C.POINTER(DecoderFwdArgs), C.c_void_p]),
    ("zeggs_decoder_window_fwd_state", C.c_int, [C.POINTER(DecoderFwdArgs), C.POINTER(DecoderStateArgs), C.c_void_p]),
    ("zeggs_decoder_packed_tc_bytes", C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    ("zeggs_decoder_tc_workspace_bytes", C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    ("zeggs_decoder_pack_weights_tc", C.c_int, [C.POINTER(DecoderFwdArgs), C.c_void_p, C.c_void_p]),
    ("zeggs_debug_set_tc_trace", None, [C.c_void_p]),
    ("zeggs_debug_set_tc_nacc", None, [C.c_int]),
    ("zeggs_debug_set_tc_gemm_variant", C.c_int, [C.c_int]),
    ("zeggs_debug_set_loss_impl", None, [C.c_int]),
    ("zeggs_debug_set_tc_cluster", None, [C.c_int]),
    ("zeggs_debug_get_tc_cluster", C.c_int, []),
    ("zeggs_decoder_packed_bwd_bytes", C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    ("zeggs_decoder_pack_weights_bwd", C.c_int, [C.POINTER(DecoderFwdArgs), C.c_void_p, C.c_void_p]),
    ("zeggs_decoder_bwd_workspace_bytes", C.c_size_t, [C.c_int] * 5),
    ("zeggs_decoder_window_bwd", C.c_int, [C.POINTER(DecoderFwdArgs), C.POINTER(DecoderBwdArgs), C.c_void_p]),
    ("zeggs_decoder_packed_bwd_tc_bytes", C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    ("zeggs_decoder_bwd_tc_workspace_bytes", C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    ("zeggs_decoder_pack_weights_bwd_tc", C.c_int, [C.POINTER(DecoderFwdArgs), C.c_void_p, C.c_void_p]),
    ("zeggs_speech_enc_workspace_bytes", C.c_size_t, [C.c_int] * 5),
    ("zeggs_speech_enc_fwd", C.c_int, [C.POINTER(SpeechEncArgs), C.c_void_p]),
    ("zeggs_speech_enc_bwd", C.c_int, [C.POINTER(SpeechEncArgs), C.POINTER(SpeechEncGrads), C.c_void_p]),
    ("zeggs_style_enc_workspace_bytes", C.c_size_t, [C.c_int] * 6),
    ("zeggs_style_enc_fwd", C.c_int, [C.POINTER(StyleEncArgs), C.c_void_p]),
    ("zeggs_style_enc_bwd", C.c_int, [C.POINTER(StyleEncArgs), C.POINTER(StyleEncGrads), C.c_void_p]),
    ("zeggs_loss_workspace_bytes", C.c_size_t, [C.c_int, C.c_int]),
    ("zeggs_loss_fwd_bwd", C.c_int, [C.POINTER(LossArgs), C.c_void_p]),
    ("zeggs_set_fast_wgrad", C.c_int, [C.c_int]),
    ("zeggs_dropout_mask", C.c_int, [C.c_void_p, C.c_size_t, C.c_float, C.c_ulonglong, C.c_void_p]),
    ("zeggs_dropout_mask_dev", C.c_int, [C.c_void_p, C.c_size_t, C.c_float, C.c_void_p, C.c_ulonglong, C.c_void_p]),
    ("zeggs_randn_dev", C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_ulonglong, C.c_void_p]),
    ("zeggs_radam_step_dev", C.c_int, [C.c_void_p] * 4 + [C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("zeggs_radam_step", C.c_int, [C.c_void_p] * 4 + [C.c_size_t, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, C.c_float, C.c_void_p]),
    ("zeggs_sgemm", C.c_int, [C.c_int] * 4 + [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                               C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("zeggs_tc_gemm_bf16", C.c_int, [C.c_int] * 3 + [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("zeggs_set_scratch", C.c_int, [C.c_void_p, C.c_size_t]),
    ("zeggs_set_gemm_mode", C.c_int, [C.c_int]),
    ("zeggs_gemm_f32", C.c_int, [C.c_int] * 4 + [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("zeggs_gemm_f32_ctx", C.c_int, [C.c_void_p] + [C.c_int] * 4 + [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("zeggs_split_bf16", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
]

_lib = None


class ZeggsError(RuntimeError):
    pass


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ZeggsError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "zeggs_b200 has no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(l, name)  # AttributeError if the ABI and the header drift apart
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().zeggs_last_error()
        raise ZeggsError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a contiguous float32/int32 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise ZeggsError("zeggs_b200 kernels take CUDA tensors (no CPU path)")
    if not t.is_contiguous():
        raise ZeggsError("tensor must be contiguous")
    return t.data_ptr()
