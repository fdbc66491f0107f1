"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from
/root/reference via oracle/ref_shim.py) on seeded synthetic inputs.

Run in the dev container (the reference tree does not exist on the GPU box):
    python -m oracle.make_golden
Weights are regenerated from zeggs_b200.synth.make_params(seed) on both sides, so only
inputs' seeds and the reference OUTPUTS are stored.
"""
import os
import types

import numpy as np
import torch

from oracle import ref_shim
from zeggs_b200 import synth

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def tt(d):
    return {k: torch.from_numpy(np.asarray(v)) for k, v in d.items()}


def build_ref_nets(P, H, S=64, Z=64, style_hidden=512, use_vae=True):
    m = ref_shim.ref_modules()
    se = m.SpeechEncoder(synth.N_AUDIO, S, S)
    de = m.Decoder(synth.P_IN, synth.P_OUT, S, Z, H, 2)
    st = m.StyleEncoder(synth.P_IN, style_hidden, Z, type="attn", use_vae=use_vae)
    Pt = tt(P)
    se.load_state_dict({k[len("speech_encoder."):]: v for k, v in Pt.items() if k.startswith("speech_encoder.")})
    de.load_state_dict({k[len("decoder."):]: v for k, v in Pt.items() if k.startswith("decoder.")})
    st.load_state_dict({k[len("style_encoder."):]: v for k, v in Pt.items() if k.startswith("style_encoder.")})
    return se, st, de


def audio_params(hop=200, n_fft=800):
    return types.SimpleNamespace(
        sampling_rate=16000, filter_length=n_fft, hop_length=hop, n_mel_channels=80, mel_fmin=20, mel_fmax=7600,
        min_clipping=1e-5, pre_emphasis=False, pre_emph_coeff=0.97, real_amplitude=True, centered=True,
        normalize_mel_bins=True, normalize_range=True, resample_method="linear", normalize_loudness=False)


def ref_train_losses(ns):
    """Execute the reference's own loss lines (train.py:277-421) where they lie, in namespace `ns`
    (expects O_*/W_* tensors, parents, dt, mu, logvar, iteration); returns the namespace."""
    ref_shim.install()
    path = os.path.join(ref_shim.REF_ZEGGS, "train.py")
    lines = open(path).read().split("\n")[275:421]       # train.py:276-421
    import textwrap
    src = textwrap.dedent("\n".join(lines))
    import anim.tquat as tq
    import anim.txform as tx
    import modules as m
    env = dict(torch=torch)
    for mod in (tq, tx):
        env.update({k: getattr(mod, k) for k in dir(mod) if not k.startswith("_")})
    env.update(compute_KL_div=m.compute_KL_div, normalize=m.normalize)
    env.update(ns)
    exec(compile(src, path, "exec"), env)
    return env


def stats_t():
    st = synth.load_stats()
    f = lambda k: torch.as_tensor(st[k], dtype=torch.float32)
    return (f("audio_input_mean"), f("audio_input_std"), f("anim_input_mean"), f("anim_input_std"),
            f("anim_output_mean"), f("anim_output_std"), torch.as_tensor(st["parents"]), float(st["dt"]))


def ref_forward_train(se, st, de, win, audio, style_ex, eps, iteration):
    """The reference's train-step forward in eval mode (no dropout) with injected VAE eps."""
    a_mu, a_sd, i_mu, i_sd, o_mu, o_sd, parents, dt = stats_t()
    W = tt(win)
    speech = se((torch.from_numpy(audio) - a_mu) / a_sd)
    # StyleEncoder.forward with eps injected (modules.py:289-304): replicate randn_like via manual formula
    enc = st.encoder((torch.from_numpy(style_ex) - i_mu) / i_sd)
    Z = st.style_embedding_size
    mu, logvar = enc[:, :Z], enc[:, Z:]
    z = mu + torch.from_numpy(eps) * torch.exp(0.5 * logvar)
    T = speech.shape[1]
    O = de(W["root_pos"][:, 0], W["root_rot"][:, 0], W["root_vel"][:, 0], W["root_vrt"][:, 0], W["lpos"][:, 0],
           W["ltxy"][:, 0], W["lvel"][:, 0], W["lvrt"][:, 0], W["gaze_pos"], speech, z.unsqueeze(1).repeat((1, T, 1)),
           parents, i_mu, i_sd, o_mu, o_sd, dt)
    names = ["root_pos", "root_rot", "root_vel", "root_vrt", "lpos", "ltxy", "lvel", "lvrt"]
    ns = {"O_" + n: o for n, o in zip(names, O)}
    ns.update({"W_" + n: W[n] for n in names})
    ns.update(W_gaze_pos=W["gaze_pos"], parents=parents, dt=dt, mu=mu, logvar=logvar, iteration=iteration)
    env = ref_train_losses(ns)
    return speech, (z, mu, logvar), O, env


TRAIN_CASES = {   # tag: (H, B, T, T_ex)
    "h64": (64, 2, 6, 16), "h128": (128, 4, 9, 24),
    # H % 128 == 0, H >= 384: the tensor-core recurrence engine is eligible (U = 4 / G = 96 CTAs at H = 384; U = 8 / G = 128
    # CTAs -- the bench geometry -- at H = 1024), so the same golden test runs tcgen05 against the REFERENCE's loss and gradients
    "h384": (384, 4, 12, 24),   # (B, T != 3: the reference's dim-less torch.cross hazard, DESIGN.md 1)
    "h1024": (1024, 2, 8, 16),
}


def write_train_golden(tag):
    H, B, T, T_ex = TRAIN_CASES[tag]
    P = synth.make_params(H=H, seed=11)
    se, st, de = build_ref_nets(P, H)
    se.eval(); st.eval(); de.eval()
    win = synth.make_pose_windows(B, T, seed=5)
    audio = synth.make_audio_features(B, T, seed=5)
    style_ex = synth.make_style_example(B, T_ex, seed=5)
    eps = np.random.RandomState(3).randn(B, 64).astype(np.float32)
    speech, (z, mu, logvar), O, env = ref_forward_train(se, st, de, win, audio, style_ex, eps, iteration=9000)
    loss = env["loss"]
    params = list(se.parameters()) + list(de.parameters()) + list(st.parameters())
    names = (["speech_encoder." + n for n, _ in se.named_parameters()] +
             ["decoder." + n for n, _ in de.named_parameters()] +
             ["style_encoder." + n for n, _ in st.named_parameters()])
    grads = torch.autograd.grad(loss, params)
    g = {"grad." + n: x.detach().numpy() for n, x in zip(names, grads) if x.numel() <= 4096}
    gn = {"gradnorm." + n: np.float64(x.double().norm().item()) for n, x in zip(names, grads)}
    d = dict(H=H, B=B, T=T, T_ex=T_ex, param_seed=11, input_seed=5, eps=eps, iteration=9000,
             speech=speech.detach().numpy(), z=z.detach().numpy(), mu=mu.detach().numpy(),
             logvar=logvar.detach().numpy(), loss=np.float64(loss.item()))
    for n, o in zip(["root_pos", "root_rot", "root_vel", "root_vrt", "lpos", "ltxy", "lvel", "lvrt"], O):
        d["O_" + n] = o.detach().numpy()
    for k in ["loss_root_pos", "loss_root_rot", "loss_root_vel", "loss_root_vrt", "loss_lpos", "loss_lrot",
              "loss_lvel", "loss_lvrt", "loss_cpos", "loss_crot", "loss_cvel", "loss_cvrt", "loss_ldvl",
              "loss_ldvt", "loss_cdvl", "loss_cdvt", "loss_gaze", "loss_kl_div"]:
        d[k] = np.float64(float(env[k]))
    d.update(g); d.update(gn)
    np.savez_compressed(os.path.join(GOLD, f"train_{tag}.npz"), **d)
    print(tag, "loss", loss.item())


V1_DIR = os.path.join(os.path.dirname(GOLD), "_v1")       # git-ignored: the shipped v1 weights as a flat .npz (travels with gpurun)


def write_v1_golden(B=2, T=96, T_ex=128):
    """The shipped v1 pickles (trained weights: larger gates, saturating GRUs) through the unmodified reference, eval mode, VAE
    noise = 0: outputs committed as tests/golden/v1_pretrained.npz; the weights themselves go to tests/_v1/weights.npz
    (git-ignored, ~112 MB) so the GPU box can run the CUDA path on them."""
    nets = ref_shim.load_pretrained("v1")
    se, st, de = nets["speech_encoder"], nets["style_encoder"], nets["decoder"]
    os.makedirs(V1_DIR, exist_ok=True)
    W = {}
    for pre, net in (("speech_encoder.", se), ("style_encoder.", st), ("decoder.", de)):
        for k, v in net.state_dict().items():
            W[pre + k] = v.detach().cpu().numpy()
    np.savez(os.path.join(V1_DIR, "weights.npz"), **W)
    a_mu, a_sd, i_mu, i_sd, o_mu, o_sd, parents, dt = stats_t()
    win = synth.make_pose_windows(B, T, seed=21)
    audio = synth.make_audio_features(B, T, seed=21)
    style_ex = synth.make_style_example(B, T_ex, seed=21)
    Wt = tt(win)
    with torch.no_grad():
        speech = se((torch.from_numpy(audio) - a_mu) / a_sd)
        enc = st.encoder((torch.from_numpy(style_ex) - i_mu) / i_sd)
        Z = st.style_embedding_size
        mu, logvar = enc[:, :Z], enc[:, Z:]
        O = de(Wt["root_pos"][:, 0], Wt["root_rot"][:, 0], Wt["root_vel"][:, 0], Wt["root_vrt"][:, 0], Wt["lpos"][:, 0],
               Wt["ltxy"][:, 0], Wt["lvel"][:, 0], Wt["lvrt"][:, 0], Wt["gaze_pos"], speech, mu.unsqueeze(1).repeat((1, T, 1)),
               parents, i_mu, i_sd, o_mu, o_sd, dt)
    d = dict(B=B, T=T, T_ex=T_ex, input_seed=21, speech=speech.numpy(), mu=mu.numpy(), logvar=logvar.numpy(),
             H=de.recurrent_decoder.layer1.hidden_size)
    for n, o in zip(["root_pos", "root_rot", "root_vel", "root_vrt", "lpos", "ltxy", "lvel", "lvrt"], O):
        d["O_" + n] = o.numpy()
    np.savez_compressed(os.path.join(GOLD, "v1_pretrained.npz"), **d)
    print("v1 golden written; weights ->", V1_DIR)


def main(only=None):
    os.makedirs(GOLD, exist_ok=True)
    torch.manual_seed(0)
    if only:
        for tag in only:
            if tag == "v1":
                write_v1_golden()
            elif tag == "generate":
                write_generate_golden()
            elif tag == "pose_post":
                write_pose_post_golden()
            elif tag in REFERENCE_IO:
                REFERENCE_IO[tag]()
            else:
                write_train_golden(tag)
        return
    # ---- mel / preprocess_audio (hop 200 reference-actual, hop 160 BASELINE.json-stated)
    pa = ref_shim.ref_preprocess_audio()
    from audio.spectrograms import extract_mel_spectrogram_for_tts
    wav = synth.make_waveforms(2, 16000, seed=7)
    wav[1, 4000:9000] = 0.0          # a silent stretch: exercises the 1.25e-8 clip floor
    out = {"wav": wav}
    for hop in (200, 160):
        p = audio_params(hop)
        n60 = int(round(60.0 * wav.shape[1] / 16000))
        feats, mels = [], []
        for i in range(wav.shape[0]):
            feats.append(pa(wav[i], 60, n60, p, ["mel_spec", "energy"]))
            mels.append(extract_mel_spectrogram_for_tts(
                wav_signal=wav[i], fs=16000, n_fft=800, step_size=hop, n_mels=80, mel_fmin=20, mel_fmax=7600,
                min_amplitude=1e-5, pre_emphasis=False, real_amplitude=True, centered=True,
                normalize_mel_bins=True, normalize_range=True)[0])
        out[f"feat_hop{hop}"] = np.stack(feats)
        out[f"mel_hop{hop}"] = np.stack(mels)
    np.savez_compressed(os.path.join(GOLD, "mel_small.npz"), **out)

    # ---- networks, eval mode: small hidden sizes (fp32 SIMT engine) and tensor-core-eligible ones
    for tag in TRAIN_CASES:
        write_train_golden(tag)
    write_v1_golden()
    write_pose_post_golden()
    write_generate_golden()
    for fn in REFERENCE_IO.values():
        fn()

    # ---- RAdam trajectory (optimizers.py), 8 steps crossing the N_sma>=5 switch (step 6)
    ref_shim.install()
    from optimizers import RAdam
    rs = np.random.RandomState(2)
    p0 = rs.randn(257).astype(np.float32)
    gs = rs.randn(8, 257).astype(np.float32)
    p = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    opt = RAdam([p], lr=1e-4, eps=1e-5)
    traj = []
    for i in range(8):
        p.grad = torch.from_numpy(gs[i].copy())
        opt.step()
        traj.append(p.detach().numpy().copy())
    np.savez_compressed(os.path.join(GOLD, "radam.npz"), p0=p0, grads=gs, traj=np.stack(traj))
    print("golden written to", GOLD)




# ---------------------------------------------------------------------------------------------- generate_gesture end to end
def _pyloudnorm_stub():
    """`pyloudnorm` is not installed: a stub backed by oracle/loudness_oracle.py (the restated 0.1.0 algorithm, parity unpinned)
    so that the reference's normalize_loudness=True code path (data_pipeline.py:34-39) can run for the golden."""
    import sys
    import types
    from oracle import loudness_oracle as lo
    m = types.ModuleType("pyloudnorm")

    class Meter:
        def __init__(self, rate):
            self.rate = rate

        def integrated_loudness(self, data):
            return lo.integrated_loudness(data, self.rate)

    m.Meter = Meter
    m.normalize = types.SimpleNamespace(loudness=lambda data, inp, target: np.power(10.0, (target - inp) / 20.0) * data)
    sys.modules["pyloudnorm"] = m


def write_generate_golden(H=256):
    """Run the UNMODIFIED reference generate_gesture (CPU) on the deterministic synthetic BVH + WAV of tests/_fixtures.py with
    synth weights (whole-module pickles of the reference's own classes) and store what it wrote: the BVH channel values and the
    returned style encoding, for three calls (one example style; two styles blended 'add'; two styles 'stitch'), with loudness
    normalisation off (pure reference arithmetic) and on (through the oracle-backed pyloudnorm stub)."""
    import json
    import pathlib
    import shutil
    import tempfile
    import torch
    from tests import _fixtures as fx
    ref_shim.install()
    _pyloudnorm_stub()
    import anim.bvh as rbvh
    import generate as rgen                     # ZEGGS/generate.py
    tmp = pathlib.Path(tempfile.mkdtemp())
    P = synth.make_params(H=H, seed=41)
    se, st, de = build_ref_nets(P, H)
    net = tmp / "net"; net.mkdir()
    torch.save(se, net / "speech_encoder.pt"); torch.save(de, net / "decoder.pt"); torch.save(st, net / "style_encoder.pt")
    _orig_load = torch.load
    torch.load = lambda *a, **k: _orig_load(*a, **{**k, "weights_only": False})       # generate.py:130-137 predates the new default
    out = {}
    try:
        for loud in (False, True):
            data = tmp / f"data{int(loud)}"; data.mkdir()
            stats = synth.load_stats()
            np.savez(data / "stats.npz", **{k: stats[k] for k in ("audio_input_mean", "audio_input_std", "anim_input_mean",
                                                                 "anim_input_std", "anim_output_mean", "anim_output_std")})
            pkg = os.path.join(os.path.dirname(GOLD), "..", "ubisoft-laforge-zeroeggs_b200", "data")
            shutil.copy(os.path.join(pkg, "data_definition_v1.json"), data / "data_definition.json")
            conf = json.load(open(os.path.join(pkg, "data_pipeline_conf_v1.json")))
            conf["audio_conf"]["normalize_loudness"] = loud
            json.dump(conf, open(data / "data_pipeline_conf.json", "w"))
            bvh_path = pathlib.Path(fx.make_synthetic_bvh(str(tmp / "style.bvh")))
            wav_path = pathlib.Path(fx.make_wav(str(tmp / "speech.wav")))
            cases = dict(one=dict(styles=[(bvh_path, (10, 300))]),
                         add=dict(styles=[(bvh_path, (10, 300)), (bvh_path, (150, 400))], blend_type="add", blend_ratio=[0.25, 0.75]),
                         stitch=dict(styles=[(bvh_path, (10, 300)), (bvh_path, None)], blend_type="stitch", blend_ratio=[0.5, 0.5]))
            for name, kw in cases.items():
                res = tmp / f"res{int(loud)}_{name}"
                enc = rgen.generate_gesture(wav_path, network_path=net, data_path=data, results_path=res, style_encoding_type="example",
                                            file_name="out", first_pose=None, temperature=1e6, seed=1234, use_gpu=False, **kw)
                b = rbvh.load(str(res / "out.bvh"))
                tag = f"loud{int(loud)}_{name}"
                out[tag + "_positions"] = b["positions"]; out[tag + "_rotations"] = b["rotations"]
                out[tag + "_encoding"] = enc.detach().numpy()
        # the embedding-only call (audio_file None) and a first_pose given as a path
        out["embedding_only"] = rgen.generate_gesture(None, [(bvh_path, (10, 300))], net, tmp / "data0", None, temperature=1e6, use_gpu=False).numpy()
    finally:
        torch.load = _orig_load
    out["H"] = H; out["param_seed"] = 41
    np.savez_compressed(os.path.join(GOLD, "generate_e2e.npz"), **out)
    print("generate_e2e golden:", {k: getattr(v, "shape", v) for k, v in out.items()})


def write_mel_clip_golden():
    """preprocess_audio (data_pipeline.py:33) on a 1.5 s clip resampled to 90 frames at 60 fps."""
    pa = ref_shim.ref_preprocess_audio()
    wav = synth.make_waveforms(1, 24000, seed=3)[0]
    feat = pa(wav, 60, 90, audio_params(200), ["mel_spec", "energy"])
    np.savez_compressed(os.path.join(GOLD, "mel_clip90.npz"), wav_seed=3, n_samples=24000, feat=feat)
    print("mel_clip90 golden written")


DATASET_CASES = [(64, 128), (100, 256), (64, 64)]      # (window, example_window_length)


def write_dataset_golden():
    """The reference SGDataset (dataset.py:9-204) on tests/_fixtures.write_processed_data: for 42 seeded windows per case, the
    window rows, range index and a fingerprint of each of the 11 tensors __getitem__ returns; and the one-hot labels of every
    window."""
    import tempfile
    from tests import _fixtures as fx
    ref_shim.install()
    import dataset as ref_dataset
    ddef, dproc = fx.write_processed_data(tempfile.mkdtemp())
    out = {}
    for window, ex_len in DATASET_CASES:
        ref = ref_dataset.SGDataset(ddef, dproc, window, "example", ex_len)
        rs = np.random.RandomState(window)
        idx = np.array(list(rs.randint(0, len(ref), size=40)) + [0, len(ref) - 1], dtype=np.int64)
        tag = f"w{window}_ex{ex_len}"
        out[tag + "_len"] = len(ref)
        out[tag + "_idx"] = idx
        out[tag + "_R"] = ref.R[idx].numpy()
        out[tag + "_S"] = ref.S[idx].numpy()
        out[tag + "_digest"] = np.array([[fx.digest(t.numpy()) for t in ref[int(i)]] for i in idx])
    out["label_w64_L"] = ref_dataset.SGDataset(ddef, dproc, 64, "label", 128).L.numpy()
    np.savez_compressed(os.path.join(GOLD, "dataset_windows.npz"), **out)
    print("dataset_windows golden written")


ANIM_KEYS = ["root_pos", "root_rot", "root_vel", "root_vrt", "lpos", "lrot", "ltxy", "lvel", "lvrt", "cpos", "crot", "ctxy", "cvel",
             "cvrt", "gaze_pos", "gaze_dir"]
ANIM_CUTS = {"full": None, "cut10_80": (10, 80)}
ANIM_SAMPLES = 128        # values kept per preprocess_animation output: a fixed seeded sample of its flat indices


def anim_sample_index(size, key):
    return np.random.RandomState(sum(map(ord, key))).randint(0, size, size=min(ANIM_SAMPLES, size))


def write_animation_io_golden():
    """The reference's BVH writer (anim/bvh.py:137) on seeded channels: the file it writes, byte for byte; its BVH loader
    (anim/bvh.py:4) and preprocess_animation (data_pipeline.py:90) on the 120-frame synthetic clip of tests/_fixtures.py:
    fingerprints of what the loader returns and, per preprocess_animation output, its shape, max |value| and a seeded sample."""
    import copy
    import tempfile
    from tests import _fixtures as fx
    ref_shim.install()
    from anim import bvh
    from data_pipeline import preprocess_animation as ref_pa
    tmp = tempfile.mkdtemp()
    d = fx.skeleton()
    rs = np.random.RandomState(0)
    pos = rs.randn(5, 75, 3).astype(np.float32); rot = (rs.randn(5, 75, 3) * 50).astype(np.float32)
    bvh.save(os.path.join(tmp, "a.bvh"), dict(order="zyx", offsets=pos[0], names=d["bone_names"], frametime=d["dt"],
                                              parents=np.array(d["parents"]), positions=pos, rotations=rot))
    with open(os.path.join(tmp, "a.bvh"), "rb") as f:
        out = {"writer_bvh": np.frombuffer(f.read(), dtype=np.uint8)}
    a_ref = bvh.load(fx.make_synthetic_bvh(os.path.join(tmp, "s.bvh"), frames=120))
    for k in ("rotations", "positions", "offsets", "parents"):
        out["load_" + k] = fx.digest(np.asarray(a_ref[k], dtype=np.float64))
    for tag, cut in ANIM_CUTS.items():
        ar = copy.deepcopy(a_ref)
        if cut:
            ar["rotations"], ar["positions"] = ar["rotations"][cut[0]:cut[1]], ar["positions"][cut[0]:cut[1]]
        for k, v in zip(ANIM_KEYS, ref_pa(ar)):
            v = np.asarray(v)
            out[f"{tag}_{k}_shape"] = np.array(v.shape)
            out[f"{tag}_{k}_absmax"] = np.float64(np.abs(v).max())
            out[f"{tag}_{k}_sample"] = v.reshape(-1)[anim_sample_index(v.size, k)]
    np.savez_compressed(os.path.join(GOLD, "animation_io.npz"), **out)
    print("animation_io golden written")


PICKLE_SIZES = dict(speech=(81, 8, 8), decoder=(1134, 1131, 8, 8, 16, 2), style=(1134, 16, 4))


def write_pickles_golden():
    """Whole-module pickles (torch.save of the module, as the reference's train.py saves its networks) of small instances of the
    reference's SpeechEncoder, Decoder and StyleEncoder, stored as the bytes of each file.  Only their layout matters to the test
    that loads them, so to keep them small every parameter is zero and the positional-encoding table the reference keeps as a
    plain attribute (20000 x embed_dim) is cut to its first 16 rows; zeggs_b200 recomputes that table."""
    import io
    m = ref_shim.ref_modules()
    sty = m.StyleEncoder(*PICKLE_SIZES["style"], type="attn", use_vae=True)
    sty.encoder.pos_enc.pos_enc = sty.encoder.pos_enc.pos_enc[:16].clone()
    out = {}
    for name, net in (("speech_encoder", m.SpeechEncoder(*PICKLE_SIZES["speech"])), ("decoder", m.Decoder(*PICKLE_SIZES["decoder"])),
                      ("style_encoder", sty)):
        with torch.no_grad():
            for p in net.parameters():
                p.zero_()
        buf = io.BytesIO()
        torch.save(net, buf)
        out[name] = np.frombuffer(buf.getvalue(), dtype=np.uint8)
    np.savez_compressed(os.path.join(GOLD, "pickles.npz"), **out)
    print("pickles golden written")


def write_pose_post_golden(T=40):
    """generate.py:389-406 + utils.write_bvh through the reference's own functions: what bvh.save receives for a synthetic clip."""
    ref_shim.install()
    import anim.bvh as rbvh
    import utils as rutils
    from anim import quat
    from anim.txform import xform_orthogonalize_from_xy
    w = synth.make_pose_windows(2, T, seed=3)
    rs = np.random.RandomState(0)
    ltxy = (w["ltxy"] + 0.05 * rs.randn(*w["ltxy"].shape)).astype(np.float32)          # not exactly orthonormal, like network output
    out = dict(root_pos=w["root_pos"], root_rot=w["root_rot"], lpos=w["lpos"], ltxy=ltxy)
    cap = {}
    orig = rbvh.save
    rutils.bvh.save = lambda fn, d: cap.update(d)
    try:
        for n in range(2):
            lrot = quat.from_xform(xform_orthogonalize_from_xy(torch.from_numpy(ltxy[n])).numpy())
            rutils.write_bvh("unused", w["root_pos"][n], w["root_rot"][n], w["lpos"][n], lrot, parents=synth.load_stats()["parents"],
                             names=None, order="zyx", dt=1 / 60, start_position=np.array([0, 0, 0]), start_rotation=np.array([1, 0, 0, 0]))
            out[f"positions{n}"] = np.asarray(cap["positions"]); out[f"rotations{n}"] = np.asarray(cap["rotations"]); out[f"lrot{n}"] = lrot
    finally:
        rutils.bvh.save = orig
    np.savez_compressed(os.path.join(GOLD, "pose_post.npz"), **out)
    print("pose_post golden written")


REFERENCE_IO = dict(mel_clip=write_mel_clip_golden, dataset=write_dataset_golden, animation_io=write_animation_io_golden,
                    pickles=write_pickles_golden)


if __name__ == "__main__":
    import sys
    main(only=sys.argv[1:] or None)
