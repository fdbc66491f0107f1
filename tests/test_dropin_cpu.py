"""Drop-in surface checks that need no GPU: class names / constructor signatures / state-dict keys match the reference,
and the reference's whole-module pickles un-pickle into zeggs_b200.modules classes when it is registered as `modules`."""
import sys

import torch

from zeggs_b200 import modules, synth


def test_state_dict_keys_and_shapes_match_reference_layout():
    P = synth.make_params(H=1024, seed=0)
    nets = dict(speech_encoder=modules.SpeechEncoder(81, 64, 64), decoder=modules.Decoder(1134, 1131, 64, 64, 1024, 2),
                style_encoder=modules.StyleEncoder(1134, 512, 64, type="attn", use_vae=True))
    for name, net in nets.items():
        sd = net.state_dict()
        want = {k[len(name) + 1:]: v.shape for k, v in P.items() if k.startswith(name + ".")}
        assert set(sd) == set(want), (name, set(sd) ^ set(want))
        for k, shp in want.items():
            assert tuple(sd[k].shape) == tuple(shp), (name, k)
    assert sum(p.numel() for n in nets.values() for p in n.parameters()) == 25543147      # SURVEY.md 8a (a13)
    d = nets["decoder"]
    assert (d.hidden_size, d.speech_encoding_size, d.style_encoding_size) == (1024, 64, 64)


def test_reference_pickles_unpickle_into_our_classes(golden_dir):
    """Whole-module pickles written by the reference's own classes (tests/golden/pickles.npz, oracle/make_golden.py pickles; small
    instances of the shipped checkpoints' classes) load as zeggs_b200.modules classes when it is registered as `modules`."""
    import io
    import os
    import numpy as np
    from oracle.make_golden import PICKLE_SIZES
    g = np.load(os.path.join(golden_dir, "pickles.npz"))
    load = lambda name: torch.load(io.BytesIO(g[name].tobytes()), map_location="cpu", weights_only=False)
    saved = sys.modules.get("modules")
    sys.modules["modules"] = modules            # what INTEGRATION.md tells a maintainer to do
    try:
        dec, enc, sty = load("decoder"), load("speech_encoder"), load("style_encoder")
    finally:
        if saved is not None:
            sys.modules["modules"] = saved
        else:
            del sys.modules["modules"]
    assert type(dec) is modules.Decoder and type(enc) is modules.SpeechEncoder and type(sty) is modules.StyleEncoder
    _, _, S, Z, H, _ = PICKLE_SIZES["decoder"]
    assert (dec.hidden_size, dec.speech_encoding_size, dec.style_encoding_size) == (H, S, Z)
    assert len(dec._weights()) == 18 and len(enc._weights()) == 6 and len(sty._weights()) == 20
    assert sty.encoder.pos_enc.table(5).shape == (5, 2 * PICKLE_SIZES["style"][2])


def test_lane_context_is_scoped_and_nestable():
    """ops.lane selects which zeggs_ctx (GEMM scratch) the calls issued inside the block travel with: default "main", restored on exit,
    also when the block raises; nested lanes restore the outer one."""
    from zeggs_b200 import ops
    assert ops.current_lane() == "main"
    with ops.lane("speech"):
        assert ops.current_lane() == "speech"
        with ops.lane("style"):
            assert ops.current_lane() == "style"
        assert ops.current_lane() == "speech"
    assert ops.current_lane() == "main"
    try:
        with ops.lane("style"):
            raise RuntimeError("x")
    except RuntimeError:
        pass
    assert ops.current_lane() == "main"

