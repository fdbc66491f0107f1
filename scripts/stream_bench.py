"""Streaming generator throughput: H = 1024 synthetic weights, sessions x chunk sizes, each session fed 60 s of audio one chunk of
samples per step (as fast as the generator accepts it).  Per configuration: device ms per step() (CUDA events around each call),
host ms per step() (the call's own wall time: Python, ctypes and launch enqueue), wall ms per step (pushes + step, synchronised),
generated frames/s, real-time factor (audio seconds per wall second, summed over sessions, and per session: above 1 the load is
sustained in real time), the rule's algorithmic lookahead and the feature-recompute factor ((context + chunk) / chunk).  JSON to
--out, with the card's name and power limit read in the same run.

    python scripts/stream_bench.py --out /tmp/stream_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 else ("?", "?")
    return dict(gpu=name, power_limit=power)


def run(nets, st, conf, clips, n_sessions, chunk, warmup, engine):
    from zeggs_b200 import ops, streaming, synth
    ops.set_decoder_engine(engine)
    dev = torch.device("cuda")
    gen = streaming.StreamingGenerator(nets, st, conf, chunk_frames=chunk, device=dev)
    ex = synth.make_style_example(1, 120, seed=3)[0]
    win = synth.make_pose_windows(1, 2, seed=3)
    fp = {k: win[k][0, 0] for k in streaming.POSE_KEYS}
    sids = [gen.open(ex, fp, win["gaze_pos"][0, 0], float(st["dt"]), eps=torch.zeros(1, 64, device=dev)) for _ in range(n_sessions)]
    piece = chunk * 16000 // 60
    n_pieces = clips.shape[1] // piece
    dev_ms, host_ms, steps, frames = [], [], 0, 0
    t_start = None
    for p in range(n_pieces):
        if p == warmup:
            torch.cuda.synchronize()
            t_start = time.perf_counter()
        for i, sid in enumerate(sids):
            gen.push(sid, clips[i % clips.shape[0], p * piece:(p + 1) * piece])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        h0 = time.perf_counter()
        out = gen.step()
        h1 = time.perf_counter()
        e1.record()
        if p >= warmup:
            host_ms.append((h1 - h0) * 1e3)
            dev_ms.append((e0, e1))
            steps += 1
            frames += sum(o[0].shape[1] for o in out.values())
    torch.cuda.synchronize()
    wall = time.perf_counter() - t_start
    for sid in sids:
        gen.close(sid)
    dms = [a.elapsed_time(b) for a, b in dev_ms]
    audio_s = frames / 60.0
    return dict(engine=engine, sessions=n_sessions, chunk_frames=chunk, steps=steps, frames=frames,
                device_ms_per_step=float(np.mean(dms)), device_ms_per_step_p90=float(np.percentile(dms, 90)),
                host_ms_per_step=float(np.mean(host_ms)), wall_ms_per_step=wall * 1e3 / steps,
                frames_per_s=frames / wall, realtime_factor=audio_s / wall, per_session_realtime_factor=audio_s / wall / n_sessions,
                lookahead_ms=gen.lookahead_seconds * 1e3, recompute_factor=gen.recompute_factor,
                window_samples=gen.n_window, window_frames=gen.window_frames)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--sessions", default="1,8,32,64")
    ap.add_argument("--chunks", default="6,15,30")
    ap.add_argument("--warmup", type=int, default=5, help="steps left out of the timing (module loads, first chunks)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_bench.py measures the GPU path: no CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    from oracle.make_golden import audio_params
    from zeggs_b200 import modules, synth
    H = 1024
    P = synth.make_params(H=H, seed=1)
    dev = torch.device("cuda")

    def load(m, prefix):
        m.load_state_dict({k[len(prefix):]: torch.from_numpy(v) for k, v in P.items() if k.startswith(prefix)})
        return m.to(dev).eval()
    nets = dict(speech_encoder=load(modules.SpeechEncoder(81, 64, 64), "speech_encoder."),
                style_encoder=load(modules.StyleEncoder(1134, 512, 64, type="attn", use_vae=True), "style_encoder."),
                decoder=load(modules.Decoder(1134, 1131, 64, 64, H, 2), "decoder."))
    st = synth.load_stats()
    conf = audio_params(200)
    sessions = [int(s) for s in args.sessions.split(",")]
    clips = synth.make_waveforms(min(8, max(sessions)), int(16000 * args.seconds), seed=11)   # sessions share 8 distinct clips
    info = gpu_info()
    lines = []
    configs = [("tc", n, c) for n in sessions for c in (int(c) for c in args.chunks.split(","))] + [("fp32", 1, 30)]
    for eng, n, c in configs:
        r = run(nets, st, conf, clips, n, c, args.warmup, eng)
        r.update(info)
        print(json.dumps(r), flush=True)
        lines.append(r)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(dict(H=H, audio_seconds=args.seconds, results=lines, **info), f, indent=1)


if __name__ == "__main__":
    main()
