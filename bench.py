#!/usr/bin/env python
"""Headline benchmark: frames/sec of the ZeroEGGS train step (60 fps, 75-joint pose frames per optimizer step).

    python bench.py --gpus N --steps K --warmup W            # N>1: launched by torchrun, one rank per GPU
    python bench.py --impl reference ...                     # the CPU implementation of the same path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

Prints ONE JSON line (rank 0).  `value` = whole-job frames/s with the batch resident in HBM; `e2e` = the same metric
through TrainStep.step() with pinned HOST batches (H2D of every input + D2H of the loss inside the timed region).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    # BASELINE.json configs[1] "train.py configs_v1 ... 1xB200": the reference-actual configs_v1 sizes (SURVEY.md top note)
    "train_v1": dict(B=32, T=256, H=1024, T_ex=384, desc="train.py configs_v1 (reference-actual: batch 32 x 256-frame windows, "
                     "decoder hidden 1024, example style T_ex=384 = mean of the reference's 256..512 draw)"),
    # the sizes BASELINE.json states in words for the same config
    "train_v1_stated": dict(B=16, T=120, H=512, T_ex=256, desc="train.py configs_v1 as worded in BASELINE.json (batch 16 x 120-frame windows, hidden 512)"),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=0.5)
        except Exception:
            try:
                self.proc.kill()          # a lingering nvidia-smi poller would keep contending for the driver lock
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=(statistics.median(sm) if sm else None), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def synth_batch(B, T, T_ex, seed, device=None, pinned=False, label_Z=0):
    from zeggs_b200 import synth
    b = {k: torch.from_numpy(v) for k, v in synth.make_pose_windows(B, T, seed=seed).items()}
    b["audio"] = torch.from_numpy(synth.make_audio_features(B, T, seed=seed))
    if label_Z:
        lab = torch.zeros(B, label_Z)
        lab[torch.arange(B), torch.arange(B) % label_Z] = 1.0
        b["style"] = lab
    else:
        b["style"] = torch.from_numpy(synth.make_style_example(B, T_ex, seed=seed))
    if pinned:
        return {k: v.pin_memory() for k, v in b.items()}
    if device is not None:
        return {k: v.to(device) for k, v in b.items()}
    return b


def build_stepper(H, device, world, seed=1234, use_graph=True, label_Z=0):
    from zeggs_b200 import modules, synth
    from zeggs_b200.train import TrainStep
    Z = label_Z or 64
    P = synth.make_params(H=H, Z=Z, seed=seed, with_style=not label_Z)
    ld = lambda m, pre: (m.load_state_dict({k[len(pre):]: torch.from_numpy(v) for k, v in P.items() if k.startswith(pre)}), m.to(device))[1]
    se = ld(modules.SpeechEncoder(81, 64, 64), "speech_encoder.")
    st = None if label_Z else ld(modules.StyleEncoder(1134, 512, 64, type="attn", use_vae=True), "style_encoder.")
    de = ld(modules.Decoder(1134, 1131, 64, Z, H, 2), "decoder.")
    stats = synth.load_stats()
    return TrainStep(se, de, st, stats, stats["parents"], float(stats["dt"]), world_size=world, use_graph=use_graph), P, stats


def decoder_flops_per_frame(H, C=128):
    """SURVEY.md 8(d): MACs of one decoder step per sample (layer0, GRU l0 ih/hh, GRU l1 ih+hh, layer2)."""
    A = 1134 + C
    mac = A * H + 3 * H * (A + H) + 3 * H * H + 6 * H * H + H * 1131
    return 2 * mac


DUMP_SAMPLE = 1 << 21      # entries of the flat parameter / gradient vectors written by --dump-outputs


def dump_outputs(d, stepper, loss):
    """What the caller of the timed train step receives from its last step: the loss, the loss terms and, as the step's effect on
    the model, the updated parameters and the gradients they were updated with.  The two flat vectors hold ~25.5 M values each
    at the default workload, so both are written as the same fixed seeded sample of DUMP_SAMPLE indices (sorted)."""
    os.makedirs(d, exist_ok=True)
    p, g = stepper.optimizer.flat_param, stepper.optimizer.flat_grad
    n = p.numel()
    idx = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.RandomState(0).randint(0, n, size=DUMP_SAMPLE))
    idx = torch.from_numpy(idx).to(p.device)
    out = dict(loss=loss, loss_terms=stepper.terms, params_sample=p[idx], grads_sample=g[idx])
    for name, v in out.items():
        np.save(os.path.join(d, name + ".npy"), v.detach().float().cpu().numpy())


SPANS = ("decoder_fwd", "decoder_bwd", "decoder_wgrad", "loss", "encoders_fwd", "encoders_bwd", "optimizer", "weight_pack")


def read_spans(lib):
    import ctypes as C
    out = {}
    for name in SPANS:
        tot, cnt = C.c_double(0), C.c_int(0)
        lib.zeggs_timing_read(name.encode(), C.byref(tot), C.byref(cnt))
        out[name] = (tot.value, cnt.value)
    return out


def run_ours(args):
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); lrank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    device = torch.device("cuda", lrank)
    torch.cuda.set_device(device)
    from zeggs_b200.train import pin_to_gpu_numa
    numa = pin_to_gpu_numa(lrank) if args.pin else None    # the launch thread next to its GPU (GPUs 4-7 hang off the second socket)
    try:
        os.nice(-10)                      # the launch thread competes with other tenants' all-core CPU jobs on a shared node
    except Exception:
        pass
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=device)
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        torch.distributed.barrier()
    from zeggs_b200 import _lib, ops
    lib = _lib.lib()
    ops.set_decoder_engine(args.engine)
    wl = WORKLOADS[args.workload]
    B, T, H, T_ex = wl["B"], wl["T"], wl["H"], wl["T_ex"]
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    def measure(B, T, H, T_ex, K, W, timing=False, label_Z=0):
        # dropout masks and VAE noise come from torch's generators, whose default seed changes from process to process: seeded
        # here, runs with the same arguments compute the same steps
        torch.manual_seed(1234)
        stepper, P, stats = build_stepper(H, device, world, use_graph=bool(args.graph), label_Z=label_Z)
        dbatch = synth_batch(B, T, T_ex, seed=100 + rank, device=device, label_Z=label_Z)
        graphed = bool(args.graph)
        # step 1 runs eagerly (first sight of the geometry), step 2 captures the CUDA graph(s); with `timing` the library's span
        # events are recorded INTO the graph as external event-record nodes, so every replay re-records them
        stepper.step(dbatch)
        if timing:
            lib.zeggs_timing_reset(); lib.zeggs_timing_enable(1)
        stepper.step(dbatch)
        graphed = graphed and stepper.use_graph and len(stepper._graphs) > 0
        if timing and graphed:
            lib.zeggs_timing_enable(0)          # no new spans: the captured pairs are re-recorded by each replay
        for _ in range(max(W - 2, 1)):
            stepper.step(dbatch)
        barrier()
        sampler = ClockSampler(lrank)
        if rank == 0 and timing:
            sampler.start()
        if timing:
            # nvidia-smi needs ~0.1-0.3 s to start reporting: every rank keeps its GPU under the same load meanwhile (untimed)
            for _ in range(24):
                stepper.step(dbatch)
            barrier()
            if not graphed:
                lib.zeggs_timing_reset()
        if world > 1:
            stepper.ar_events = []
        n0 = lib.zeggs_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_host0 = time.perf_counter()
        e0.record()
        for _ in range(K):
            loss = stepper.step(dbatch)
        e1.record()
        host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / K
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1))
        host_enqueue_ms = max_over_ranks(host_enqueue_ms)
        launches = int(lib.zeggs_launch_count() - n0) if not graphed else stepper.graph_launches * K
        ar_ms = None
        if world > 1 and stepper.ar_events:
            ar_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in stepper.ar_events) / len(stepper.ar_events))
        stepper.ar_events = None
        clocks = sampler.stop() if (rank == 0 and timing) else None
        if timing and rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, stepper, loss)
        if clocks is not None:
            clocks["note"] = "nvidia-smi every 200 ms from the start of 24 untimed warm steps of the same loop through the timed region"
        spans, span_src = {}, None
        if timing:
            if graphed:
                # the last timed replay's spans are readable now; average over K more synchronised replays of the same graph
                acc = {n: [0.0, 0] for n in SPANS}
                for _ in range(K):
                    stepper.step(dbatch)
                    torch.cuda.synchronize()
                    for n, (tot, cnt) in read_spans(lib).items():
                        acc[n][0] += tot; acc[n][1] = cnt
                spans = {n: dict(ms_per_step=v[0] / K, launches=v[1]) for n, v in acc.items()}
                span_src = "CUDA events recorded inside the replayed graph (external event-record nodes), mean of K synchronised replays after the timed region"
            else:
                lib.zeggs_timing_enable(0)
                spans = {n: dict(ms_per_step=tot / max(K, 1), launches=cnt) for n, (tot, cnt) in read_spans(lib).items()}
                span_src = "CUDA events on the launching stream over the timed region (eager launches)"
        # end to end: pinned host batch -> H2D every step, loss read back every step
        hbatch = synth_batch(B, T, T_ex, seed=200 + rank, pinned=True, label_Z=label_Z)
        h2d = sum(v.numel() * v.element_size() for v in hbatch.values())
        # the public input pipeline (zeggs_b200.data.DevicePrefetcher, used by train()): every step's batch is copied from pinned
        # host memory inside the timed region, on a side stream, while the previous step's kernels run
        # ... and every step's loss is read back (4 bytes) through the package's LaggedScalarReader: the value of step i reaches the
        # host while step i+1 runs (all K values are on the host before the clock stops)
        from zeggs_b200.data import DevicePrefetcher, LaggedScalarReader
        pf = DevicePrefetcher(device)
        for _ in range(2):
            stepper.step(pf.acquire(pf.upload(hbatch))).item()
        barrier()
        rd = LaggedScalarReader(device, lag=int(os.environ.get("ZEGGS_BENCH_LOSS_LAG", "1")))
        got = []
        # steady state of the input pipeline: the batch of the first timed step is already in flight when the clock starts and the
        # batch of step K+1 is uploaded during step K, so exactly K host->device copies (one per step) run inside the timed region
        tok = pf.upload(hbatch)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            db = pf.acquire(tok)
            tok = pf.upload(hbatch)
            got += rd.push(stepper.step(db))
        got += rd.drain()
        torch.cuda.synchronize()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        assert len(got) == K and all(np.isfinite(got)), got
        barrier()
        r = dict(ms=ms, e2e_ms=e2e_ms, launches=launches, clocks=clocks, spans=spans, span_src=span_src, h2d=h2d, loss=float(loss.item()),
                 P=P, stats=stats, graphed=graphed, host_enqueue_ms=host_enqueue_ms, ar_ms=ar_ms)
        del stepper
        torch.cuda.empty_cache()
        return r

    if os.environ.get("ZEGGS_TC_GEMM_VARIANT"):          # experiment knob (profiles/r02_tc_gemm_variants.md)
        lib.zeggs_debug_set_tc_gemm_variant(int(os.environ["ZEGGS_TC_GEMM_VARIANT"]))
    r = measure(B, T, H, T_ex, K, W, timing=True)
    frames = world * B * T
    value = frames / (r["ms"] / K) * 1e3
    peaks = load_peaks()
    # roofline of the dominant kernel (the slower of the two persistent recurrence kernels): algorithmic FLOPs = the
    # (transposed) GEMMs of every step
    fl_step = decoder_flops_per_frame(H) - 2 * 128 * 4 * H          # the speech/style columns are hoisted out of the recurrence
    dom = "decoder_bwd" if r["spans"]["decoder_bwd"]["ms_per_step"] >= r["spans"]["decoder_fwd"]["ms_per_step"] else "decoder_fwd"
    dom_ms = r["spans"][dom]["ms_per_step"]
    achieved = fl_step * B * (T - 1) / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0
    wbytes = (fl_step / 2) * (2 if args.engine != "fp32" else 4)    # operand bytes streamed per step: bf16 images (tc) / fp32 (SIMT), L2 resident
    roofline = dict(bound="tensor", kernel=(f"{dom}_tc_kernel" if args.engine != "fp32" else f"{dom}_kernel"), achieved=round(achieved, 3), peak=peaks["bf16_tflops_sustained"],
                    unit="TFLOP/s", frac=round(achieved / peaks["bf16_tflops_sustained"], 5), traffic=None,
                    peak_source=peaks["src"] + " (cuBLAS bf16, sustained)", ms_per_launch=round(dom_ms, 3),
                    timing_source=r["span_src"],
                    weight_stream_gbs=round(wbytes * (T - 1) / (dom_ms * 1e-3) / 1e9, 1),
                    note=("decoder forward and BPTT recurrences on tcgen05 (bf16 operands from smem images, fp32 accumulators in TMEM, fp32 state; "
                          "forward: layer 2 folded into the next step's input GEMM -> 3 all-to-all exchanges per step, M=64 MMAs, one mbarrier wait per 16 MMAs); "
                          "weight-gradient GEMMs tcgen05 bf16, encoder GEMMs tcgen05 split-bf16; B=32 rows per step: the recurrences are bound by operand "
                          "delivery per SM, grid-barrier latency and MMA issue, not by tensor peak; "
                          if args.engine != "fp32" else "fp32 SIMT recurrence; batched GEMMs tcgen05 split-bf16; ") +
                         "per-step arithmetic intensity at B=32 is 32 FLOP per bf16 operand byte (weight streaming from L2), see DESIGN.md")
    for tname in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        tp = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tp) and args.workload == "train_v1":
            try:
                tr = json.load(open(tp)).get(roofline["kernel"])
                if tr:
                    roofline["traffic"] = tr["dram_bytes_per_launch"]
                    roofline["traffic_source"] = tr["source"]
                    break
            except Exception:
                pass
    kms = {k: round(v["ms_per_step"], 3) for k, v in r["spans"].items()}
    if r["ar_ms"] is not None:
        kms["allreduce"] = round(r["ar_ms"], 3)
    out = dict(metric="frames/sec (train step, 60fps 75-joint pose)", value=round(value, 1), unit="frames/s", n_gpus=world, steps=K, warmup=W,
               ms_per_step=round(r["ms"] / K, 3), higher_is_better=True, scaling="weak", vs_baseline=None,
               dtype=("bf16" if args.engine != "fp32" else "f32"), data="synthetic",
               config=dict(workload=wl["desc"], per_gpu_batch=B, global_batch=world * B, window=T, hidden=H, style_example_len=T_ex,
                           parallelism=f"dp{world}", decoder_engine=args.engine, cuda_graph=r["graphed"], numa_node=numa,
                           lanes=(os.environ.get("ZEGGS_LANES", "1") == "1"),
                           l2="per-step working set ~1.4 GB of saved activations >> 126 MB L2 (no explicit flush)"),
               e2e=dict(value=round(frames / (r["e2e_ms"] / K) * 1e3, 1), unit="frames/s", h2d_bytes_per_step=r["h2d"], d2h_bytes_per_step=4),
               gpu_launches=r["launches"], host_enqueue_ms_per_step=round(r["host_enqueue_ms"], 3), clocks=r["clocks"], roofline=roofline,
               kernel_ms_per_step=kms,
               kernel_ms_note=("spans are per library call on the stream it was issued on; with lanes the two encoders (forward) and "
                               "encoders_bwd / decoder_wgrad (backward) run concurrently on three streams, so those spans overlap in time "
                               "and their sum exceeds the step"),
               loss=r["loss"])
    if args.alt and args.workload == "train_v1":
        a = WORKLOADS["train_v1_stated"]
        ra = measure(a["B"], a["T"], a["H"], a["T_ex"], K, W)
        out["alt_config"] = dict(workload=a["desc"], value=round(world * a["B"] * a["T"] / (ra["ms"] / K) * 1e3, 1), unit="frames/s",
                                 ms_per_step=round(ra["ms"] / K, 3),
                                 e2e=round(world * a["B"] * a["T"] / (ra["e2e_ms"] / K) * 1e3, 1))
    if args.extras and args.workload == "train_v1":
        try:
            out["other_configs"] = run_extras(args, device, world, rank, peaks, measure, barrier, max_over_ranks)
        except Exception as e:                      # an auxiliary config must never take the headline line down
            out["other_configs"] = dict(error=f"{type(e).__name__}: {e}")
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle.train_oracle import measure_cpu_train
        cb = measure_cpu_train(r["P"], r["stats"], lambda b, t, tx: synth_batch(b, t, tx, seed=300), B, T, T_ex, steps=3, warmup=1,
                               budget_s=45.0)
        out["cpu_baseline"] = dict(value=round(cb["value"], 1), unit="frames/s", cores=cb["cores"], kind="port",
                                   sample=cpu_sample_text(cb, H), sweep_frames_per_s=cb["sweep"], step_seconds=cb["step_s"], spread=cb["spread"],
                                   same_config=cb["same_config"])
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        torch.distributed.destroy_process_group()


def cpu_sample_text(cb, H):
    return (f"{len(cb['step_s'])} timed CPU train steps (oracle port of train.py:196-432) at B={cb['B']}, T={cb['T']}, H={H}, T_ex={cb['T_ex']} "
            f"with {cb['cores']} threads{' pinned to NUMA node 0' if cb['pinned_node0'] else ''} = best of the thread sweep {cb['sweep']} "
            f"(frames/s at a 32-frame window); os.cpu_count()={os.cpu_count()}")


def run_extras(args, device, world, rank, peaks, measure, barrier, max_over_ranks):
    """BASELINE.json configs 1, 3, 4, 5 next to the headline (config 2): each with the bound that applies to it."""
    from zeggs_b200 import audio, generate, modules, ops, synth
    from tests._util import NAMES
    res = {}
    stats = synth.load_stats()
    st = {k: torch.as_tensor(stats[k], dtype=torch.float32, device=device) for k in
          ("anim_input_mean", "anim_input_std", "anim_output_mean", "anim_output_std")}

    def timed(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    # ---- config 5: batch inference, 64 concurrent 60 s clips, sharded 64/N per GPU, no collective (frames generated per second)
    from zeggs_b200 import dp
    lo, hi = dp.shard_range(64, rank, world)
    Bi, Ti, Hi = hi - lo, 3600, 1024
    P = synth.make_params(H=Hi, seed=1, with_style=False)
    dec = modules.Decoder(1134, 1131, 64, 64, Hi, 2)
    dec.load_state_dict({k[len("decoder."):]: torch.from_numpy(v) for k, v in P.items() if k.startswith("decoder.")})
    dec = dec.to(device).eval()
    win = {k: torch.from_numpy(v).to(device) for k, v in synth.make_pose_windows(Bi, 2, seed=1 + rank).items()}
    g = torch.Generator(device="cpu").manual_seed(5 + rank)
    speech = (torch.randn(Bi, Ti, 64, generator=g) * 0.5).to(device)
    style = torch.randn(Bi, 1, 64, generator=g).to(device).repeat(1, Ti, 1)
    gaze = win["gaze_pos"][:, :1].repeat(1, Ti, 1)
    dargs = [win[n][:, 0] for n in NAMES] + [gaze, speech, style, None, st["anim_input_mean"], st["anim_input_std"],
                                             st["anim_output_mean"], st["anim_output_std"], float(stats["dt"])]
    with torch.no_grad():
        barrier()
        ms = max_over_ranks(timed(lambda: dec(*dargs), reps=3, warm=1))
    fl = decoder_flops_per_frame(Hi) * 64 * (Ti - 1)
    res["batch_inference_64x60s"] = dict(
        config=f"BASELINE config 5: 64 clips x {Ti} frames (60 s), H={Hi}, {Bi} clips per GPU, no collective", ms=round(ms, 2),
        value=round(64 * (Ti - 1) / ms * 1e3, 1), unit="generated frames/s", engine=args.engine,
        roofline=dict(bound="tensor", achieved=round(fl / (ms * 1e-3) / 1e12 / world, 3), unit="TFLOP/s per GPU", peak=peaks["bf16_tflops_sustained"],
                      frac=round(fl / (ms * 1e-3) / 1e12 / world / peaks["bf16_tflops_sustained"], 5)))
    if world > 1:
        return res
    # ---- config 1: one 10 s clip (B=1, T=600), wav -> mel -> encoders -> free-running decoder; latency through generate_motion
    Pg = synth.make_params(H=1024, seed=77)
    ld = lambda m, pre: (m.load_state_dict({k[len(pre):]: torch.from_numpy(v) for k, v in Pg.items() if k.startswith(pre)}), m.to(device).eval())[1]
    nets = dict(speech_encoder=ld(modules.SpeechEncoder(81, 64, 64), "speech_encoder."),
                style_encoder=ld(modules.StyleEncoder(1134, 512, 64, type="attn", use_vae=True), "style_encoder."),
                decoder=ld(modules.Decoder(1134, 1131, 64, 64, 1024, 2), "decoder."))
    wav1 = synth.make_waveforms(1, 160000, seed=9)[0]
    ex = synth.make_style_example(1, 600, seed=9)[0]
    w2 = synth.make_pose_windows(1, 2, seed=9)
    fp = {k: w2[k][0, 0] for k in NAMES}
    from types import SimpleNamespace
    ac = SimpleNamespace(sampling_rate=16000, filter_length=800, hop_length=200, n_mel_channels=80, mel_fmin=20, mel_fmax=7600, min_clipping=1e-5,
                         pre_emphasis=False, pre_emph_coeff=0.97, real_amplitude=True, centered=True, normalize_mel_bins=True, normalize_range=True,
                         resample_method="linear", normalize_loudness=False)
    gen = {}
    for eng in ("tc", "fp32"):
        ops.set_decoder_engine(eng)
        def one():
            out, _ = generate.generate_motion(nets, stats, ac, wav1, ex, fp, w2["gaze_pos"][0, 0], float(stats["dt"]), device=device)
            return out[0].cpu()            # the pose leaves the device (the caller writes a BVH from it)
        one(); torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter(); one(); ts.append((time.perf_counter() - t0) * 1e3)
        gen[eng] = dict(latency_ms=round(float(np.median(ts)), 2), frames_per_s=round(599 / float(np.median(ts)) * 1e3, 1))
    ops.set_decoder_engine(args.engine)
    res["generate_10s_clip"] = dict(config="BASELINE config 1: B=1, T=600 (10 s WAV @16 kHz -> mel -> SpeechEncoder, StyleEncoder on a 600-frame example, "
                                           "free-running decoder H=1024), host wall-clock through generate_motion incl. H2D of the wav and D2H of the pose", **gen)
    # ---- config 3: mel front end, 1024 x 10 s clips, hop 200 (reference-actual) and hop 160 (as worded)
    wav = torch.from_numpy(synth.make_waveforms(8, 160000, seed=1)).to(device).repeat(128, 1)
    mel = {}
    for hop in (200, 160):
        fe = audio.MelFrontEnd(device, hop_length=hop)
        L = fe.num_frames(160000)
        for mode in ("mel", "feat60"):
            fn = (lambda: fe.forward(wav, 60, 600)) if mode == "feat60" else (lambda: fe.forward(wav, want_mel=True, want_feat=False))
            ms = timed(fn, reps=10, warm=3)
            byt = wav.numel() * 4 + (wav.shape[0] * 600 * 81 * 4 if mode == "feat60" else wav.shape[0] * 80 * L * 4)
            mel[f"hop{hop}_{mode}"] = dict(ms=round(ms, 3), clips_per_s=round(wav.shape[0] / ms * 1e3), frames=L,
                                           roofline=dict(bound="hbm", achieved=round(byt / ms / 1e6, 1), unit="GB/s", peak=peaks["hbm_gbs"],
                                                         frac=round(byt / ms / 1e6 / peaks["hbm_gbs"], 4), algorithmic_bytes=byt))
    res["mel_1024x10s"] = dict(config="BASELINE config 3: 1024 x 160000-sample clips, n_fft 800, 80 mels; 'mel' = [80,L] dB-normalised spectrogram out, "
                                      "'feat60' = fused 60 fps [600,81] features out (what preprocess_audio returns)", **mel)
    del wav
    torch.cuda.empty_cache()
    # ---- config 4 geometry: label style (Z=9, no style encoder), per-GPU batch 32 (global 256 on 8 GPUs under --gpus 8 of the headline)
    rv = measure(32, 256, 1024, 0, args.steps, args.warmup, label_Z=9)
    res["train_v2_label_style"] = dict(config="BASELINE config 4 geometry on this GPU count: configs_v2 label style Z=9 (A=1207), B=32 per GPU, T=256, H=1024",
                                       value=round(32 * 256 / (rv["ms"] / args.steps) * 1e3, 1), unit="frames/s", ms_per_step=round(rv["ms"] / args.steps, 3),
                                       e2e=round(32 * 256 / (rv["e2e_ms"] / args.steps) * 1e3, 1), cuda_graph=rv["graphed"])
    return res


def run_reference(args):
    """The CPU implementation of the same path (oracle port; the Python reference cannot travel to the GPU box): real batch size,
    thread sweep pinned to one NUMA node, best thread count, full window when the run fits the budget."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.train_oracle import measure_cpu_train
    from zeggs_b200 import synth
    wl = WORKLOADS[args.workload]
    B, T, H, T_ex = wl["B"], wl["T"], wl["H"], wl["T_ex"]
    P = synth.make_params(H=H, seed=1234)
    stats = synth.load_stats()
    K, W = max(args.steps, 1), max(args.warmup, 0)      # >= 3 timed steps recommended (the spread is reported)
    cb = measure_cpu_train(P, stats, lambda b, t, tx: synth_batch(b, t, tx, seed=300), B, T, T_ex, steps=K, warmup=W, budget_s=150.0)
    fps = cb["value"]
    sample = cpu_sample_text(cb, H)
    med = sorted(cb["step_s"])[len(cb["step_s"]) // 2]
    print(json.dumps(dict(impl="reference", metric="frames/sec (train step, 60fps 75-joint pose)", value=round(fps, 1), unit="frames/s",
                          n_gpus=args.gpus, steps=K, warmup=W, ms_per_step=round(med * 1e3, 2), higher_is_better=True, scaling="weak",
                          vs_baseline=None, dtype="f32", data="synthetic",
                          config=dict(workload=wl["desc"], per_gpu_batch=cb["B"], window=cb["T"], hidden=H, style_example_len=cb["T_ex"], sample=sample,
                                      same_config=cb["same_config"]),
                          cpu_baseline=dict(value=round(fps, 1), unit="frames/s", cores=cb["cores"], kind="port", sample=sample,
                                            sweep_frames_per_s=cb["sweep"], step_seconds=cb["step_s"], spread=cb["spread"]),
                          e2e=dict(value=round(fps, 1), unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train_v1", choices=list(WORKLOADS))
    ap.add_argument("--alt", type=int, default=1, help="also time the BASELINE.json-worded sizes (reported under alt_config)")
    ap.add_argument("--extras", type=int, default=1, help="also time BASELINE configs 1, 3, 4, 5 (reported under other_configs)")
    ap.add_argument("--graph", type=int, default=1, help="replay the train step from CUDA graphs (0: eager launches)")
    ap.add_argument("--pin", type=int, default=1, help="bind the launch thread to the CPUs of the GPU's NUMA node")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--engine", default="tc", choices=["tc", "fp32", "auto"], help="decoder recurrence engine: tcgen05 bf16 (default) or fp32 SIMT")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32): loss, loss_terms, and a "
                         "fixed seeded sample of the updated parameters (params_sample) and of their gradients (grads_sample)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA train step (--impl ours)")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
