#!/usr/bin/env python
"""bench.py -- Kokoro-82M TTS audio-seconds synthesised per wall-second on N B200s (BASELINE.json metric).

Workload (BASELINE.json configs[1], SURVEY.md section 8d cfg2): one 128-phoneme utterance (T = 130 tokens with BOS/EOS) through the
model's OWN duration head (3 frames / token on the synthetic checkpoint -> F = 390 frames -> 234 000 samples = 9.75 s of 24 kHz
audio), synthetic bf16 checkpoint at the real Kokoro-82M shapes (81.8 M parameters), SineGen noise drawn on device every step from
an advancing Philox state.  A "step" = one utterance per GPU (weak scaling: every rank synthesises its own).

  value      device-resident inputs through the public graph path (`Model.synthesize_ids`: text-side graph -> ONE host read of the
             frame count -> acoustic-side graph), K steps between barrier+synchronize brackets, CUDA events, max over ranks.
             `value_pinned_durations` = the same with the durations supplied (no host read in the middle).
  e2e        the call a user makes, with HOST buffers: `model(phonemes, ref_s_pinned, out=pinned)` -- phoneme string -> ids, H2D
             copies, both graphs, waveform D2H into pinned memory, stream synchronised -- wall clock.
  parity_rel_rms   the same graph path once more on the committed fixture inputs (tests/golden/bench_shapes_golden.npz: injected SineGen
             noise + the oracle's float32 F0/N curves) against the cached float64-oracle waveform of THIS shape.
  roofline   the dominant kernel family (dense conv1d / transposed conv of the decoder+generator stack).  Times are those of the
             REPLAYED graph: an instrumented copy of the graphs carries event-record nodes around every launch; `kernel_ms` is the
             wall-clock coverage (union of the intervals) of the family inside one replay, so it can never exceed ms_per_step.
             Algorithmic bytes per utterance (SURVEY.md section 8d: 137.2 MB per audio-second, bf16 convention) / that time,
             against MEASURED_PEAKS.json hbm_gbs; `tensor` repeats it in flops against the sustained bf16 peak.
  cpu_baseline  the oracle port (torch-CPU fp32 restatement of the reference; MLX is not installable) on the host cores, bounded sample.
`--impl reference` times that same CPU restatement as the reference arm (rank 0 only).
`--workload whisper|codec|qwen3` select the other BASELINE configurations (see the functions below).
`--dump-outputs DIR` writes the waveform and durations of the last timed step as .npy files; weights, inputs and the noise state
are seeded, so two runs with the same arguments are comparable output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PHONEMES = 128
CONV_STACK_MB_PER_AUDIO_S = 137.2          # SURVEY.md section 8(d), Kokoro decoder+generator, bf16 convention
CONV_STACK_GFLOP_PER_AUDIO_S = 58.84       # 573.7 GF per 9.75 s utterance (VERDICT r01 / SURVEY 8d), one bf16 product per MAC
METRIC = "audio-sec/sec Kokoro-82M TTS (128-phoneme utterance, 9.75 s)"


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1590.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_port_run(n_utts: int, threads: int):
    """Time the oracle port (fp32 torch-CPU restatement of the reference) on `n_utts` cfg2 utterances, durations from its own
    duration head exactly like the GPU arm.  Returns (seconds per utterance list, audio seconds per utterance)."""
    import torch
    from mlx_audio_b200 import synth
    from mlx_audio_b200.configs import KOKORO_82M
    from oracle import kokoro as OK
    torch.set_num_threads(threads)
    print(f"[bench] cpu port: {n_utts} utterance(s) on {threads} threads", file=sys.stderr, flush=True)
    P = synth.kokoro_weights(KOKORO_82M)
    ids, ref = synth.kokoro_inputs(N_PHONEMES)
    times, audio = [], None
    for _ in range(n_utts):
        t0 = time.perf_counter()
        audio, _ = OK.forward(P, ids, ref, noise=lambda n: synth.kokoro_noise(n)[1])
        times.append(time.perf_counter() - t0)
    return times, audio.shape[0] / 24000.0


def host_threads() -> int:
    """Threads the CPU arm may use: the cores this process is actually allowed to run on (cgroup / affinity aware), capped
    at 32 -- the restatement's small ops stop scaling long before that."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, p = f.read().split()
            if q != "max":
                n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    return max(1, min(n, 32))


WORKLOAD_NAME = "kokoro-82m cfg2: 128 phonemes (T=130), model duration head -> F=390 frames, 234000 samples = 9.75 s per step per GPU"


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU implementation of the path, here its restatement (MLX cannot be installed)."""
    if rank != 0:
        return
    cores = host_threads()
    cpu_port_run(1, cores)           # warm-up (bounded: one utterance)
    times, audio_s = cpu_port_run(args.steps, cores)
    total = sum(times)
    v = audio_s * len(times) / total
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_NAME, "parallelism": "cpu"},
            "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": cores, "kind": "port",
                             "sample": f"{len(times)} full cfg2 utterances, torch-CPU fp32 restatement of the reference (oracle/kokoro.py)"},
            "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, **arrays):
    """Write each tensor as out_dir/<name>.npy (float32 or float64), so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().cpu().numpy())


def _union_ms(intervals):
    """Total length of the union of (start, end) intervals."""
    tot, cur_s, cur_e = 0.0, None, None
    for s, e in sorted(intervals):
        if cur_e is None or s > cur_e:
            if cur_e is not None:
                tot += cur_e - cur_s
            cur_s, cur_e = s, e
        else:
            cur_e = max(cur_e, e)
    if cur_e is not None:
        tot += cur_e - cur_s
    return tot


def kokoro_graph_profile(model, ops, torch, ids_d, ref_d, dev, reps=3):
    """Per-launch times INSIDE the replayed graphs: a second model object (same weights) captures its graphs while ops.PROFILE is on
    with external events, so every launch is bracketed by event-record nodes; each replay re-stamps them."""
    from mlx_audio_b200.tts.models.kokoro import Model
    prof = {}
    twin = Model(model.config, device=dev)
    twin._w, twin._ada_slices, twin._ada_pred, twin._raw = model._w, model._ada_slices, model._ada_pred, getattr(model, "_raw", None)
    twin.seed(7)
    tags = {}
    ops.PROFILE, ops.PROFILE_EXTERNAL, ops.PROFILE_TAGS = prof, True, tags
    try:
        twin.synthesize_ids(ids_d, ref_d)                 # captures both graphs with the event nodes (the eager warm-ups also append)
    finally:
        ops.PROFILE, ops.PROFILE_EXTERNAL, ops.PROFILE_TAGS = None, False, None
    # keep only the events recorded during the two captures: they are the LAST n of each kind, where n = launches in the captured pass;
    # simplest robust filter: an event pair that was never re-stamped by a replay raises / returns garbage -> use a base event in-graph
    t_base = torch.cuda.Event(enable_timing=True)
    per_kind, cover = {}, {}
    for _ in range(reps):
        t_base.record()
        twin.synthesize_ids(ids_d, ref_d)
        torch.cuda.synchronize(dev)
        top = []
        for kind, evs in prof.items():
            iv = []
            for i, (a, b) in enumerate(evs):
                try:
                    s, e = t_base.elapsed_time(a), t_base.elapsed_time(b)
                except Exception:
                    continue
                if s >= 0.0 and e >= s and tags.get(kind) and tags[kind][i]:
                    top.append((round((e - s) * 1e3, 1), tags[kind][i]))
                if s >= 0.0 and e >= s:                   # events of the eager warm-up passes lie BEFORE t_base: negative -> dropped
                    iv.append((s, e))
            per_kind.setdefault(kind, []).append(sum(e - s for s, e in iv))
            cover.setdefault(kind, []).append(iv)
    n_launch = {k: len(v[-1]) for k, v in cover.items()}
    by_kind = {k: sum(v) / len(v) for k, v in per_kind.items()}
    kokoro_graph_profile.top_launches = sorted(top, reverse=True)[:24]          # (us, label) of the last replay's slowest tagged launches
    kokoro_graph_profile.tagged_us = round(sum(t for t, _ in top), 1)
    return by_kind, {k: v[-1] for k, v in cover.items()}, n_launch


def main_kokoro(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import numpy as np
    from mlx_audio_b200 import ops, synth
    from mlx_audio_b200.configs import KOKORO_82M
    from mlx_audio_b200.tts.models.kokoro import Model, ModelConfig

    W = max(args.warmup, 3)
    K = args.steps
    log = lambda m: print(f"[bench r{rank} {time.strftime('%H:%M:%S')}] {m}", file=sys.stderr, flush=True)
    log("building synthetic checkpoint")
    P = synth.kokoro_weights(KOKORO_82M, seed=0)
    model = Model(ModelConfig.from_dict(KOKORO_82M), device=dev).load_weights(list(P.items()))
    model.use_graphs = not args.no_graph
    model.seed(1234 + rank)
    ids, ref_s = synth.kokoro_inputs(N_PHONEMES, seed=1 + rank)
    T = ids.shape[1]
    ids_d, ref_d = ids[0].to(dev), ref_s.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)            # > 126 MB L2
    # vocabulary for the string entry point: symbol i <-> token id i (ids 1..177 are used by the synthetic utterance)
    model.vocab = {chr(0x100 + i): i for i in range(1, KOKORO_82M["n_token"])}
    phonemes = "".join(chr(0x100 + int(i)) for i in ids[0, 1:-1])

    run_ids = model.synthesize_ids if model.use_graphs else model.forward_ids

    def step():
        return run_ids(ids_d, ref_d)

    if args.ncu:
        for _ in range(2):
            model.forward_ids(ids_d, ref_d)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        model.forward_ids(ids_d, ref_d)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return
    if args.ncu_graph:
        for _ in range(3):
            step()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        step()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return

    log("model ready; capturing")
    audio = step()[0]
    torch.cuda.synchronize(dev)
    n_samples = int(audio.shape[0])
    F = n_samples // 600
    audio_s = n_samples / 24000.0
    dur_d = torch.full((T,), F // T, dtype=torch.int64, device=dev)
    dur_d[0] += F - int(dur_d.sum().item())
    launches_per_step = None
    if model.use_graphs:
        launches_per_step = sum(v["launches"] for v in model._graphs.values()) + 2       # + the Philox draw (2 launches) between the graphs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn):
        for _ in range(W):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            flush.zero_()                                                      # L2 flush between timed iterations
            out = fn()
        e1.record()
        barrier()
        return e0.elapsed_time(e1), out

    log("timing device-resident steps")
    n0 = ops.LAUNCHES[0]
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms, (audio, pred_dur) = timed(step)
    clocks = sampler.stop()
    launches = ops.LAUNCHES[0] - n0
    assert audio.shape[0] == n_samples and bool(torch.isfinite(audio).all())
    if args.dump_outputs and rank == 0:
        # the graph path returns static buffers that the next call overwrites: copy them out before anything else runs
        dump_outputs(args.dump_outputs, audio=audio.float(), pred_dur=pred_dur.double())
    ms_pinned, _ = timed(lambda: run_ids(ids_d, ref_d, pred_dur=dur_d, n_frames=F)[0])
    # L2 flush cost measured separately and subtracted (it is not part of the step)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    f0.record()
    for _ in range(K):
        flush.zero_()
    f1.record()
    torch.cuda.synchronize(dev)
    ms_flush = f0.elapsed_time(f1)

    def rank_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # where the step goes: the two graphs timed separately (same buffers, no flush in between)
    side_ms = {}
    if model.use_graphs:
        tgs = [v for k, v in model._graphs.items() if k[0] == "text" and not k[3]]
        ags = [v for k, v in model._graphs.items() if k[0] == "acoustic" and v["text"] is (tgs[0] if tgs else None) and not k[4]]
        if tgs and ags:
            for name, g in (("text_side", tgs[0]["graph"]), ("acoustic_side", ags[0]["graph"])):
                torch.cuda.synchronize(dev)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(10):
                    g.replay()
                b.record()
                torch.cuda.synchronize(dev)
                side_ms[name] = a.elapsed_time(b) / 10
    ms_max = rank_max(max(ms - ms_flush, 1e-6))
    ms_pinned_max = rank_max(max(ms_pinned - ms_flush, 1e-6))
    value = world * K * audio_s / (ms_max / 1e3)

    log(f"value done: {ms_max / K:.3f} ms/step ({ms_pinned_max / K:.3f} with pinned durations); timing e2e")
    # ---------------- end-to-end through the public call with host buffers
    ref_h = ref_s.clone().pin_memory()
    out_h = torch.empty(n_samples, dtype=torch.float32).pin_memory()

    def step_e2e():
        model(phonemes, ref_h, 1.0, out=out_h)                                 # phoneme string -> ids -> H2D -> graphs -> D2H into pinned memory
        torch.cuda.current_stream(dev).synchronize()                           # the caller owns the waveform when this returns
        return out_h

    for _ in range(W):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        flush.zero_()
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0 - ms_flush / 1e3
    e2e_value = world * K * audio_s / rank_max(e2e_s)
    assert bool(torch.isfinite(out_h).all()) and float(out_h.abs().max()) > 0

    # ---------------- parity of this very shape against the cached oracle waveform
    parity = None
    gpath = os.path.join(ROOT, "tests", "golden", "bench_shapes_golden.npz")
    if os.path.exists(gpath) and rank == 0:
        g = np.load(gpath)
        ids0, ref0 = synth.kokoro_inputs(N_PHONEMES, seed=1)
        nz = synth.kokoro_noise(ids0.shape[1] * 3 * 600, 3)[1].to(dev).contiguous()
        f0n = (torch.as_tensor(g["kokoro_f0"]).to(dev), torch.as_tensor(g["kokoro_n"]).to(dev))
        a, pd = run_ids(ids0[0].to(dev), ref0.to(dev), noise=nz, f0n_override=f0n)
        want = torch.as_tensor(g["kokoro_audio"]).double()
        got = a.double().cpu()
        if got.shape == want.shape:
            parity = float(torch.sqrt(((got - want) ** 2).mean()) / torch.sqrt((want ** 2).mean()))
        else:
            parity = float("nan")
        log(f"parity vs cached oracle waveform (cfg2 shape, graph path): rel RMS {parity:.3e}")

    log("e2e done; instrumented pass")
    # ---------------- roofline of the dominant kernel family, timed inside the replayed graph
    conv_kinds = ("conv", "conv_tc", "prep", "adain_stats")     # the dense conv stack: convs, their bf16 prologue and InstanceNorm statistics
    timing_path = "graph event nodes"
    try:
        if not model.use_graphs:
            raise RuntimeError("eager run requested")
        by_kind, cover, n_launch = kokoro_graph_profile(model, ops, torch, ids_d, ref_d, dev)
        if not by_kind or sum(n_launch.values()) == 0:
            raise RuntimeError("no in-graph events came back")
        conv_iv = [iv for k in conv_kinds for iv in cover.get(k, [])]
        conv_ms = _union_ms(conv_iv)
        conv_sum_ms = sum(by_kind.get(k, 0.0) for k in conv_kinds)
        n_conv = sum(n_launch.get(k, 0) for k in conv_kinds)
        all_ms = _union_ms([iv for v in cover.values() for iv in v])
    except Exception as exc:                                   # older driver without timed event nodes: eager instrumented pass
        log(f"graph-node timing unavailable ({exc}); falling back to the eager instrumented pass")
        timing_path = "eager pass (serialises the graph's parallel branches)"
        prof = {}
        ops.PROFILE = prof
        for _ in range(3):
            model.forward_ids(ids_d, ref_d)
        torch.cuda.synchronize(dev)
        ops.PROFILE = None
        by_kind = {k: sum(a.elapsed_time(b) for a, b in v) / 3 for k, v in prof.items()}
        conv_ms = conv_sum_ms = sum(by_kind.get(k, 0.0) for k in conv_kinds)
        n_conv = sum(len(prof.get(k, [])) for k in conv_kinds) // 3
        all_ms = sum(by_kind.values())
    peaks, peak_kind = _peaks()
    alg_bytes = CONV_STACK_MB_PER_AUDIO_S * 1e6 * audio_s                    # per utterance, all conv launches
    alg_flops = CONV_STACK_GFLOP_PER_AUDIO_S * 1e9 * audio_s
    achieved = alg_bytes / (conv_ms / 1e3) / 1e9
    traffic = None                                                           # measured DRAM bytes of the same kernels (ncu capture, committed)
    for name in ("r02_traffic.json", "r01b_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            try:
                traffic = float(json.load(open(tpath))["conv_stack_bytes_per_step"])
                break
            except Exception:
                traffic = None
    tf = alg_flops / (conv_ms / 1e3) / 1e12
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                "traffic": traffic, "peak_kind": peak_kind,
                "kernel": "dense conv stack of the decoder + generator (tcgen05 conv kernels + CUDA-core strided / narrow convs, incl. their prologue and InstanceNorm statistics)",
                "timing": timing_path, "launches_per_utterance": n_conv, "kernel_ms_per_utterance": conv_ms,
                "kernel_ms_summed": conv_sum_ms, "all_kernels_ms_per_utterance": all_ms,
                "ms_by_kind": {k: round(v, 3) for k, v in sorted(by_kind.items(), key=lambda kv: -kv[1])},
                "top_launches_us": getattr(kokoro_graph_profile, "top_launches", None), "fused_launches_us_total": getattr(kokoro_graph_profile, "tagged_us", None),
                "algorithmic_bytes_per_utterance": alg_bytes,
                "tensor": {"bound": "tensor", "achieved": tf, "peak": peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]), "unit": "TFLOP/s",
                           "frac": tf / peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]), "algorithmic_flops_per_utterance": alg_flops,
                           "note": "one bf16 product per MAC; the x2 (hi+lo) mode issues two"}}

    log("instrumented pass done")
    if rank == 0:
        cores = host_threads()
        cpu = None
        if world == 1 and args.cpu_utts > 0:
            times, cpu_audio_s = cpu_port_run(args.cpu_utts, cores)
            cpu = {"value": cpu_audio_s * len(times) / sum(times), "unit": "audio-s/s", "cores": cores, "kind": "port",
                   "sample": f"{len(times)} full cfg2 utterances ({sum(times):.1f} s), torch-CPU fp32 restatement of the reference"}
        line = {"metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if ops.TC_MODE[0] == "off" else ("bf16x2" if ops.TC_MODE[0] == "x2" else "bf16"), "data": "synthetic",
                "config": {"workload": WORKLOAD_NAME,
                           "parallelism": f"utterance-sharded x{world} (no data-path collective)", "l2": "256 MiB flush between timed steps (its cost subtracted)",
                           "launch": "eager" if args.no_graph else "cuda-graph replay through Model.synthesize_ids (2 graphs + 1 host read of F)",
                           "weights": "synthetic bf16 checkpoint, 81.8 M params",
                           "activations": "fp32 in HBM; tensor-core mode " + ops.TC_MODE[0] + " (x2 = hi+lo bf16 planes, fp32-grade products)",
                           "frames": F, "audio_s_per_step": audio_s},
                "clocks": clocks, "gpu_launches": launches,
                "value_pinned_durations": world * K * audio_s / (ms_pinned_max / 1e3), "ms_per_step_pinned_durations": ms_pinned_max / K,
                "parity_rel_rms": parity, "ms_by_side": {k: round(v, 3) for k, v in side_ms.items()},
                "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": int(T * 8 + ref_h.numel() * 4),
                        "d2h_bytes_per_step": int(out_h.numel() * 4 + 8), "call": "Model.__call__(phonemes, ref_s, out=pinned)"},
                "roofline": roofline}
        if cpu:
            line["cpu_baseline"] = cpu
        if launches_per_step:
            line["config"]["kernels_per_step"] = launches_per_step
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    # rank 0 prints ONE JSON line on stdout: NCCL's version banner (NCCL_DEBUG=VERSION, set by some launch environments) would be a second one
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="kokoro", choices=["kokoro", "whisper", "codec", "qwen3"])
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--cpu-utts", type=int, default=4, help="utterances in the cpu_baseline sample")
    ap.add_argument("--ncu", action="store_true", help="profiling aid: 2 eager warm-up steps, then ONE eager step between "
                    "cudaProfilerStart/Stop (run under `ncu --profile-from-start off`); prints no bench line")
    ap.add_argument("--ncu-graph", action="store_true", help="like --ncu but the profiled step is the graph replay "
                    "(run under `ncu --profile-from-start off --graph-profiling node`)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (rank 0: audio as float32, "
                    "pred_dur as float64) to DIR/<name>.npy; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "kokoro" or args.impl != "b200" or args.ncu or args.ncu_graph):
        ap.error("--dump-outputs is available for the timed kokoro run of --impl b200 only")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload != "kokoro":
        import bench_workloads
        return bench_workloads.main(args, rank, world, local_rank)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    main_kokoro(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
