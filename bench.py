#!/usr/bin/env python3
"""bench.py — headline benchmark of the B200-native Qwen3-TTS engine (contract: task prompt §④ / "bench.py").

Workload (BASELINE.json configs[1]): Qwen3-TTS-12Hz-0.6B-Base voice clone, streaming chunk_size=8, bs=1, random-init
weights of the named architecture, the reference's own benchmark text (benchmarks/throughput.py:16), x-vector
mode, sampling defaults (T=0.9, top_k=50, rep 1.05), 256 frames (20.48 s of audio; EOS is held off with
min_new_tokens so the work per step is fixed).

One step = one utterance.  Metric = audio seconds generated per wall second (== RTF at bs=1, == the box's aggregate
audio-sec/sec at N GPUs, one replica and one utterance stream per GPU, no collective on the data path).
  value : prompt embeddings already resident in HBM; prefill + 32 launches of 8 frames + streaming codec decode,
          audio left on the device.  Timed with CUDA events on the launching stream.
  e2e   : the public API call a user makes — FasterQwen3TTS.generate_voice_clone_streaming(text, ...) with HOST
          inputs (text string, wav path) and HOST outputs (numpy audio per chunk): tokenisation, prompt build,
          host->device copies of the ids, device->host copies of every audio chunk inside the timed region.
  roofline : the persistent decode kernel (fq3_stream_kernel), algorithmic bytes = streaming bound of SURVEY.md
          §8(d) (all weights a frame touches + valid KV), duration from CUDA events around each launch.
  cpu_baseline / --impl reference : the oracle (CPU restatement of the reference path; the reference has no CPU
          path and its arithmetic lives in the absent `qwen_tts`, so kind = "port") on the host cores, on a bounded sample
          of the same workload (first 40 frames, same prompt / sampling / streaming codec policy).
  gpu_anchor : the reference's execution style (static caches + masks + CUDA-graph replays) restated on the same weights
          and timed on the same GPU (oracle/graph_anchor.py) — ms per frame beside decode_ms_per_frame.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
import wave

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TEXT = ("Ladies and gentlemen, I have just been informed that this speech is being generated faster than I can speak it. "
        "The robots have officially won. Please remain calm.")  # benchmarks/throughput.py:16
REF_TEXT = "I'm confused why some people have super short timelines."  # ignored in x-vector mode (cache key only)
FRAME_S = 0.08  # 1920 samples @ 24 kHz
METRIC = "audio_seconds_per_second"
UNIT = "audio-s/s"


def make_ref_wav() -> str:
    import numpy as np

    path = os.path.join(tempfile.gettempdir(), f"fq3_bench_ref_{os.getpid()}.wav")
    sr = 24000
    t = np.arange(int(3.0 * sr)) / sr
    pcm = (0.2 * np.sin(2 * np.pi * 180 * t) * 32767).astype("int16")
    with wave.open(path, "wb") as wf:
        wf.setnchannels(1)
        wf.setsampwidth(2)
        wf.setframerate(sr)
        wf.writeframes(pcm.tobytes())
    return path


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def n_prompt_rows(text: str) -> int:
    return len([w for w in text.replace("\n", " \n ").split(" ") if w]) + 11  # model.py prompt layout, x-vector + nsm


# ------------------------------------------------------------------------------------------------
# CPU oracle leg (cpu_baseline and --impl reference)
# ------------------------------------------------------------------------------------------------
class CpuOracleArm:
    """The reference path restated on the host cores (oracle/), on a bounded sample of the bench workload: the SAME prompt
    (T = 39 rows), the SAME sampling policy and the SAME streaming policy — chunks of `chunk` frames, codec decode per chunk
    with the reference's accumulate-then-25-frame-window rule (model.py:737-826) — for the first `frames` frames of the
    256-frame utterance.  Prefill is therefore amortised over `frames` frames instead of 256; the line's
    `config.reference_sample` says so."""

    CONTEXT = 25  # model.py:741

    def __init__(self, model_name: str, frames: int, chunk: int):
        import torch

        from oracle.codec_oracle import CodecOracle
        from oracle.qwen3_tts_oracle import OracleTTS
        from qwen3_tts_cuda_graphs_b200.codec import init_codec_synthetic
        from qwen3_tts_cuda_graphs_b200.config import preset
        from qwen3_tts_cuda_graphs_b200.weights import init_synthetic

        self.torch = torch
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        cfg = preset(model_name)
        w = init_synthetic(cfg, seed=0, skip_text_embedding=True)
        self.orc = OracleTTS(cfg, w)
        self.codec = CodecOracle(cfg.codec, init_codec_synthetic(cfg.codec, seed=1))
        self.frames, self.chunk = frames, chunk
        T, H = n_prompt_rows(TEXT), cfg.talker.hidden_size
        g = torch.Generator().manual_seed(1)
        self.prompt = ((0.05 * torch.randn(1, T, H, generator=g)).to(torch.bfloat16), torch.ones(1, T, dtype=torch.long),
                       (0.05 * torch.randn(1, 1, H, generator=g)).to(torch.bfloat16),
                       (0.05 * torch.randn(1, 1, H, generator=g)).to(torch.bfloat16))
        self.decoded = 0
        self.sample = (f"first {frames} of the utterance's frames: prefill T={T} + {frames} frames in chunks of {chunk}, codec decode per "
                       f"chunk (accumulated until {max(self.CONTEXT, chunk)} frames, then {self.CONTEXT}-frame window), oracle on {self.cores} threads")

    def step(self) -> float:
        torch = self.torch
        t0 = time.perf_counter()
        self.decoded = 0
        with torch.inference_mode():
            gen = torch.Generator().manual_seed(0)
            frames, calibrated, n_new = [], False, 0
            for fr in self.orc.generate_frames(*self.prompt, max_new_tokens=self.frames, min_new_tokens=self.frames, generator=gen):
                frames.append(fr)
                n_new += 1
                if n_new < self.chunk and len(frames) < self.frames:
                    continue
                n_total = len(frames)
                if not calibrated:  # phase 1 (model.py:774-806): decode everything so far
                    window = frames
                    calibrated = n_total >= max(self.CONTEXT, self.chunk)
                else:               # phase 2 (model.py:807-826): new frames + 25 frames of left context
                    window = frames[max(0, n_total - n_new - self.CONTEXT):]
                self.codec.decode(torch.stack(window))
                self.decoded += len(window)
                n_new = 0
        dt = time.perf_counter() - t0
        return len(frames) * FRAME_S / dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuOracleArm(args.model, args.cpu_frames, args.chunk)
    for _ in range(args.warmup):
        arm.step()
    t0 = time.perf_counter()
    vals = [arm.step() for _ in range(args.steps)]
    dt = time.perf_counter() - t0
    v = args.steps * args.cpu_frames * FRAME_S / dt
    cfg = workload_config(args)
    cfg["reference_sample"] = {"frames_per_step": args.cpu_frames, "of_frames": args.frames, "codec_frames_decoded_per_step": arm.decoded,
                               "note": "bounded sample of the workload: prefill amortised over the sample's frames; one CPU process on rank 0"}
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1000, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": arm.cores, "kind": "port", "sample": arm.sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "per_step": vals,
    }
    print(json.dumps(line), flush=True)


def workload_config(args) -> dict:
    return {
        "workload": f"Qwen3-TTS-12Hz-{args.model} voice clone streaming chunk_size={args.chunk}, bs=1, {args.frames} frames/utterance "
                    f"({args.frames * FRAME_S:.2f} s audio), x-vector mode, sampling T=0.9 top_k=50 rep=1.05, random-init weights",
        "prompt_rows": n_prompt_rows(TEXT), "chunk_size": args.chunk, "frames": args.frames, "max_seq_len": 2048,
        "replicas": args.gpus, "l2_policy": "inputs larger than L2: every frame streams 3.3 GB of weights (L2 = 126 MB)",
    }


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def aggregate_over_ranks(times_ms, totals, device, world):
    """Replicas only (DESIGN.md §7): the job time is the MAX over ranks of each timed leg, the work is the SUM.
    times_ms / totals: sequences of floats of this rank; returns (max-reduced times, sum-reduced totals)."""
    import torch
    import torch.distributed as dist

    t = torch.tensor(list(times_ms), dtype=torch.float64, device=device)
    tot = torch.tensor(list(totals), dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    return [float(x) for x in t], [float(x) for x in tot]


def kernel_source_hash() -> str:
    """sha256 over the decode kernel's sources: ties a committed ncu capture to the code it was taken from."""
    import hashlib
    h = hashlib.sha256()
    for f in ("fq3_kernel.cuh", "fq3_common.cuh", "fq3_api.cu"):
        with open(os.path.join(ROOT, "qwen3_tts_cuda_graphs_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def ncu_traffic(frames_per_launch):
    """DRAM bytes per launch of the decode kernel from the committed `ncu --set full` capture (profiles/ncu_traffic.json,
    written by scripts/evidence.sh).  Returned only if the capture was taken from THIS kernel source (kernel_hash) and launch
    shape; otherwise (None, why) — a stale number is worse than none."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except (OSError, ValueError):
        return None, "no capture committed"
    if int(d.get("frames_per_launch", -1)) != int(frames_per_launch):
        return None, "capture has another launch shape"
    if d.get("kernel_hash") != kernel_source_hash():
        return None, f"capture is from kernel source {d.get('kernel_hash')}, this is {kernel_source_hash()}"
    return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"]), f"ncu --set full, kernel source {d['kernel_hash']}, {d.get('source', '')}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="0.6B-Base")
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--chunk", type=int, default=8)
    ap.add_argument("--cpu-frames", type=int, default=40, dest="cpu_frames",
                    help="frames of the utterance the CPU arm generates per step (bounded sample of the workload)")
    ap.add_argument("--anchor-frames", type=int, default=48, dest="anchor_frames",
                    help="frames timed by the same-box GPU anchor (oracle restated as CUDA-graph replays); 0 = skip")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--batched-streams", type=str, default="4,16,64", dest="batched_streams",
                    help="extra (reported, not the headline) leg at N=1: this many utterances decoded request-parallel on one GPU "
                         "(comma list; lock-step groups of up to 16 share a weight sweep); 0 = skip")
    ap.add_argument("--serving-requests", type=int, default=32, dest="serving_requests",
                    help="extra leg at N=1: this many requests through serving.BatchScheduler (16 concurrent); 0 = skip")
    ap.add_argument("--dump-outputs", default=None, dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of the headline leg returned as DIR/<name>.npy "
                         "(float32: codes [frames, 16] and the streamed audio), so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    # every utterance draws its sampling seed from torch's RNG (generate._fresh_seed): seeded, the same arguments sample the same ids
    torch.manual_seed(0)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from qwen3_tts_cuda_graphs_b200 import FasterQwen3TTS
    from qwen3_tts_cuda_graphs_b200.streaming import fast_generate_streaming
    from qwen3_tts_cuda_graphs_b200.weights import param_bytes

    dev = f"cuda:{local}"
    model = FasterQwen3TTS.from_pretrained(f"synthetic://{args.model}", device=dev, dtype=torch.bfloat16,
                                           attn_implementation="eager", max_seq_len=2048, seed=0)
    eng = model.model.engine
    codec = model.model.model.speech_tokenizer.decoder
    ref_wav = make_ref_wav()
    gen_kw = dict(max_new_tokens=args.frames, min_new_tokens=args.frames)
    api_kw = dict(text=TEXT, language="English", ref_audio=ref_wav, ref_text=REF_TEXT, chunk_size=args.chunk, **gen_kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- e2e through the public API (host in, host out) -------------------------------------------
    def e2e_step():
        n_samples, d2h = 0, 0
        for audio, sr, _ in model.generate_voice_clone_streaming(**api_kw):
            n_samples += len(audio)
            d2h += audio.nbytes
        return n_samples / sr, d2h

    # ---- device-resident leg -------------------------------------------------------------------------
    m, talker, tconf, tie, tam, tth, tpe, _ = model._prepare_generation(TEXT, ref_wav, REF_TEXT, language="English",
                                                                        non_streaming_mode=True)
    launch_events = []

    def keep_codes(stream, into):
        for chunk, timing in stream:
            into.append(chunk)
            yield chunk, timing

    def dev_step(events=None, keep=None):
        """keep: None, or a dict whose "codes" / "audio" lists receive the step's device tensors (references, no copies)."""
        stream = fast_generate_streaming(
            talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth, tts_pad_embed=tpe,
            config=tconf, predictor_graph=model.predictor_graph, talker_graph=model.talker_graph, chunk_size=args.chunk,
            launch_events=events, **gen_kw)
        if keep is not None:
            stream = keep_codes(stream, keep["codes"])
        n = 0
        for audio, sr, _ in model._stream_audio(m, stream, None, args.chunk, to_host=False):
            n += audio.numel()
            if keep is not None:
                keep["audio"].append(audio)
        return n / sr

    for _ in range(args.warmup):
        dev_step()
        e2e_step()

    # TTFA as benchmarks/throughput.py:50-61 (5 warm runs, time to the first yielded audio chunk)
    ttfa = []
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g = model.generate_voice_clone_streaming(**api_kw)
        next(g)
        torch.cuda.synchronize()
        ttfa.append((time.perf_counter() - t0) * 1000)
        g.close()

    clocks = ClockSampler(local)
    clocks.start()
    # value: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks
    l0 = eng.launch_count + codec.launch_count
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    audio_s = 0.0
    last = {"codes": [], "audio": []}
    for i in range(args.steps):
        audio_s += dev_step(launch_events, last if args.dump_outputs and i == args.steps - 1 else None)
    ev1.record()
    barrier()
    launches = eng.launch_count + codec.launch_count - l0
    dev_ms = ev0.elapsed_time(ev1)
    # e2e: wall clock around the API calls (host work is part of the metric), synchronised both sides
    barrier()
    t0 = time.perf_counter()
    e2e_audio_s, d2h = 0.0, 0
    for _ in range(args.steps):
        a, b = e2e_step()
        e2e_audio_s += a
        d2h += b
    barrier()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop()

    (dev_ms, e2e_ms), (audio_all, e2e_audio_all) = aggregate_over_ranks([dev_ms, e2e_s * 1000.0], [audio_s, e2e_audio_s], dev, world)

    if args.dump_outputs and rank == 0:
        # codes [frames, 16] and audio [frames * 1920]: at most 16 MB in all, since max_seq_len 2048 bounds the frames
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, parts in last.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), torch.cat(parts).float().cpu().numpy())

    if rank == 0:
        pb = param_bytes(model.model.cfg)
        # roofline of the persistent decode kernel: per launch of `chunk` frames
        durs = [e0.elapsed_time(e1) for e0, e1, _ in launch_events]
        nfr = [n for _, _, n in launch_events]
        t_cfg = model.model.cfg.talker
        kv_row = 2 * t_cfg.num_hidden_layers * t_cfg.num_key_value_heads * t_cfg.head_dim * 2  # K+V bytes per position
        T0 = tie.shape[1]
        kv_bytes = 0.0
        for j, n in enumerate(nfr):
            start = T0 + (j % (args.frames // args.chunk)) * args.chunk
            kv_bytes += sum(kv_row * (start + i + 1) for i in range(n))
        alg_bytes = (pb["frame_streaming"] * sum(nfr) + kv_bytes) / max(len(durs), 1)
        avg_ms = sum(durs) / max(len(durs), 1)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
        ids_bytes = 8 * (n_prompt_rows(TEXT) - 11 + 8)
        line = {
            "metric": METRIC, "value": audio_all / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args),
            "e2e": {"value": e2e_audio_all / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": ids_bytes,
                    "d2h_bytes_per_step": d2h // max(args.steps, 1), "api": "FasterQwen3TTS.generate_voice_clone_streaming"},
            "gpu_launches": int(launches),
            "clocks": clk,
            "ttfa_ms": {"mean": float(np.mean(ttfa)), "std": float(np.std(ttfa)), "runs": 5, "chunk_size": args.chunk},
            "rtf": audio_all / world / (dev_ms * 1e-3) if world > 1 else audio_all / (dev_ms * 1e-3),
            "roofline": {
                "bound": "hbm", "kernel": "fq3_stream_kernel (persistent decode: predictor + talker + sampling)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s",
                "traffic": ncu_traffic(args.chunk)[0], "traffic_source": ncu_traffic(args.chunk)[1], "bytes_per_launch": alg_bytes, "launch_ms": avg_ms, "frames_per_launch": args.chunk,
                "bytes_model": "streaming bound: 15 predictor passes + heads + talker step + valid KV per frame (SURVEY.md 8d)",
            },
            "decode_ms_per_frame": avg_ms / args.chunk,
        }
        batch_sizes = [int(x) for x in str(args.batched_streams).split(",") if x.strip() and int(x) > 1]
        if world == 1 and batch_sizes:
            # request-parallel decode inside one GPU (BASELINE configs[3] / [4]): the same prompt on every stream, non-streaming,
            # codec decode of every utterance included; wall clock between synchronisations
            from qwen3_tts_cuda_graphs_b200.generate import fast_generate_batch
            model_b = FasterQwen3TTS.from_pretrained(f"synthetic://{args.model}", device=dev, dtype=torch.bfloat16,
                                                     attn_implementation="eager", max_seq_len=1024, seed=0, max_streams=max(batch_sizes))
            mb, _, _, tie_b, tam_b, tth_b, tpe_b, _ = model_b._prepare_generation(TEXT, ref_wav, REF_TEXT, language="English",
                                                                                  non_streaming_mode=True)
            by = {}
            for ns in batch_sizes:
                reqs = [(tie_b, tam_b, tth_b, tpe_b)] * ns

                def batched_step():
                    codes, _ = fast_generate_batch(model_b.talker_graph, model_b.predictor_graph, reqs, **gen_kw)
                    n = 0
                    for c in codes:
                        a, sr_b = model_b._decode_full(mb, c)
                        n += len(a[0])
                    return n / sr_b

                batched_step()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                reps = max(1, args.steps - 1) if ns <= 16 else 1
                a_s = sum(batched_step() for _ in range(reps))
                torch.cuda.synchronize()
                by[str(ns)] = a_s / (time.perf_counter() - t0)
            line["batched"] = {"by_streams": by, "unit": UNIT, "lockstep_group": model_b.model.engine.lockstep_group,
                               "streams": max(batch_sizes), "value": by[str(max(batch_sizes))],
                               "what": "request-parallel decode of identical prompts on one GPU (groups of up to lockstep_group streams share "
                                       "every weight sweep; more streams run group after group), non-streaming, max_seq_len 1024, prefill and "
                                       "codec decode of every utterance included"}
            if args.serving_requests > 0:
                # the same GPU through the serving layer (SURVEY.md §8 f4): requests submitted at once to the continuous-batching
                # scheduler, audio streamed back chunk by chunk; wall clock incl. prompt build, prefill, codec, D2H
                try:
                    import threading
                    from qwen3_tts_cuda_graphs_b200.serving import BatchScheduler, TTSRequest
                    conc = min(16, max(batch_sizes))

                    def serve(n_req):
                        got = []
                        with BatchScheduler(model_b, chunk_frames=args.chunk, max_concurrent=conc) as sched:
                            t0 = time.perf_counter()
                            hs = [sched.submit(TTSRequest(TEXT + f" Request {i}.", ref_audio=ref_wav, ref_text=REF_TEXT, language="English", **gen_kw))
                                  for i in range(n_req)]
                            ths = [threading.Thread(target=lambda h=h: got.append(len(h.result()[0]) / model_b.sample_rate)) for h in hs]
                            for th in ths:
                                th.daemon = True
                                th.start()
                            deadline = time.perf_counter() + 180.0
                            for th in ths:
                                th.join(max(0.0, deadline - time.perf_counter()))
                            if any(th.is_alive() for th in ths):
                                raise TimeoutError("serving leg did not finish within 180 s")
                            dt = time.perf_counter() - t0
                        return sum(got) / dt, [h.ttfa_s for h in hs if h.ttfa_s is not None]
                    serve(4)
                    v, ttfas = serve(args.serving_requests)
                    line["serving"] = {"value": v, "unit": UNIT, "requests": args.serving_requests, "concurrent": conc, "chunk_frames": args.chunk,
                                       "ttfa_ms_first_wave_mean": 1000.0 * float(np.mean(sorted(ttfas)[:conc])) if ttfas else None,
                                       "what": "serving.BatchScheduler (continuous batching, windowed streaming codec per utterance on four codec lanes, "
                                               "host work beside the next launch): all requests submitted at once, audio streamed back per chunk"}
                except Exception as ex:  # a reported extra: never fail the bench on it
                    line["serving"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:200]}
            model_b.model.engine.close()
            del model_b
            torch.cuda.empty_cache()
        if world == 1 and args.anchor_frames > 0:
            # same-box GPU anchor (SURVEY.md §2c): the reference's execution style — static caches, attention over all slots
            # with a mask, CUDA-graph replays of the talker step and the predictor loop — restated on the same weights
            # (oracle/graph_anchor.py).  Reported beside decode_ms_per_frame; greedy, no codec, frame loop only.
            try:
                from oracle.graph_anchor import GraphAnchor
                from qwen3_tts_cuda_graphs_b200.weights import init_synthetic
                torch.cuda.empty_cache()
                wts = init_synthetic(model.model.cfg, seed=0, skip_text_embedding=True)
                anchor = GraphAnchor(model.model.cfg, wts, max_seq_len=2048, device=dev)
                anchor.capture()
                ms = anchor.time_frames(tie, tpe, args.anchor_frames)
                line["gpu_anchor"] = {
                    "ms_per_frame": ms, "frames": args.anchor_frames, "rtf_frame_loop_only": FRAME_S * 1000.0 / ms,
                    "what": "oracle restated in the reference's style (StaticCache + masks over max_seq_len=2048 slots + torch.cuda.CUDAGraph "
                            "replays of talker step and 15-step predictor loop, eager glue as generate.py:149-199), greedy, same B200, same weights",
                    "ours_ms_per_frame": avg_ms / args.chunk,
                }
                del anchor, wts
                torch.cuda.empty_cache()
            except Exception as ex:  # the anchor is a reported extra: never fail the bench on it
                line["gpu_anchor"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:200]}
        if world == 1 and not args.no_cpu_baseline:
            arm = CpuOracleArm(args.model, args.cpu_frames, args.chunk)
            t0 = time.perf_counter()
            reps = 0
            while reps < 1 or (time.perf_counter() - t0 < 12.0 and reps < 4):
                arm.step()
                reps += 1
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": reps * args.cpu_frames * FRAME_S / dt, "unit": UNIT, "cores": arm.cores,
                                    "kind": "port", "sample": f"{reps} x [{arm.sample}]"}
        print(json.dumps(line), flush=True)
    try:
        os.remove(ref_wav)
    except OSError:
        pass
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
