"""Cost and gain of per-stream sampling policies (fq3_set_stream_policy; DESIGN.md §3.5, §7.1).

(a) frame-step of 16 lock-step streams at 0.6B dims (synthetic weights, contexts of 60 positions), device events around one
    decode_frames launch: one launch-wide policy for all streams vs 16 distinct per-stream policies with top_p = 1 vs the same
    with one stream at top_p = 0.9 (that stream takes the generic sorted-distribution sampler; its group waits for it).
(b) serving: `--requests` concurrent requests of `--frames` frames (EOS suppressed) whose policies cycle through four sampling
    policies in arrival order, through serving.BatchScheduler in cohort mode and with mixed_policies=True, alternated
    `--rounds` times: audio-s/s (wall clock) and time to first audio p50 / p90.
usage: python scripts/mixed_policy_bench.py [--part a|b|ab] [--requests 16] [--frames 250] [--rounds 2]"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ap = argparse.ArgumentParser()
ap.add_argument("--part", default="ab")
ap.add_argument("--requests", type=int, default=16)
ap.add_argument("--frames", type=int, default=250)
ap.add_argument("--rounds", type=int, default=2)
ap.add_argument("--step-frames", type=int, default=64, dest="step_frames")
args = ap.parse_args()

print(json.dumps({"gpu": torch.cuda.get_device_name(0), "power_limit_w": os.popen(
    "nvidia-smi --query-gpu=power.limit --format=csv,noheader,nounits -i 0").read().strip()}), flush=True)

FOUR = [dict(temperature=0.9, top_k=50, repetition_penalty=1.05),
        dict(temperature=0.7, top_k=20, repetition_penalty=1.1),
        dict(temperature=1.0, top_k=50, repetition_penalty=1.0),
        dict(temperature=0.8, top_k=30, repetition_penalty=1.2)]


def part_a():
    from helpers import make_cfg, make_engine, make_weights, synth_prompt
    from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy, SubPolicy

    cfg = make_cfg("0.6B-Base")
    w = make_weights(cfg, seed=0, norm_jitter=0.0)
    ns, nf = 16, args.step_frames
    eng = make_engine(cfg, w, max_seq_len=1024, max_streams=ns, max_frames=2048)
    big = 10 ** 6  # min_new_tokens: no stream stops early
    launch = SamplingPolicy(do_sample=True, temperature=0.9, top_k=50, repetition_penalty=1.05, min_new_tokens=big, seed=1)
    sub = SubPolicy(do_sample=True, top_k=50, temperature=0.9)
    distinct = [SamplingPolicy(do_sample=True, temperature=0.6 + 0.05 * i, top_k=10 + 5 * i, repetition_penalty=1.0 + 0.02 * i,
                               min_new_tokens=big, seed=100 + i) for i in range(ns)]
    one_top_p = list(distinct)
    one_top_p[7] = SamplingPolicy(**{**distinct[7].__dict__, "top_p": 0.9})
    cases = {"uniform": [None] * ns, "distinct_top_p_1": distinct, "distinct_one_top_p_0.9": one_top_p}
    prompts = [synth_prompt(cfg, T=60, seed=1 + s) for s in range(ns)]
    ev = lambda: torch.cuda.Event(enable_timing=True)
    res = {k: [] for k in cases}
    for rnd in range(3):
        for name, pols in cases.items():
            for s in range(ns):
                tie, tam, tth, tpe = prompts[s]
                eng.set_stream_policy(s, pols[s])
                eng.set_text_conditioning(s, tth[0].cuda(), tpe.cuda())
                eng.prefill(s, tie[0].cuda(), 0, launch)
            eng.decode_frames(ns, 4, launch, sub)  # warm
            a, b = ev(), ev()
            torch.cuda.synchronize()
            a.record()
            eng.decode_frames(ns, nf, launch, sub)
            b.record()
            torch.cuda.synchronize()
            st = [eng.status(s) for s in range(ns)]
            assert all(x.error == 0 and x.n_frames == nf + 4 for x in st), [(x.error, x.n_frames) for x in st]
            res[name].append(a.elapsed_time(b) / nf)
    for s in range(ns):
        eng.set_stream_policy(s, None)
    eng.close()
    out = {"part": "a", "what": f"ms per 16-stream frame-step, 0.6B dims, context 60..{60 + 4 + nf}, {nf} frames per launch, 3 rounds alternated",
           "ms_per_frame_step": {k: [round(x, 4) for x in v] for k, v in res.items()},
           "median": {k: round(float(np.median(v)), 4) for k, v in res.items()}}
    print(json.dumps(out), flush=True)


def part_b():
    import bench
    from qwen3_tts_cuda_graphs_b200 import FasterQwen3TTS
    from qwen3_tts_cuda_graphs_b200.serving import BatchScheduler, TTSRequest

    n = args.requests
    model = FasterQwen3TTS.from_pretrained("synthetic://0.6B-Base", device="cuda", dtype=torch.bfloat16, max_seq_len=1024, seed=0,
                                           max_streams=16)
    ref_wav = bench.make_ref_wav()
    texts = [bench.TEXT + f" Request number {i}." for i in range(n)]

    def run(mixed, n_req, frames):
        done = []
        with BatchScheduler(model, chunk_frames=8, max_concurrent=16, mixed_policies=mixed) as sched:
            def consume(h):
                a, sr = h.result()
                done.append((h, len(a) / sr))
            t0 = time.perf_counter()
            threads = []
            for i in range(n_req):
                h = sched.submit(TTSRequest(texts[i], ref_audio=ref_wav, ref_text=bench.REF_TEXT, language="English",
                                            max_new_tokens=frames, min_new_tokens=frames, **FOUR[i % 4]))
                th = threading.Thread(target=consume, args=(h,))
                th.start()
                threads.append(th)
            for th in threads:
                th.join()
            dt = time.perf_counter() - t0
            stats = dict(sched.stats)
        ttfa = np.array([h.ttfa_s for h, _ in done]) * 1000
        return {"mode": "mixed" if mixed else "cohort", "audio_s_per_s": round(sum(s for _, s in done) / dt, 1), "seconds": round(dt, 3),
                "ttfa_ms": {"p50": round(float(np.percentile(ttfa, 50)), 1), "p90": round(float(np.percentile(ttfa, 90)), 1)},
                "launches": stats["launches"], "max_batch": stats["max_batch"]}

    run(False, 4, 24)  # warm-up: plans, graphs, voice prompt cache, codec lanes
    run(True, 4, 24)
    for rnd in range(args.rounds):
        for mixed in (False, True):
            r = run(mixed, n, args.frames)
            r.update(part="b", round=rnd, requests=n, frames=args.frames, policies=4)
            print(json.dumps(r), flush=True)


if "a" in args.part:
    part_a()
if "b" in args.part:
    part_b()
