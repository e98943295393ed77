"""Cost and gain of incremental text input (fq3_open_text / fq3_append_text; DESIGN.md §3.1, text_stream.py).

(a) frame-step of 16 lock-step streams at 0.6B dims (synthetic weights, contexts of 60 positions), device events around one
    decode_frames launch of `--step-frames` frames: 16 open streams whose text is always ahead of them against the same streams
    with closed text, alternated three times.  The difference is the cost of the open-text test in the talker sampler.
(b) one stream of 0.6B- and 1.7B-CustomVoice (synthetic weights), words arriving at 5 / 20 / 100 words/s from a thread: time from
    the first piece to the first audio chunk of generate_custom_voice_streaming(text=<pieces>), against the one-shot str call made
    after the last piece (its time to first audio plus the time the text took to arrive), and the launches the stream spent
    waiting (status.done = 4 after a launch).
(c) `--sessions` concurrent open requests (TTSRequest(text_open=True), what the WebSocket endpoint submits) through
    serving.BatchScheduler(mixed_policies=True) on 0.6B-Base (synthetic weights, x-vector voice), each fed `--words` words at
    `--rate` words/s from its own thread, like an LLM's reply: audio-s/s (wall clock) and time from the first piece to the first
    audio chunk, p50 / p90.
usage: python scripts/text_stream_bench.py [--part a|b|c|abc] [--step-frames 64] [--words 40] [--sessions 16] [--rate 20]"""
import argparse
import json
import os
import queue
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ap = argparse.ArgumentParser()
ap.add_argument("--part", default="ab")
ap.add_argument("--step-frames", type=int, default=64, dest="step_frames")
ap.add_argument("--words", type=int, default=40)
ap.add_argument("--sessions", type=int, default=16)
ap.add_argument("--rate", type=float, default=20.0)
args = ap.parse_args()

print(json.dumps({"gpu": torch.cuda.get_device_name(0), "power_limit_w": os.popen(
    "nvidia-smi --query-gpu=power.limit --format=csv,noheader,nounits -i 0").read().strip()}), flush=True)


def part_a():
    from helpers import make_cfg, make_engine, make_weights, synth_prompt
    from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy, SubPolicy

    cfg = make_cfg("0.6B-Base")
    w = make_weights(cfg, seed=0, norm_jitter=0.0)
    ns, nf = 16, args.step_frames
    eng = make_engine(cfg, w, max_seq_len=1024, max_streams=ns, max_frames=2048)
    pol = SamplingPolicy(do_sample=True, temperature=0.9, top_k=50, repetition_penalty=1.05, min_new_tokens=10 ** 6, seed=1)
    sub = SubPolicy(do_sample=True, top_k=50, temperature=0.9)
    prompts = [synth_prompt(cfg, T=60, R=nf + 8, seed=1 + s) for s in range(ns)]
    ev = lambda: torch.cuda.Event(enable_timing=True)
    res = {"closed": [], "open_ahead": []}
    for rnd in range(3):
        for name in res:
            for s in range(ns):
                tie, tam, tth, tpe = prompts[s]
                if name == "closed":
                    eng.set_text_conditioning(s, tth[0].cuda(), tpe.cuda())
                else:
                    eng.open_text(s, tpe.cuda())
                    eng.append_text(s, tth[0].cuda())  # every row the launch needs, text still open
                eng.prefill(s, tie[0].cuda(), 0, pol)
            eng.decode_frames(ns, 4, pol, sub)  # warm
            a, b = ev(), ev()
            torch.cuda.synchronize()
            a.record()
            eng.decode_frames(ns, nf, pol, sub)
            b.record()
            torch.cuda.synchronize()
            st = [eng.status(s) for s in range(ns)]
            assert all(x.error == 0 and x.n_frames == nf + 4 and x.done == 0 for x in st), [(x.error, x.n_frames, x.done) for x in st]
            res[name].append(a.elapsed_time(b) / nf)
    print(json.dumps({"part": "a", "streams": ns, "frames": nf,
                      "ms_per_frame_step": {k: [round(v, 4) for v in vs] for k, vs in res.items()}}), flush=True)
    eng.close()


WORDS = ("the quick brown fox jumps over the lazy dog while a calm voice reads every word of this sentence aloud "
         "and the listener hears it before the writer has finished").split()


def part_b():
    from qwen3_tts_cuda_graphs_b200 import FasterQwen3TTS

    words = [WORDS[i % len(WORDS)] for i in range(args.words)]
    text = " ".join(words)
    for name in ("0.6B-CustomVoice", "1.7B-CustomVoice"):
        tts = FasterQwen3TTS.from_pretrained(f"synthetic://{name}", device="cuda", max_seq_len=512)
        spk = tts.model.get_supported_speakers()[0]
        kw = dict(max_new_tokens=200, min_new_tokens=200, chunk_size=8, do_sample=False)
        for _ in range(2):  # warm both paths
            list(tts.generate_custom_voice_streaming(text, spk, "English", **kw))
            list(tts.generate_custom_voice_streaming(iter([w + " " for w in words]), spk, "English", **kw))
        eng = tts.model.engine
        for rate in (5, 20, 100):
            q = queue.Queue()

            def writer():
                for i, w_ in enumerate(words):
                    q.put(w_ + (" " if i + 1 < len(words) else ""))
                    time.sleep(1.0 / rate)
                q.put(None)

            waits = {"launches_waiting": 0}
            dec = eng.decode_frames

            def counting(n_streams, n_frames, policy, sub):
                dec(n_streams, n_frames, policy, sub)
                waits["launches_waiting"] += int(eng.status(0).done == 4)

            eng.decode_frames = counting

            def pieces():
                while True:
                    p = q.get()
                    if p is None:
                        return
                    yield p

            t0 = time.perf_counter()
            threading.Thread(target=writer, daemon=True).start()
            gen = tts.generate_custom_voice_streaming(pieces(), spk, "English", **kw)
            next(gen)
            ttfa_open = time.perf_counter() - t0
            for _ in gen:
                pass
            del eng.decode_frames
            arrival = len(words) / rate
            t1 = time.perf_counter()
            next(tts.generate_custom_voice_streaming(text, spk, "English", **kw))
            ttfa_str = time.perf_counter() - t1
            print(json.dumps({"part": "b", "model": name, "words": len(words), "words_per_s": rate,
                              "first_piece_to_first_audio_ms": round(ttfa_open * 1000, 1),
                              "one_shot_after_last_piece_ms": round((arrival + ttfa_str) * 1000, 1),
                              "one_shot_ttfa_ms": round(ttfa_str * 1000, 1), **waits}), flush=True)
        eng.close()


def part_c():
    import wave

    import numpy as np

    from qwen3_tts_cuda_graphs_b200 import FasterQwen3TTS
    from qwen3_tts_cuda_graphs_b200.serving import BatchScheduler, TTSRequest

    ref = os.path.join(os.environ.get("TMPDIR", "/tmp"), "text_stream_bench_ref.wav")
    sr = 24000
    with wave.open(ref, "wb") as wf:
        wf.setnchannels(1)
        wf.setsampwidth(2)
        wf.setframerate(sr)
        wf.writeframes((0.3 * np.sin(2 * np.pi * 220 * np.arange(int(1.2 * sr)) / sr) * 32767).astype(np.int16).tobytes())
    tts = FasterQwen3TTS.from_pretrained("synthetic://0.6B-Base", device="cuda", max_seq_len=512, max_streams=args.sessions)
    words = [WORDS[i % len(WORDS)] for i in range(args.words)]
    for rnd in range(2):  # the first round warms the codec lanes
        with BatchScheduler(tts, chunk_frames=8, mixed_policies=True, seed=rnd) as sched:
            t0 = time.perf_counter()
            hs = [sched.submit(TTSRequest(words[0] + " ", ref_audio=ref, language="English", max_new_tokens=250,
                                          min_new_tokens=250, non_streaming_mode=False, text_open=True))
                  for _ in range(args.sessions)]

            def feed(h):
                for k, w_ in enumerate(words[1:]):
                    time.sleep(1.0 / args.rate)
                    h.push_text(w_ + (" " if k + 2 < len(words) else ""))
                h.close_text()

            ts = [threading.Thread(target=feed, args=(h,), daemon=True) for h in hs]
            for t in ts:
                t.start()
            frames = 0
            for h in hs:
                for _a, _sr, info in h:
                    frames += info["chunk_steps"]
            dt = time.perf_counter() - t0
            firsts = [h.ttfa_s for h in hs]  # the scheduler stamps a request's first audio chunk
        print(json.dumps({"part": "c", "round": rnd, "sessions": args.sessions, "words": len(words), "words_per_s": args.rate,
                          "audio_s_per_s": round(frames * 0.08 / dt, 1),
                          "first_piece_to_first_audio_ms_p50_p90": [round(float(np.percentile(firsts, q)) * 1000, 1) for q in (50, 90)]}),
              flush=True)
    tts.model.engine.close()


if "a" in args.part:
    part_a()
if "b" in args.part:
    part_b()
if "c" in args.part:
    part_c()
