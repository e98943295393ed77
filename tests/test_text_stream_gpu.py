"""Incremental text input (fq3.h: fq3_open_text / fq3_append_text; text_stream.py).

The contract: whatever the arrival schedule of its text rows, an open stream's codes equal, bit for bit, the codes of the same
stream with the whole text given up front — at the engine level in every frame program, and through the public streaming
generators, whose `str` call's codes and audio an iterable of pieces reproduces."""
import numpy as np
import pytest
import torch

from helpers import make_cfg, make_engine, make_weights, synth_prompt

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

N_FRAMES = 24


def _sp(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy
    return SamplingPolicy(**kw)


def _sub(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SubPolicy
    return SubPolicy(**kw)


GREEDY = dict(do_sample=False, repetition_penalty=1.05, min_new_tokens=2)
SAMPLED = dict(do_sample=True, top_k=50, temperature=0.9, repetition_penalty=1.05, min_new_tokens=2, seed=4242)


@pytest.fixture(scope="module")
def tiny():
    cfg = make_cfg("tiny-CustomVoice")
    w = make_weights(cfg, seed=0)
    eng = make_engine(cfg, w, max_seq_len=256, max_streams=16)
    yield cfg, eng
    eng.close()


def _codes(eng, idx):
    st = eng.status(idx)
    assert st.error == 0
    return eng.read_codes(idx, 0, st.n_frames), st


def _closed(eng, prompt, n_rows, pol, sub, own_policy=False):
    """The stream with the first n_rows text rows given up front, alone in slot 0, one launch."""
    tie, tam, tth, tpe = prompt
    eng.set_stream_policy(0, pol if own_policy else None)
    eng.set_text_conditioning(0, tth[0, :n_rows].cuda(), tpe.cuda())
    eng.prefill(0, tie[0].cuda(), 0, pol)
    eng.decode_frames(1, N_FRAMES, pol, sub)
    codes, _ = _codes(eng, 0)
    eng.set_stream_policy(0, None)
    return codes


# schedule(launch k, rows given so far, R) -> (rows to append before launch k, close)
SCHEDULES = {
    "all_then_close": lambda k, g, R: (R, True) if k == 0 else (0, False),
    "one_per_launch": lambda k, g, R: (1, g + 1 == R) if g < R else (0, False),
    "nothing_at_prefill": lambda k, g, R: (0, False) if k < 2 else ((2, False) if g + 2 < R else (R - g, True)),
    "burst_after_wait": lambda k, g, R: (0, False) if k < 5 else ((R - g, True) if k == 5 else (0, False)),
    "close_without_rows": lambda k, g, R: (3, False) if k == 0 else ((0, False) if k < 4 else ((0, True) if k == 4 else (0, False))),
}


def _rows_total(name, R):
    return 3 if name == "close_without_rows" else R


def _run_open(eng, slots, prompts, schedules, pol, sub, launch, n_streams, check_wait=True):
    """Open streams in `slots` (others of [0, n_streams) must be set up by the caller) follow their schedules; launches of
    `launch` frames until every open stream has N_FRAMES frames or has finished.  Returns {slot: codes}."""
    given = {s: 0 for s in slots}
    closed = {s: False for s in slots}
    for s, prompt in zip(slots, prompts):
        tie, tam, tth, tpe = prompt
        eng.open_text(s, tpe.cuda())
        eng.prefill(s, tie[0].cuda(), 0, pol)
    for k in range(200):
        for s, prompt, sched in zip(slots, prompts, schedules):
            if closed[s]:
                continue
            R = prompt[2].shape[1]
            n, close = sched(k, given[s], R)
            if n or close:
                eng.append_text(s, prompt[2][0, given[s]:given[s] + n].cuda(), close=close)
                given[s] += n
                closed[s] = close
        before = {s: eng.status(s) for s in slots}
        eng.decode_frames(n_streams, launch, pol, sub)
        after = {s: eng.status(s) for s in slots}
        for s in slots:
            if check_wait and before[s].done == 4:
                assert after[s].done == 4 and after[s].n_frames == before[s].n_frames, (s, k)
                assert after[s].gen_step == before[s].gen_step and after[s].position == before[s].position
        if all(after[s].done in (1, 2) or after[s].n_frames >= N_FRAMES for s in slots):
            break
    else:
        raise AssertionError("open streams did not finish")
    return {s: _codes(eng, s)[0] for s in slots}


def _same(got, want):
    """got ran until it had at least N_FRAMES frames or finished; want is the closed-text run of N_FRAMES frames."""
    if want.shape[0] < N_FRAMES:
        assert got.shape[0] == want.shape[0]  # the same EOS frame
    else:
        assert got.shape[0] >= N_FRAMES
    m = min(got.shape[0], want.shape[0])
    assert torch.equal(got[:m], want[:m])


@pytest.mark.parametrize("schedule", sorted(SCHEDULES))
@pytest.mark.parametrize("launch", [1, 3, 8])
@pytest.mark.parametrize("mode", ["greedy", "sampled", "own_policy"])
def test_single_stream_any_schedule_matches_closed_text(tiny, schedule, launch, mode):
    cfg, eng = tiny
    prompt = synth_prompt(cfg, T=14, R=10, seed=3)
    pol = _sp(**(GREEDY if mode == "greedy" else SAMPLED))
    sub = _sub(do_sample=mode != "greedy", top_k=50, temperature=0.9)
    own = mode == "own_policy"
    want = _closed(eng, prompt, _rows_total(schedule, 10), pol, sub, own_policy=own)
    eng.set_stream_policy(0, pol if own else None)
    got = _run_open(eng, [0], [prompt], [SCHEDULES[schedule]], pol, sub, launch, 1)[0]
    eng.set_stream_policy(0, None)
    _same(got, want)


def test_waiting_stream_reports_done_4_and_resumes(tiny):
    cfg, eng = tiny
    prompt = synth_prompt(cfg, T=14, R=6, seed=5)
    pol, sub = _sp(**{**GREEDY, "min_new_tokens": 8}), _sub(do_sample=False)  # no EOS in the frames this test counts
    tie, tam, tth, tpe = prompt
    eng.open_text(0, tpe.cuda())
    eng.prefill(0, tie[0].cuda(), 0, pol)
    st = eng.status(0)
    assert st.done == 4 and st.n_frames == 0 and st.gen_step == 0  # no second text token yet: prefilled, waiting
    eng.decode_frames(1, 4, pol, sub)
    st2 = eng.status(0)
    assert (st2.done, st2.n_frames, st2.position, st2.token) == (4, 0, st.position, st.token)
    eng.append_text(0, tth[0, :2].cuda())
    assert eng.status(0).done == 0
    eng.decode_frames(1, 8, pol, sub)
    st3 = eng.status(0)
    assert st3.done == 4 and st3.n_frames == 2 and st3.gen_step == 2  # frames 0 and 1 used rows 0 and 1


@pytest.mark.parametrize("n_streams,wide", [(2, False), (5, True), (16, True)])
def test_lockstep_streams_stall_independently(tiny, monkeypatch, n_streams, wide):
    """Each open stream stalls at its own frames beside streams that never stall and streams that are not open; every stream
    equals its single-stream closed-text run (2 streams: the reference-shaped program; 5, 16: the wide one)."""
    cfg, eng = tiny
    from qwen3_tts_cuda_graphs_b200._lib import Fq3Error

    monkeypatch.setenv("FQ3_WIDE_FROM", "3")  # fq3_decode_frames: the wide program from three streams on
    sub = _sub(do_sample=True, top_k=50, temperature=0.9)
    launch_pol = _sp(**SAMPLED)
    prompts = [synth_prompt(cfg, T=9 + (i * 5) % 13, R=4 + (i * 3) % 9, seed=60 + i) for i in range(n_streams)]
    pols = [_sp(**{**SAMPLED, "seed": 100 + i, "top_k": 20 + i}) for i in range(n_streams)]
    names = sorted(SCHEDULES)
    kinds = ["open" if i % 3 != 2 else "closed" for i in range(n_streams)]  # every third stream is not open
    try:
        for i in range(n_streams):
            eng.set_stream_policy(i, pols[i])
            if kinds[i] == "closed":
                tie, tam, tth, tpe = prompts[i]
                eng.set_text_conditioning(i, tth[0].cuda(), tpe.cuda())
                eng.prefill(i, tie[0].cuda(), 0, launch_pol)
        slots = [i for i in range(n_streams) if kinds[i] == "open"]
        scheds = [SCHEDULES[names[i % len(names)]] for i in slots]
        got = _run_open(eng, slots, [prompts[i] for i in slots], scheds, launch_pol, sub, 3, n_streams)
        closed_got = {i: _codes(eng, i)[0] for i in range(n_streams) if kinds[i] == "closed"}
        # which frame program ran: the talker-logits hook answers after a reference-shaped launch only (fq3.h)
        if wide:
            with pytest.raises(Fq3Error):
                eng.debug_talker_logits(0)
        else:
            eng.debug_talker_logits(0)
    finally:
        for i in range(n_streams):
            eng.set_stream_policy(i, None)
    for i in range(n_streams):
        R = prompts[i][2].shape[1]
        rows = _rows_total(names[i % len(names)], R) if kinds[i] == "open" else R
        want = _closed(eng, prompts[i], rows, pols[i], sub, own_policy=True)
        _same(got[i] if kinds[i] == "open" else closed_got[i], want)


def test_lockstep_16_streams_full_depth_0p6b():
    cfg = make_cfg("0.6B-CustomVoice")
    w = make_weights(cfg, seed=1)
    eng = make_engine(cfg, w, max_seq_len=256, max_streams=16, max_frames=64)
    try:
        sub = _sub(do_sample=True, top_k=50, temperature=0.9)
        prompts = [synth_prompt(cfg, T=12 + i % 5, R=5 + i % 7, seed=200 + i) for i in range(16)]
        pols = [_sp(**{**SAMPLED, "seed": 300 + i}) for i in range(16)]
        for i in range(16):
            eng.set_stream_policy(i, pols[i])
        names = sorted(SCHEDULES)
        got = _run_open(eng, list(range(16)), prompts, [SCHEDULES[names[i % len(names)]] for i in range(16)], pols[0], sub, 4, 16)
        for i in range(16):
            eng.set_stream_policy(i, None)
        for i in range(16):
            want = _closed(eng, prompts[i], _rows_total(names[i % len(names)], prompts[i][2].shape[1]), pols[i], sub, own_policy=True)
            _same(got[i], want)
    finally:
        eng.close()


def test_abi_edges(tiny):
    from qwen3_tts_cuda_graphs_b200._lib import Fq3Error

    cfg, eng = tiny
    H = cfg.talker.hidden_size
    pol, sub = _sp(**GREEDY), _sub(do_sample=False)
    prompt = synth_prompt(cfg, T=14, R=8, seed=9)
    tie, tam, tth, tpe = prompt
    want = _closed(eng, prompt, 8, pol, sub)
    # appending to a stream whose text is closed (set_text_conditioning, or a close) fails
    with pytest.raises(Fq3Error):
        eng.append_text(0, tth[0, :1].cuda())
    eng.open_text(0, tpe.cuda())
    eng.append_text(0, tth[0, :1].cuda(), close=True)
    with pytest.raises(Fq3Error):
        eng.append_text(0, tth[0, :1].cuda())
    # past max_seq_len rows
    eng.open_text(0, tpe.cuda())
    eng.append_text(0, torch.zeros(250, H, dtype=torch.bfloat16, device="cuda"))
    with pytest.raises(RuntimeError) as too_long:
        eng.append_text(0, torch.zeros(7, H, dtype=torch.bfloat16, device="cuda"))
    assert not isinstance(too_long.value, Fq3Error)  # -FQ3_E_TOO_LONG, not -FQ3_E_INVALID
    # a reused slot given its text up front decodes as before
    assert torch.equal(_closed(eng, prompt, 8, pol, sub), want)
    # retiring a waiting stream
    eng.open_text(0, tpe.cuda())
    eng.prefill(0, tie[0].cuda(), 0, pol)
    assert eng.status(0).done == 4
    eng.retire_stream(0)
    assert eng.status(0).done == 3
    eng.set_text_conditioning(0, tth[0].cuda(), tpe.cuda())


# ---- public API ------------------------------------------------------------------------------------------------------------
TEXT = "the quick brown fox jumps over the lazy dog. speak slowly, calm voice!"


def _load(name):
    from qwen3_tts_cuda_graphs_b200 import FasterQwen3TTS
    return FasterQwen3TTS.from_pretrained(name, device="cuda", dtype=torch.bfloat16, max_seq_len=256)


def _splits(text):
    words = text.split(" ")
    yield "words", [w + " " for w in words[:-1]] + [words[-1]]
    yield "chars", list(text)
    rng = np.random.default_rng(7)
    cuts = sorted(set(int(x) for x in rng.integers(1, len(text), 12)))
    yield "mid_word", [text[a:b] for a, b in zip([0] + cuts, cuts + [len(text)])]


@pytest.fixture(scope="module")
def ref_wav(tmp_path_factory):
    import wave
    p = tmp_path_factory.mktemp("audio") / "ref.wav"
    sr = 24000
    t = np.arange(int(1.2 * sr)) / sr
    with wave.open(str(p), "wb") as wf:
        wf.setnchannels(1)
        wf.setsampwidth(2)
        wf.setframerate(sr)
        wf.writeframes((0.3 * np.sin(2 * np.pi * 220 * t) * 32767).astype(np.int16).tobytes())
    return str(p)


def _collect(gen):
    chunks = list(gen)
    return [a for a, _, _ in chunks], [t for _, _, t in chunks]


@pytest.mark.parametrize("kind", ["CustomVoice", "VoiceDesign", "Base"])
def test_public_generators_pieces_equal_str_call(kind, ref_wav):
    tts = _load(f"tiny-{kind}")
    try:
        from qwen3_tts_cuda_graphs_b200.text_stream import MAX_PROJECTION_ROWS

        # the one-shot prompt's projection call: bos / eos / pad, the instruct ids, 3 role ids and the text ids
        tok = tts.model.tokenizer
        n_rows = 3 + (len(tok.instruct("a calm voice")) if kind == "VoiceDesign" else 0) + 3 + len(tok.assistant(TEXT)[3:-5])
        assert n_rows <= MAX_PROJECTION_ROWS
        if kind == "CustomVoice":
            spk = tts.model.get_supported_speakers()[0]
            call = lambda text, **kw: tts.generate_custom_voice_streaming(text, spk, "English", **kw)
        elif kind == "VoiceDesign":
            call = lambda text, **kw: tts.generate_voice_design_streaming(text, "a calm voice", "English", **kw)
        else:
            call = lambda text, **kw: tts.generate_voice_clone_streaming(text, "English", ref_wav, "", xvec_only=True,
                                                                        non_streaming_mode=False, **kw)
        for do_sample in (False, True):
            kw = dict(max_new_tokens=40, chunk_size=8, do_sample=do_sample)
            torch.manual_seed(11)
            want, want_t = _collect(call(TEXT, **kw))
            assert len(want) >= 2
            for name, pieces in _splits(TEXT):
                assert "".join(pieces) == TEXT
                torch.manual_seed(11)
                got, got_t = _collect(call(iter(pieces), **kw))
                assert [g.shape for g in got] == [w.shape for w in want], (kind, name, do_sample)
                for g, w in zip(got, want):
                    assert np.array_equal(g, w), (kind, name, do_sample)
                assert [t["chunk_steps"] for t in got_t] == [t["chunk_steps"] for t in want_t]
                assert got_t[-1]["is_final"]
    finally:
        tts.model.engine.close()


def test_open_codes_equal_str_codes():
    """The codes themselves (generate_open against fast_generate_streaming on the same prompt), sampled."""
    from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy
    from qwen3_tts_cuda_graphs_b200.streaming import fast_generate_streaming
    from qwen3_tts_cuda_graphs_b200.text_stream import TextFeed, generate_open

    tts = _load("tiny-CustomVoice")
    try:
        spk = tts.model.get_supported_speakers()[0]
        m, talker, config, tie, tam, tth, tpe = tts._prepare_generation_custom(TEXT, "English", spk, None)
        kw = dict(max_new_tokens=40, temperature=0.9, top_k=50, do_sample=True, repetition_penalty=1.05, chunk_size=8)
        want = torch.cat([c for c, _ in fast_generate_streaming(
            talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth, tts_pad_embed=tpe,
            config=config, predictor_graph=tts.predictor_graph, talker_graph=tts.talker_graph, seed=99, **kw)])

        def prepare(s):
            _, t, _, a, b, _, c = tts._prepare_generation_custom(s, "English", spk, None)
            return a, b, c, t

        for _, pieces in _splits(TEXT):
            feed = TextFeed(tts.model.tokenizer.assistant, m.config.tts_eos_token_id)
            pol = lambda: SamplingPolicy(do_sample=True, top_k=50, temperature=0.9, repetition_penalty=1.05, min_new_tokens=2,
                                         suppress_tail=1024, seed=99)
            got = torch.cat([c for c, _ in generate_open(tts.talker_graph, tts.predictor_graph, prepare, feed, iter(pieces), pol,
                                                         40, 8)])
            assert torch.equal(got, want)
            assert feed.ids[:-1] == tts.model.tokenizer.assistant(TEXT)[3:-5]
    finally:
        tts.model.engine.close()


def test_public_refusals(ref_wav, monkeypatch):
    tts = _load("tiny-Base")
    try:
        with pytest.raises(ValueError):
            list(tts.generate_voice_clone_streaming(iter(["hello ", "world"]), "English", ref_wav, "ref words", xvec_only=False,
                                                    non_streaming_mode=False))
        with pytest.raises(ValueError):
            list(tts.generate_voice_clone_streaming(iter(["hello ", "world"]), "English", ref_wav, "", xvec_only=True,
                                                    non_streaming_mode=True))
        from qwen3_tts_cuda_graphs_b200 import generate
        monkeypatch.setattr(generate, "is_fused", lambda *a: False)
        with pytest.raises(ValueError):
            list(tts.generate_voice_clone_streaming(iter(["hello ", "world"]), "English", ref_wav, "", xvec_only=True,
                                                    non_streaming_mode=False))
    finally:
        tts.model.engine.close()


# ---- serving ---------------------------------------------------------------------------------------------------------------
OPEN_TEXTS = ["the quick brown fox jumps over the lazy dog.", "speak slowly, calm voice!", "hello world, this is a test.",
              "reference clip says this quick test."]
CLOSED_TEXTS = ["short parity test.", "the lazy dog says hello."]


def _single_open_layout(tts, ref_wav, text, n, pol, chunk):
    """The one-shot streaming run of the same request (streaming-text layout, x-vector clone) in slot 0 with the same seed."""
    from qwen3_tts_cuda_graphs_b200.streaming import fast_generate_streaming

    m, talker, config, tie, tam, tth, tpe, ref_codes = tts._prepare_generation(
        text, ref_wav, "", language="English", xvec_only=True, non_streaming_mode=False, append_silence=True)
    stream = fast_generate_streaming(talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth,
                                     tts_pad_embed=tpe, config=config, chunk_size=chunk, seed=pol["seed"],
                                     **tts._gen_kwargs(n, 2, pol["temperature"], pol["top_k"], 1.0, True, 1.05))
    codes, audio = [], []

    def capture(s):
        for c, info in s:
            codes.append(c)
            yield c, info

    for a, _, _ in tts._stream_audio(m, capture(stream), ref_codes, chunk):
        audio.append(a)
    return torch.cat(codes).cpu(), np.concatenate(audio)


def test_scheduler_open_requests_fed_from_threads_match_one_shot_runs(ref_wav):
    import threading
    import time

    from qwen3_tts_cuda_graphs_b200 import FasterQwen3TTS
    from qwen3_tts_cuda_graphs_b200.serving import BatchScheduler, TTSRequest

    tts = FasterQwen3TTS.from_pretrained("tiny-Base", device="cuda", dtype=torch.bfloat16, max_seq_len=256, max_streams=6)
    chunk, n = 8, 40
    texts = OPEN_TEXTS + CLOSED_TEXTS
    pols = [dict(temperature=0.7 + 0.1 * i, top_k=20 + 5 * i, seed=500 + i) for i in range(len(texts))]
    try:
        want = [_single_open_layout(tts, ref_wav, t, n, p, chunk) for t, p in zip(texts, pols)]
        sched = BatchScheduler(tts, chunk_frames=chunk, codec_mode="windowed", mixed_policies=True, seed=3).start()
        try:
            def req(i, **kw):
                return TTSRequest(kw.pop("text", texts[i]), ref_audio=ref_wav, language="English", max_new_tokens=n,
                                  non_streaming_mode=False, **pols[i], **kw)

            words = [t.split(" ") for t in OPEN_TEXTS]
            handles = [sched.submit(req(i, text=words[i][0] + " ", text_open=True)) for i in range(4)]
            handles += [sched.submit(req(4 + j)) for j in range(2)]

            def feed(h, ws, seed):
                rng = np.random.default_rng(seed)
                for k, w in enumerate(ws[1:]):
                    time.sleep(float(rng.uniform(0.0, 0.15)))
                    h.push_text(w + (" " if k + 2 < len(ws) else ""))
                h.close_text()

            ts = [threading.Thread(target=feed, args=(handles[i], words[i], i)) for i in range(4)]
            for t in ts:
                t.start()
            audio = [[a for a, _, _ in h] for h in handles]
            for t in ts:
                t.join()
            for i, h in enumerate(handles):
                assert h.finish_reason in ("length", "stop"), (i, h.finish_reason)
                assert torch.equal(torch.cat(h.codes), want[i][0]), f"request {i}: codes differ from the one-shot run"
                a = np.concatenate(audio[i])
                assert a.shape == want[i][1].shape and np.array_equal(a, want[i][1]), f"request {i}: audio differs"
            # a cancelled waiting request frees its slot
            w = sched.submit(req(0, text="hello ", text_open=True))
            t0 = time.time()
            while not any(a.handle is w and a.waiting for a in list(sched._active.values())):
                assert time.time() - t0 < 30
                time.sleep(0.01)
            slot = next(s for s, a in list(sched._active.items()) if a.handle is w)
            w.cancel()
            list(w)
            assert w.finish_reason == "cancelled"
            t0 = time.time()
            while slot in sched._active:
                assert time.time() - t0 < 30
                time.sleep(0.01)
            h = sched.submit(req(4))  # the freed slot serves the next request
            list(h)
            assert torch.equal(torch.cat(h.codes), want[4][0])
        finally:
            sched.stop()
    finally:
        tts.model.engine.close()
