"""Per-stream sampling policy in the lock-step frame loop (fq3.h: fq3_set_stream_policy; DESIGN.md §3.1, §3.5).

The contract: a stream's codes in a launch whose streams carry different policies equal, bit for bit, the codes of a
single-stream run in slot 0 with a launch-wide policy of the same values and seed — whatever the slot, the frame program
(reference-shaped / wide), the lock-step group, the prefill path (dense head / tail, chunked + left-padded).  Streams without a
record sample exactly as before.  And the serving scheduler in mixed mode gives every sampled request the codes and audio of
its single-stream streaming run with the same seed."""
import time
import wave

import numpy as np
import pytest
import torch

from helpers import make_cfg, make_engine, make_weights, synth_prompt

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]


def _sp(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy
    return SamplingPolicy(**kw)


def _sub(**kw):
    from qwen3_tts_cuda_graphs_b200.engine import SubPolicy
    return SubPolicy(**kw)


# greedy, several top_k / temperatures, top_p < 1 (the generic sampler), repetition penalty 1.0 / 1.3, min_new_tokens 0 / 2 / 8
POLICIES = [
    dict(do_sample=False, repetition_penalty=1.0, min_new_tokens=0),
    dict(do_sample=True, top_k=50, temperature=0.9, repetition_penalty=1.05, min_new_tokens=2, seed=11),
    dict(do_sample=True, top_k=5, temperature=0.7, repetition_penalty=1.3, min_new_tokens=8, seed=12),
    dict(do_sample=True, top_k=50, top_p=0.8, temperature=1.0, repetition_penalty=1.0, min_new_tokens=2, seed=13),
    dict(do_sample=True, top_k=20, temperature=1.3, repetition_penalty=1.3, min_new_tokens=0, seed=14),
    dict(do_sample=False, repetition_penalty=1.3, min_new_tokens=8),
    dict(do_sample=True, top_k=0, top_p=0.9, temperature=1.1, repetition_penalty=1.05, min_new_tokens=0, seed=15),
    dict(do_sample=True, top_k=50, temperature=0.9, repetition_penalty=1.05, min_new_tokens=2, seed=2**63 + 5),
]
LAUNCH = dict(do_sample=True, top_k=30, temperature=0.8, repetition_penalty=1.1, min_new_tokens=1, seed=777)


@pytest.fixture(scope="module")
def tiny():
    cfg = make_cfg("tiny")
    w = make_weights(cfg, seed=0)
    eng = make_engine(cfg, w, max_streams=40)
    yield cfg, w, eng
    eng.close()


def _prefill(eng, idx, prompt, pol, n_pad=0, dense=None):
    tie, tam, tth, tpe = prompt
    eng.set_text_conditioning(idx, tth[0].cuda(), tpe.cuda())
    eng.prefill(idx, tie[0].cuda(), n_pad, pol, dense=dense)


def _codes(eng, idx):
    st = eng.status(idx)
    assert st.error == 0
    return eng.read_codes(idx, 0, st.n_frames)


def _single(eng, prompt, pol, sub, n_frames, n_pad=0, dense=None):
    """Slot 0, no record, the launch's policy: the reference-shaped program with one stream."""
    eng.set_stream_policy(0, None)
    _prefill(eng, 0, prompt, pol, n_pad, dense)
    first = eng.status(0).token
    eng.decode_frames(1, n_frames, pol, sub)
    return first, _codes(eng, 0)


def _batch(eng, prompts, pols, sub, n_frames, launch):
    """Streams 0..n-1 in one lock-step decode (two launches: the second starts from the state the first left); pols[i] is
    stream i's own policy or None (no record).  Clears every record afterwards."""
    n = len(prompts)
    try:
        for i, prompt in enumerate(prompts):
            eng.set_stream_policy(i, pols[i])
            _prefill(eng, i, prompt, launch)
        eng.decode_frames(n, n_frames // 2, launch, sub)
        eng.decode_frames(n, n_frames - n_frames // 2, launch, sub)
        return [_codes(eng, i) for i in range(n)]
    finally:
        for i in range(n):
            eng.set_stream_policy(i, None)


def _mixed_vs_single(eng, cfg, n_streams, n_frames, sub, lens=(14, 9, 21, 5), none_every=3):
    prompts = [synth_prompt(cfg, T=lens[i % len(lens)], seed=40 + i) for i in range(n_streams)]
    launch = _sp(**LAUNCH)
    pols = [None if (none_every and i % none_every == none_every - 1) else _sp(**POLICIES[i % len(POLICIES)])
            for i in range(n_streams)]
    got = _batch(eng, prompts, pols, sub, n_frames, launch)
    # streams without a record: as in a launch where no stream has one
    plain = _batch(eng, prompts, [None] * n_streams, sub, n_frames, launch) if any(p is None for p in pols) else None
    bad = []
    for i in range(n_streams):
        if pols[i] is None:
            want = plain[i]
        else:
            _, want = _single(eng, prompts[i], pols[i], sub, n_frames)
        if got[i].shape != want.shape or not torch.equal(got[i], want):
            bad.append(i)
    assert not bad, (bad, [pols[i] for i in bad])
    return got


@pytest.mark.parametrize("n_streams,wide_from", [(2, None), (4, "5"), (5, None), (16, None), (40, None)])
def test_mixed_policies_match_single_stream_tiny(tiny, monkeypatch, n_streams, wide_from):
    """2 streams and 4 with FQ3_WIDE_FROM=5: the reference-shaped program; 5, 16: the wide one; 40: three lock-step groups."""
    cfg, w, eng = tiny
    if wide_from:
        monkeypatch.setenv("FQ3_WIDE_FROM", wide_from)
    got = _mixed_vs_single(eng, cfg, n_streams, 12, _sub(do_sample=True, top_k=50, temperature=0.9))
    assert any(g.shape[0] > 1 for g in got)


def test_mixed_policies_greedy_predictor(tiny):
    cfg, w, eng = tiny
    _mixed_vs_single(eng, cfg, 8, 10, _sub(do_sample=False))


def test_mixed_policies_full_depth_16_streams():
    """The real 0.6B stack at full depth, 16 streams with contexts from 14 to 201 positions."""
    cfg = make_cfg("0.6B-Base")
    w = make_weights(cfg, seed=0)
    eng = make_engine(cfg, w, max_streams=16, max_seq_len=256)
    try:
        _mixed_vs_single(eng, cfg, 16, 8, _sub(do_sample=True, top_k=50, temperature=0.9), lens=(14, 60, 137, 201), none_every=5)
    finally:
        eng.close()


def test_same_policy_and_seed_in_different_slots_give_identical_codes(tiny):
    cfg, w, eng = tiny
    prompt = synth_prompt(cfg, T=12, seed=3)
    pol = _sp(do_sample=True, top_k=40, temperature=1.2, repetition_penalty=1.1, min_new_tokens=2, seed=424242)
    prompts = [synth_prompt(cfg, T=8 + i, seed=60 + i) for i in range(14)]
    pols = [_sp(**POLICIES[i % len(POLICIES)]) for i in range(14)]
    prompts[3] = prompts[11] = prompt
    pols[3] = pols[11] = pol
    got = _batch(eng, prompts, pols, _sub(do_sample=True), 16, _sp(**LAUNCH))
    assert got[3].shape[0] > 2 and torch.equal(got[3], got[11])
    # and without records the two slots draw differently (the launch key depends on the slot)
    plain = _batch(eng, prompts, [None] * 14, _sub(do_sample=True), 16, _sp(do_sample=True, top_k=40, temperature=1.2, seed=424242))
    assert not torch.equal(plain[3], plain[11])


@pytest.mark.parametrize("mode", ["full", "tail", "chunked"])
def test_first_token_honours_the_record(tiny, monkeypatch, mode):
    """fq3_prefill_head (dense, default), fq3_prefill_tail (FQ3_DENSE_FULL=0) and the chunked, left-padded fq3_prefill."""
    cfg, w, eng = tiny
    if mode != "chunked":
        monkeypatch.setenv("FQ3_DENSE_FULL", "1" if mode == "full" else "0")
        if eng._dense is not None:
            eng._dense.close()
        eng._dense, eng._dense_tried = None, False
    T, n_pad = 40, (3 if mode == "chunked" else 0)
    dense = mode != "chunked"
    prompt = synth_prompt(cfg, T=T, seed=8)
    sub = _sub(do_sample=True)
    firsts = set()
    for seed in range(6):
        pol = _sp(do_sample=True, top_k=0, temperature=2.0, repetition_penalty=1.0, min_new_tokens=0, seed=1000 + seed)
        want_first, want = _single(eng, prompt, pol, sub, 4, n_pad=n_pad, dense=dense)
        if dense:
            assert eng._dense is not None and eng._dense.full == (mode == "full")
        try:
            eng.set_stream_policy(0, _sp(do_sample=False))
            eng.set_stream_policy(5, pol)
            for i in range(6):
                _prefill(eng, i, prompt if i == 5 else synth_prompt(cfg, T=T, seed=20 + i), _sp(**LAUNCH), n_pad, dense)
            assert eng.status(5).token == want_first, seed
            eng.decode_frames(6, 4, _sp(**LAUNCH), sub)
            assert torch.equal(_codes(eng, 5), want), seed
        finally:
            eng.set_stream_policy(0, None)
            eng.set_stream_policy(5, None)
        firsts.add(want_first)
    assert len(firsts) > 1  # the record's sampled policy really drew (a greedy launch policy would give one token)
    if eng._dense is not None:
        eng._dense.close()
    eng._dense, eng._dense_tried = None, False


def test_no_change_without_a_record(tiny):
    """After set_stream_policy(k, None) and after fq3_reset_stream, slot k samples exactly as on an engine that never had a
    record."""
    cfg, w, eng = tiny
    fresh = make_engine(cfg, w, max_streams=4)
    launch = _sp(**LAUNCH)
    sub = _sub(do_sample=True)
    prompts = [synth_prompt(cfg, T=10 + i, seed=80 + i) for i in range(3)]

    def run(e, before=None):
        for i, p in enumerate(prompts):
            if before is not None and i == 2:
                before(e)
            _prefill(e, i, p, launch)
        e.decode_frames(3, 12, launch, sub)
        return [_codes(e, i) for i in range(3)]

    try:
        want = run(fresh)
        own = _sp(do_sample=True, top_k=3, temperature=0.5, seed=5)
        cleared = run(eng, lambda e: (e.set_stream_policy(2, own), e.set_stream_policy(2, None)))
        reset = run(eng, lambda e: (e.set_stream_policy(2, own), e.reset_stream(2)))
        with_record = run(eng, lambda e: e.set_stream_policy(2, own))
        eng.set_stream_policy(2, None)
    finally:
        fresh.close()
    for i in range(3):
        assert torch.equal(cleared[i], want[i]) and torch.equal(reset[i], want[i]), i
    assert torch.equal(with_record[0], want[0]) and torch.equal(with_record[1], want[1])
    assert not torch.equal(with_record[2], want[2])  # the record did apply


def test_set_stream_policy_refuses_bad_values(tiny):
    from qwen3_tts_cuda_graphs_b200._lib import Fq3Error

    cfg, w, eng = tiny
    for bad in (dict(top_k=-1), dict(top_p=0.0), dict(top_p=1.5), dict(temperature=0.0), dict(suppress_tail=cfg.talker.vocab_size + 1),
                dict(repetition_penalty=0.0)):
        with pytest.raises(Fq3Error):
            eng.set_stream_policy(1, _sp(**bad))
    with pytest.raises(Fq3Error):
        eng.set_stream_policy(40, _sp())
    eng.set_stream_policy(1, _sp(do_sample=False, temperature=0.0))  # greedy: the temperature is not used
    eng.set_stream_policy(1, None)


def test_fast_generate_batch_with_policies(tiny):
    from qwen3_tts_cuda_graphs_b200.generate import fast_generate_batch

    cfg, w, eng = tiny
    tg = type("TG", (), {})()
    tg.engine = eng
    pg = type("PG", (), {"policy": staticmethod(lambda: _sub(do_sample=True))})()
    prompts = [synth_prompt(cfg, T=9 + i, seed=90 + i) for i in range(6)]
    pols = [_sp(**POLICIES[i]) for i in range(6)]
    out, _ = fast_generate_batch(tg, pg, [tuple(t.cuda() for t in p) for p in prompts], max_new_tokens=10, seed=1, policies=pols)
    for i in range(6):
        _, want = _single(eng, prompts[i], pols[i], _sub(do_sample=True), 10)
        assert out[i] is not None and torch.equal(out[i].cpu(), want), i


# ---- the serving scheduler in mixed mode ------------------------------------------------------------------------------------
TEXTS = [
    "Short parity test.",
    "The quick brown fox jumps over the lazy dog and keeps running through the field.",
    "Hello world!",
    "Speak slowly, in a calm voice, and do not stop before the sentence has ended.",
    "One more request that arrives late.",
]
LENGTHS = [40, 21, 64, 33, 16]
REQ_POLICIES = [
    dict(temperature=0.9, top_k=50, repetition_penalty=1.05, min_new_tokens=2, seed=101),
    dict(temperature=0.6, top_k=10, repetition_penalty=1.3, min_new_tokens=8, seed=202),
    dict(temperature=1.0, top_k=50, top_p=0.85, repetition_penalty=1.0, min_new_tokens=0, seed=303),
    dict(do_sample=False, repetition_penalty=1.05, min_new_tokens=2, seed=0),
    dict(temperature=1.2, top_k=30, repetition_penalty=1.1, min_new_tokens=2, seed=404),
]


@pytest.fixture(scope="module")
def ref_wav(tmp_path_factory):
    p = tmp_path_factory.mktemp("audio") / "ref.wav"
    sr = 24000
    t = np.arange(int(1.2 * sr)) / sr
    pcm = (0.3 * np.sin(2 * np.pi * 220 * t) * 32767).astype(np.int16)
    with wave.open(str(p), "wb") as wf:
        wf.setnchannels(1)
        wf.setsampwidth(2)
        wf.setframerate(sr)
        wf.writeframes(pcm.tobytes())
    return str(p)


@pytest.fixture(scope="module")
def tts():
    from qwen3_tts_cuda_graphs_b200 import FasterQwen3TTS

    m = FasterQwen3TTS.from_pretrained("tiny-Base", device="cuda", dtype=torch.bfloat16, max_seq_len=256, max_streams=6)
    yield m  # the predictor samples too (its seed is the request's)
    m.model.engine.close()


def _single_stream(tts, ref_wav, text, n, pol, chunk=8):
    """fast_generate_streaming(..., seed=S) in slot 0, through the windowed codec of the streaming API."""
    from qwen3_tts_cuda_graphs_b200.streaming import fast_generate_streaming

    # the prompt TTSRequest's defaults build (and generate_voice_clone_streaming's)
    m, talker, config, tie, tam, tth, tpe, ref_codes = tts._prepare_generation(
        text, ref_wav, "", language="English", xvec_only=True, non_streaming_mode=True, append_silence=True)
    kw = dict(dict(do_sample=True, temperature=0.9, top_k=50, top_p=1.0, repetition_penalty=1.05, min_new_tokens=2), **pol)
    seed = kw.pop("seed")
    stream = fast_generate_streaming(talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth,
                                     tts_pad_embed=tpe, config=config, chunk_size=chunk, seed=seed,
                                     **tts._gen_kwargs(n, kw["min_new_tokens"], kw["temperature"], kw["top_k"], kw["top_p"],
                                                       kw["do_sample"], kw["repetition_penalty"]))
    codes, audio = [], []
    for a, sr, info in tts._stream_audio(m, _capture(stream, codes), ref_codes, chunk):
        audio.append(a)
    return torch.cat(codes).cpu(), np.concatenate(audio)


def _capture(stream, into):
    for chunk, info in stream:
        into.append(chunk)
        yield chunk, info


def test_scheduler_mixed_policies_match_single_stream_runs(tts, ref_wav):
    from qwen3_tts_cuda_graphs_b200.serving import BatchScheduler, TTSRequest

    want = [_single_stream(tts, ref_wav, t, n, p) for t, n, p in zip(TEXTS, LENGTHS, REQ_POLICIES)]
    sched = BatchScheduler(tts, chunk_frames=8, codec_mode="windowed", mixed_policies=True, seed=9).start()
    try:
        def req(i):
            return TTSRequest(TEXTS[i], ref_audio=ref_wav, language="English", max_new_tokens=LENGTHS[i], **REQ_POLICIES[i])

        handles = {0: sched.submit(req(0)), 1: sched.submit(req(1))}
        first = next(iter(handles[0]))            # request 0 is mid-utterance ...
        handles[2] = sched.submit(req(2))         # ... when the next ones arrive
        handles[3] = sched.submit(req(3))
        time.sleep(0.05)
        handles[4] = sched.submit(req(4))
        audio = {0: [first[0]] + [a for a, _, _ in handles[0]]}
        for i in range(1, 5):
            audio[i] = [a for a, _, _ in handles[i]]
    finally:
        sched.stop()
    for i in range(5):
        h = handles[i]
        got = torch.cat(h.codes)
        assert h.finish_reason in ("length", "stop")
        assert torch.equal(got, want[i][0]), f"request {i}: codes differ from the single-stream run"
        a = np.concatenate(audio[i])
        assert a.shape == want[i][1].shape and np.array_equal(a, want[i][1]), f"request {i}: audio differs"
    assert sched.stats["max_batch"] >= 3  # requests of different policies shared launches
    # the scheduler left no record behind: the single-stream API in slot 0 is unchanged
    again = _single_stream(tts, ref_wav, TEXTS[0], LENGTHS[0], REQ_POLICIES[0])
    assert torch.equal(again[0], want[0][0])
