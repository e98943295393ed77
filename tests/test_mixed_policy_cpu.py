"""Host logic of per-stream sampling policies (fq3.h: fq3_set_stream_policy) against engine / model doubles — no GPU: the
scheduler's mixed mode (no cohorts, the request's policy and seed set on its slot before its prefill, a seed that does not depend
on the slot, one fixed launch policy), cohort mode refusing a seed, fast_generate_batch(policies=...),
generate_voice_clone_batch(per_request=...), the HTTP front's `seed` field and its 400s.  tests/test_mixed_policy_gpu.py holds
the device side bit for bit."""
import types

import numpy as np
import pytest
import torch
from starlette.testclient import TestClient

from qwen3_tts_cuda_graphs_b200 import server
from qwen3_tts_cuda_graphs_b200.engine import SamplingPolicy
from qwen3_tts_cuda_graphs_b200.serving import BatchScheduler, TTSRequest

from test_serving_cpu import SPF, FakeEngine, FakeTTS, _audio_ok

pytestmark = pytest.mark.timeout(120)


class PolicyEngine(FakeEngine):
    """FakeEngine + per-slot policy records: events gain ("policy", slot, SamplingPolicy | None); a launch records the launch
    policy object and, per live slot, the policy that slot samples with."""

    def __init__(self, **kw):
        super().__init__(**kw)
        self.records = {}
        self.launch_pols = []

    def set_stream_policy(self, s, policy):
        assert policy is None or isinstance(policy, SamplingPolicy)
        if policy is not None:
            policy.validate()
        self.records[s] = policy
        self.events.append(("policy", s, policy))

    def prefill(self, s, embeds, n_pad, policy):
        super().prefill(s, embeds, n_pad, policy)
        self.events[-1] = ("prefill", s, self.records.get(s))

    def decode_frames(self, hi, n, policy, sub):
        live = [s for s in range(hi) if self.st[s]["done"] == 0]
        self.launch_pols.append((policy, {s: self.records.get(s) for s in live}))
        super().decode_frames(hi, n, policy, sub)


FOUR = [dict(do_sample=False), dict(temperature=0.7, top_k=20), dict(temperature=1.1, top_p=0.8, repetition_penalty=1.3),
        dict(temperature=0.9, min_new_tokens=8, seed=1234)]


def _req(key, frames, eos_at=10 ** 9, **kw):
    kw = dict(dict(do_sample=True), **kw)
    return TTSRequest(f"{key},{eos_at}", ref_audio="v.wav", language="English", max_new_tokens=frames, **kw)


def test_mixed_mode_requests_of_several_policies_share_launches_from_the_first_chunk():
    eng = PolicyEngine(max_streams=4)
    tts = FakeTTS(eng)
    sched = BatchScheduler(tts, chunk_frames=8, mixed_policies=True, seed=3)
    hs = [sched.submit(_req(100 + i, 24, **FOUR[i])) for i in range(4)]
    with sched:
        for i, h in enumerate(hs):
            h.id_key = 100 + i
            _audio_ok(h, 24)
    assert eng.launches[0][1] == [0, 1, 2, 3]               # all four policies in the first launch: none was deferred
    assert len(eng.launches) == 3 and all(live == [0, 1, 2, 3] for _, live, _ in eng.launches)
    launch_pol = eng.launch_pols[0][0]
    for pol, per_slot in eng.launch_pols:
        assert pol == launch_pol                             # one fixed launch-wide policy ...
        assert all(p is not None and p != launch_pol for p in per_slot.values())  # ... that no live stream uses
    assert sched.stats["max_batch"] == 4


def test_the_slots_policy_is_set_before_its_prefill_with_the_requests_values_and_seed():
    eng = PolicyEngine(max_streams=4)
    tts = FakeTTS(eng)
    with BatchScheduler(tts, chunk_frames=8, mixed_policies=True, seed=3) as sched:
        hs = [sched.submit(_req(10 + i, 9, **FOUR[i])) for i in range(4)]
        for h in hs:
            h.result()
    prefills = [(i, e) for i, e in enumerate(eng.events) if e[0] == "prefill"]
    assert len(prefills) == 4
    for i, (_, slot, pol) in prefills:
        assert eng.events[i - 1] == ("policy", slot, pol)    # set right before the prefill, on the same slot
        h = next(h for h in hs if h.id == slot)  # admitted in order into slots 0..3
        r = h.request
        assert (pol.do_sample, pol.top_k, pol.top_p, pol.temperature, pol.repetition_penalty, pol.min_new_tokens) == \
            (r.do_sample, r.top_k, r.top_p, r.temperature, r.repetition_penalty, r.min_new_tokens)
        assert pol.seed == (r.seed if r.seed is not None else sched.request_seed(h))
    assert prefills[3][1][2].seed == 1234
    # a finished request's record is cleared with its slot: a later user of the slot samples with its own arguments
    assert all(eng.records[s] is None for s in range(4))


def test_a_derived_seed_depends_on_the_request_not_on_its_slot():
    seeds = []
    for cancel_first in (False, True):
        eng = PolicyEngine(max_streams=2)
        tts = FakeTTS(eng)
        sched = BatchScheduler(tts, chunk_frames=8, mixed_policies=True, seed=77)
        first = sched.submit(_req(1, 8))
        second = sched.submit(_req(2, 8, temperature=0.5))   # id 1, no seed of its own
        if cancel_first:
            first.cancel()                                    # never takes a slot: `second` lands in slot 0
        with sched:
            second.result()
            if not cancel_first:
                first.result()
        (slot, pol), = [(e[1], e[2]) for e in eng.events if e[0] == "prefill" and e[2].temperature == 0.5]
        seeds.append((slot, pol.seed))
    assert seeds[0][0] == 1 and seeds[1][0] == 0                # different slots ...
    assert seeds[0][1] == seeds[1][1]                          # ... same seed
    other = BatchScheduler(FakeTTS(PolicyEngine(max_streams=2)), mixed_policies=True, seed=78)
    h = other.submit(_req(2, 8))
    h = other.submit(_req(2, 8))
    assert other.request_seed(h) != seeds[0][1]                # the scheduler's seed enters the derivation


def test_cohort_mode_refuses_a_seed_and_mixed_mode_refuses_bad_values():
    eng = PolicyEngine(max_streams=2)
    sched = BatchScheduler(FakeTTS(eng), chunk_frames=8)
    with pytest.raises(ValueError, match="mixed_policies"):
        sched.submit(_req(1, 8, seed=5))
    mixed = BatchScheduler(FakeTTS(PolicyEngine(max_streams=2)), chunk_frames=8, mixed_policies=True)
    for bad in (dict(top_p=0.0), dict(top_p=1.2), dict(top_k=-1), dict(temperature=0.0), dict(seed=-1), dict(seed=2 ** 64),
                dict(repetition_penalty=0.0), dict(min_new_tokens=-1)):
        with pytest.raises(ValueError):
            mixed.submit(_req(1, 8, **bad))
    mixed.submit(_req(1, 8, do_sample=False, temperature=0.0))  # greedy: the temperature is not used


def test_cohort_mode_is_unchanged_and_sets_no_records():
    eng = PolicyEngine(max_streams=4)
    with BatchScheduler(FakeTTS(eng), chunk_frames=8) as sched:
        hs = [sched.submit(_req(10 + i, 16, do_sample=False)) for i in range(3)]
        for h in hs:
            h.result()
    assert not [e for e in eng.events if e[0] == "policy"]


# ---- fast_generate_batch / generate_voice_clone_batch ------------------------------------------------------------------------
class BatchEngine:
    def __init__(self):
        self.max_streams, self.lockstep_group, self.max_seq_len, self.max_frames = 4, 16, 64, 4096
        self.device = torch.device("cpu")
        self.log = []

    def set_text_conditioning(self, idx, tth, tpe):
        pass

    def set_stream_policy(self, idx, policy):
        self.log.append(("policy", idx, policy))

    def prefill(self, idx, embeds, n_pad, policy):
        self.log.append(("prefill", idx, policy))

    def decode_frames(self, n_streams, n_frames, policy, sub):
        self.log.append(("launch", n_streams, policy))

    def status(self, idx=0):
        return types.SimpleNamespace(n_frames=3, done=0, error=0)

    def read_codes(self, idx, first, n):
        return torch.full((n, 16), idx, dtype=torch.int64)


@pytest.fixture()
def no_cuda(monkeypatch):
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)


def _reqs(n, T=6, H=8):
    return [(torch.zeros(1, T, H), torch.ones(1, T, dtype=torch.long), torch.zeros(1, 1, H), torch.zeros(1, 1, H)) for _ in range(n)]


def test_fast_generate_batch_sets_each_streams_policy_before_its_prefill_and_clears_it(no_cuda):
    from qwen3_tts_cuda_graphs_b200.generate import fast_generate_batch

    eng = BatchEngine()
    tg, pg = types.SimpleNamespace(engine=eng), types.SimpleNamespace(policy=lambda: None)
    pols = [SamplingPolicy(temperature=0.5 + 0.1 * i, seed=10 + i) for i in range(6)]
    out, _ = fast_generate_batch(tg, pg, _reqs(6), max_new_tokens=8, seed=1, policies=pols)
    assert [c[0, 0].item() for c in out] == [0, 1, 2, 3, 0, 1]
    launches = [e for e in eng.log if e[0] == "launch"]
    assert [n for _, n, _ in launches] == [4, 2]
    launch_pol = launches[0][2]
    i = 0
    for g0, n in ((0, 4), (4, 2)):
        for s in range(n):
            assert eng.log[i] == ("policy", s, pols[g0 + s]) and eng.log[i + 1] == ("prefill", s, launch_pol)
            i += 2
        assert eng.log[i][0] == "launch"
        assert eng.log[i + 1:i + 1 + n] == [("policy", s, None) for s in range(n)]  # cleared after the group
        i += 1 + n
    # without policies: the path of before, no record is touched
    eng2 = BatchEngine()
    fast_generate_batch(types.SimpleNamespace(engine=eng2), pg, _reqs(3), max_new_tokens=8, seed=1)
    assert not [e for e in eng2.log if e[0] == "policy"]
    with pytest.raises(ValueError):
        fast_generate_batch(tg, pg, _reqs(3), policies=pols[:2])
    with pytest.raises(ValueError):
        fast_generate_batch(tg, pg, _reqs(1), policies=[dict(temperature=0.5)])


def test_fast_generate_batch_clears_the_records_when_a_prefill_fails(no_cuda):
    from qwen3_tts_cuda_graphs_b200.generate import fast_generate_batch

    eng = BatchEngine()
    eng.max_seq_len = 5
    reqs = _reqs(1, T=4) + _reqs(1, T=9)
    with pytest.raises(RuntimeError, match="Input is too long"):
        fast_generate_batch(types.SimpleNamespace(engine=eng), types.SimpleNamespace(policy=lambda: None), reqs,
                            policies=[SamplingPolicy(seed=1), SamplingPolicy(seed=2)])
    assert eng.log[-2:] == [("policy", 0, None), ("policy", 1, None)]


def test_generate_voice_clone_batch_per_request(monkeypatch):
    from qwen3_tts_cuda_graphs_b200 import generate
    from qwen3_tts_cuda_graphs_b200.model import FasterQwen3TTS

    seen = {}

    def fake_batch(tg, pg, reqs, **kw):
        seen.update(kw, n=len(reqs))
        return [torch.zeros(2, 16, dtype=torch.int64)] * len(reqs), {"frames": 2 * len(reqs), "total_s": 1.0, "audio_s_per_s": 1.0}

    monkeypatch.setattr(generate, "fast_generate_batch", fake_batch)
    fake = types.SimpleNamespace(
        _prepare_generation=lambda *a, **k: (None, None, None, torch.zeros(1, 4, 8), torch.ones(1, 4), torch.zeros(1, 1, 8),
                                             torch.zeros(1, 1, 8), None),
        talker_graph=None, predictor_graph=None, sample_rate=24000,
        _decode_full=lambda m, c, r: ([np.zeros(3840, dtype=np.float32)], 24000))
    call = FasterQwen3TTS.generate_voice_clone_batch
    audio, sr = call(fake, ["a", "b", "c"], "English", "v.wav", "", temperature=0.8, top_k=40, repetition_penalty=1.2,
                     per_request=[{"temperature": 0.5, "seed": 9}, {}, {"top_p": 0.7, "do_sample": False, "min_new_tokens": 0, "top_k": 5,
                                                                          "repetition_penalty": 1.0, "seed": 3}])
    assert len(audio) == 3 and sr == 24000 and seen["n"] == 3
    p0, p1, p2 = seen["policies"]
    assert (p0.temperature, p0.top_k, p0.repetition_penalty, p0.seed, p0.do_sample) == (0.5, 40, 1.2, 9, True)
    assert (p1.temperature, p1.top_k, p1.top_p, p1.min_new_tokens) == (0.8, 40, 1.0, 2) and 0 <= p1.seed < 2 ** 62
    assert (p2.top_p, p2.do_sample, p2.min_new_tokens, p2.top_k, p2.repetition_penalty, p2.seed) == (0.7, False, 0, 5, 1.0, 3)
    call(fake, ["a"], "English", "v.wav", "")
    assert seen["policies"] is None  # without per_request: the path of before
    with pytest.raises(ValueError, match="entries"):
        call(fake, ["a", "b"], "English", "v.wav", "", per_request=[{}])
    with pytest.raises(ValueError, match="unknown"):
        call(fake, ["a"], "English", "v.wav", "", per_request=[{"speed": 2.0}])
    with pytest.raises(ValueError, match="top_p"):
        call(fake, ["a"], "English", "v.wav", "", per_request=[{"top_p": 0.0}])


# ---- HTTP front ------------------------------------------------------------------------------------------------------------
class StubBackend:
    def __init__(self, refuse_seed=False):
        self.requests = []
        self.refuse_seed = refuse_seed

    def submit(self, req):
        from qwen3_tts_cuda_graphs_b200.serving import _DONE, RequestHandle

        if self.refuse_seed and req.seed is not None:
            raise ValueError("a per-request seed needs BatchScheduler(mixed_policies=True)")
        h = RequestHandle(req, len(self.requests))
        self.requests.append(req)
        h.q.put((np.zeros(2400, dtype=np.float32), 24000, {}))
        h.finish_reason = "stop"
        h.q.put(_DONE)
        return h


VOICES = {"alloy": {"ref_audio": "alloy.wav", "ref_text": "hi", "language": "English"},
          "seeded": {"speaker": "aiden", "language": "English", "seed": 42, "temperature": 0.6}}


def test_server_forwards_seed_and_answers_400_out_of_range():
    b = StubBackend()
    c = TestClient(server.create_app([b], VOICES, "alloy"))
    r = c.post("/v1/audio/speech", json={"input": "Hi", "voice": "alloy", "response_format": "pcm", "seed": 7})
    assert r.status_code == 200 and b.requests[-1].seed == 7
    r = c.post("/v1/audio/speech", json={"input": "Hi", "voice": "alloy", "response_format": "pcm"})
    assert r.status_code == 200 and b.requests[-1].seed is None
    r = c.post("/v1/audio/speech", json={"input": "Hi", "voice": "seeded", "response_format": "pcm"})
    assert r.status_code == 200 and b.requests[-1].seed == 42 and b.requests[-1].temperature == 0.6  # a voices entry's seed
    for bad in (-1, 2 ** 64):
        r = c.post("/v1/audio/speech", json={"input": "Hi", "voice": "alloy", "response_format": "pcm", "seed": bad})
        assert r.status_code == 400, bad
    n = len(b.requests)
    form = dict(text="Hello", mode="voice_clone", voice="alloy")
    r = c.post("/generate", data=dict(form, seed="11", temperature="0.5", top_k="7", repetition_penalty="1.2"))
    assert r.status_code == 200
    q = b.requests[-1]
    assert (q.seed, q.temperature, q.top_k, q.repetition_penalty) == (11, 0.5, 7, 1.2)
    r = c.post("/generate/stream", data=dict(form, seed="12"))
    assert r.status_code == 200 and b.requests[-1].seed == 12
    for bad in (dict(temperature="0"), dict(top_k="-3"), dict(repetition_penalty="0"), dict(seed="-5")):
        for path in ("/generate", "/generate/stream"):
            r = c.post(path, data=dict(form, **bad))
            assert r.status_code == 400, (path, bad)
    assert len(b.requests) == n + 2  # nothing out of range reached the backend


def test_server_answers_400_when_the_backend_refuses_a_seed():
    c = TestClient(server.create_app([StubBackend(refuse_seed=True)], VOICES, "alloy"))
    r = c.post("/v1/audio/speech", json={"input": "Hi", "voice": "alloy", "response_format": "pcm", "seed": 7})
    assert r.status_code == 400 and "mixed_policies" in r.text
    r = c.post("/generate", data=dict(text="Hello", mode="voice_clone", voice="alloy", seed="3"))
    assert r.status_code == 400
    assert c.get("/health").json()["in_flight"] == [0]


def test_server_parser_and_build_backends_take_mixed_policies(monkeypatch):
    import sys

    from qwen3_tts_cuda_graphs_b200 import model as model_mod
    from qwen3_tts_cuda_graphs_b200 import serving

    made = []

    class Sched:
        def __init__(self, tts, **kw):
            made.append(kw)

        def start(self):
            return self

    monkeypatch.setattr(model_mod.FasterQwen3TTS, "from_pretrained", classmethod(lambda cls, *a, **k: object()))
    monkeypatch.setattr(serving, "BatchScheduler", Sched)
    server.build_backends("m", 1, 4, 8, mixed_policies=True)
    server.build_backends("m", 1, 4, 8)
    assert made[0]["mixed_policies"] is True and made[1]["mixed_policies"] is False
    captured = {}
    monkeypatch.setattr(server, "build_backends", lambda *a, **k: captured.update(k) or (_ for _ in ()).throw(SystemExit(0)))
    monkeypatch.setitem(sys.modules, "uvicorn", types.SimpleNamespace(run=lambda *a, **k: None))
    with pytest.raises(SystemExit):
        server.main(["--ref-audio", "r.wav", "--mixed-policies", "--no-warmup"])
    assert captured["mixed_policies"] is True
