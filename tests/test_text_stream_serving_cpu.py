"""Open text in the serving layer against doubles (no GPU): serving.BatchScheduler with TTSRequest(text_open=True) and the
WebSocket endpoint /v1/audio/speech/stream of server.py.  A waiting stream (status.done = 4) is running, not finished; no launch
happens while every running stream waits; push_text wakes the loop; a silent request is cancelled after text_timeout and a
cancelled waiting request frees its slot; chunks are whole chunk_frames except the last."""
import threading
import time
import types

import numpy as np
import pytest
import torch

from qwen3_tts_cuda_graphs_b200.serving import _DONE, BatchScheduler, RequestHandle, TTSRequest

pytestmark = pytest.mark.timeout(120)
SPF = 1920
CF = 4


class OpenEngine:
    """Streams keyed by slot; a frame's codes row is [request key, frame index, 0, ...]; frame g needs trailing row g of the
    stream's text, and a stream whose row has not arrived while the text is open waits (done = 4), as on the device."""

    def __init__(self, max_streams=4):
        self.device = torch.device("cpu")
        self.max_streams, self.lockstep_group, self.max_seq_len, self.max_frames = max_streams, 16, 64, 4096
        self.st = {s: dict(n=0, done=3, key=-1, eos_at=10 ** 9, codes=[], rows=0, open=False, gs=0) for s in range(max_streams)}
        self.launches = []  # [slots with done == 0 at the launch's start]
        self.events = []

    def retire_stream(self, s):
        self.st[s]["done"] = self.st[s]["done"] or 3
        self.events.append(("retire", s))

    def set_text_conditioning(self, s, tth, tpe):
        self.st[s].update(rows=int(tth.shape[0]), open=False)

    def set_stream_policy(self, s, policy):
        pass

    def open_text(self, s, tpe):
        self.st[s].update(rows=0, open=True)

    def append_text(self, s, rows, close=False):
        st = self.st[s]
        st["rows"] += int(rows.shape[0])
        st["open"] = st["open"] and not close
        if st["done"] == 4 and (not st["open"] or st["gs"] < st["rows"]):
            st["done"] = 0

    def prefill(self, s, embeds, n_pad, policy):
        st = self.st[s]
        key, eos_at = int(embeds[0, 0]), int(embeds[0, 1])
        st.update(n=0, key=key, eos_at=eos_at, codes=[], gs=0)
        st["done"] = 4 if st["open"] and st["rows"] == 0 else 0
        self.events.append(("prefill", s))

    def decode_frames(self, hi, n, policy, sub):
        live = [s for s in range(hi) if self.st[s]["done"] == 0]
        self.launches.append(live)
        for s in live:
            st = self.st[s]
            for _ in range(n):
                if st["n"] >= st["eos_at"]:
                    st["done"] = 1
                    break
                st["codes"].append([st["key"], st["n"]] + [0] * 14)
                st["n"] += 1
                st["gs"] += 1
                if st["open"] and st["gs"] >= st["rows"]:
                    st["done"] = 4
                    break

    def status(self, s):
        st = self.st[s]
        return types.SimpleNamespace(n_frames=st["n"], done=st["done"] if st["done"] in (1, 2, 4) else 0, gen_step=st["gs"], error=0)

    def read_codes(self, s, first, n):
        return torch.tensor(self.st[s]["codes"][first:first + n], dtype=torch.int64)


class FakeDecoder:
    def __init__(self):
        self.cfg = types.SimpleNamespace(trans_conv_trim="right", sample_rate=24000)
        self.device = torch.device("cpu")
        self._plans = {}

    def decode(self, codes, skip_samples=0):
        return codes[:, 1].float().repeat_interleave(SPF)


class FakeTTS:
    """ref_audio "key:eos_at" keys the request; the text goes through the synthetic tokenizer."""

    def __init__(self, engine):
        from qwen3_tts_cuda_graphs_b200.base_model import SyntheticTokenizer
        from qwen3_tts_cuda_graphs_b200.codec import SpeechTokenizer
        from qwen3_tts_cuda_graphs_b200.config import preset

        cfg = preset("tiny")
        tok = SpeechTokenizer(FakeDecoder())
        talker = types.SimpleNamespace(device=torch.device("cpu"), config=types.SimpleNamespace(hidden_size=8),
                                       text_projection=lambda x: x,
                                       get_text_embeddings=lambda: (lambda t: t.float().unsqueeze(-1).repeat(1, 8)))
        inner = types.SimpleNamespace(speech_tokenizer=tok, tts_model_type="base", tts_model_size="0b6", talker=talker,
                                      config=types.SimpleNamespace(tts_eos_token_id=cfg.tts_eos_token_id))
        self.model = types.SimpleNamespace(engine=engine, model=inner, tokenizer=SyntheticTokenizer(cfg))
        self.sample_rate = 24000
        self.predictor_graph = types.SimpleNamespace(policy=lambda: None)
        self.prompts = []

    def _prepare_generation(self, text, ref_audio, ref_text, language="Auto", **kw):
        self.prompts.append(text)
        key, eos_at = (int(x) for x in ref_audio.split(":"))
        tie = torch.zeros(1, 5, 8)
        tie[0, 0, 0], tie[0, 0, 1] = key, eos_at
        return self.model.model, None, None, tie, torch.ones(1, 5, dtype=torch.long), torch.zeros(1, 3, 8), torch.zeros(1, 1, 8), None

    @staticmethod
    def _to_numpy(a):
        return a.flatten().float().cpu().numpy()


def _open(key, text="", eos_at=10 ** 9, frames=200, **kw):
    return TTSRequest(text, ref_audio=f"{key}:{eos_at}", language="English", max_new_tokens=frames, do_sample=False,
                      non_streaming_mode=False, text_open=True, **kw)


def _closed(key, frames, eos_at=10 ** 9):
    return TTSRequest("closed text here", ref_audio=f"{key}:{eos_at}", language="English", max_new_tokens=frames, do_sample=False)


def _frames_ok(h, key, n):
    codes = torch.cat(h.codes)
    assert codes.shape == (n, 16) and torch.equal(codes[:, 1], torch.arange(n)) and (codes[:, 0] == key).all()
    sizes = [int(c.shape[0]) for c in h.codes]
    assert all(s == CF for s in sizes[:-1]) and 0 < sizes[-1] <= CF  # whole chunks, only the last one shorter


def _wait(cond, t=10.0):
    t0 = time.time()
    while not cond():
        assert time.time() - t0 < t, "timed out"
        time.sleep(0.01)


def test_waiting_is_running_no_launch_while_all_wait_and_push_text_wakes():
    eng = OpenEngine(max_streams=2)
    with BatchScheduler(FakeTTS(eng), chunk_frames=CF, overlap_codec="none") as sched:
        h = sched.submit(_open(7, "hello "))
        _wait(lambda: ("prefill", 0) in eng.events)
        time.sleep(0.3)
        assert eng.launches == [] and h.finish_reason is None  # prefilled without a second token: waits, is not finished
        assert sched._active[0].waiting
        h.push_text("big brown fox jumps over ")
        _wait(lambda: len(eng.launches) > 0)
        time.sleep(0.3)
        assert h.finish_reason is None
        h.push_text("the lazy dog")
        h.close_text()
        with pytest.raises(ValueError):
            h.push_text("more")
        h.result(timeout=10)
    assert h.finish_reason == "length"  # after the text the stream runs on tts_pad until its budget
    _frames_ok(h, 7, 200)
    assert all(live for live in eng.launches)  # no launch in which every running stream waited


def test_open_requests_beside_ordinary_ones_from_a_feeding_thread():
    eng = OpenEngine(max_streams=8)
    words = "one two three four five six seven eight nine ten eleven twelve".split()
    with BatchScheduler(FakeTTS(eng), chunk_frames=CF, overlap_codec="none", mixed_policies=True) as sched:
        opens = [sched.submit(_open(10 + i, eos_at=9 + 3 * i)) for i in range(4)]
        closed = [sched.submit(_closed(20 + i, 13 + i)) for i in range(2)]

        def feed(h, seed):
            rng = np.random.default_rng(seed)
            for w in words:
                time.sleep(float(rng.uniform(0, 0.02)))
                h.push_text(w + " ")
            h.close_text()

        ts = [threading.Thread(target=feed, args=(h, i)) for i, h in enumerate(opens)]
        for t in ts:
            t.start()
        for i, h in enumerate(opens):
            h.result(timeout=20)
            assert h.finish_reason == "stop"
            _frames_ok(h, 10 + i, 9 + 3 * i)
        for i, h in enumerate(closed):
            h.result(timeout=20)
            _frames_ok(h, 20 + i, 13 + i)
        for t in ts:
            t.join()


def test_text_timeout_cancels_a_silent_request_and_frees_its_slot():
    eng = OpenEngine(max_streams=1)
    with BatchScheduler(FakeTTS(eng), chunk_frames=CF, overlap_codec="none", text_timeout=0.3) as sched:
        silent = sched.submit(_open(1, "only these words "))
        silent.result(timeout=10)
        assert silent.finish_reason == "text_timeout"
        never = sched.submit(_open(2, ""))  # no text at all: times out before it takes a slot
        never.result(timeout=10)
        assert never.finish_reason == "text_timeout"
        h = sched.submit(_closed(3, 6))
        h.result(timeout=10)
        _frames_ok(h, 3, 6)
    assert ("retire", 0) in eng.events


def test_cancelling_a_waiting_request_frees_its_slot():
    eng = OpenEngine(max_streams=1)
    with BatchScheduler(FakeTTS(eng), chunk_frames=CF, overlap_codec="none") as sched:
        w = sched.submit(_open(1, "a b c "))
        _wait(lambda: 0 in sched._active and sched._active[0].waiting)
        w.cancel()
        w.result(timeout=10)
        assert w.finish_reason == "cancelled"
        h = sched.submit(_closed(2, 5))
        h.result(timeout=10)
        _frames_ok(h, 2, 5)


def test_submit_time_refusals():
    eng = OpenEngine(max_streams=1)
    sched = BatchScheduler(FakeTTS(eng), chunk_frames=CF)
    with pytest.raises(ValueError):
        sched.submit(_open(1, "x ", xvec_only=False))
    with pytest.raises(ValueError):
        sched.submit(TTSRequest("x ", ref_audio="1:9", text_open=True))  # voice clone with non_streaming_mode=True
    h = sched.submit(_closed(1, 4))
    with pytest.raises(ValueError):
        h.push_text("x")
    with pytest.raises(ValueError):
        h.close_text()


# ---- WebSocket protocol against a stand-in backend -------------------------------------------------------------------------
class EchoBackend:
    """Every piece of text becomes one chunk of 4 samples of 0.25; the request ends when its text is closed."""

    def __init__(self):
        self.handles = []
        self.requests = []

    def submit(self, req):
        assert req.text_open
        self.requests.append(req)
        h = RequestHandle(req, len(self.handles))
        h._wake = threading.Event()
        self.handles.append(h)

        def run():
            while True:
                pieces, closed, _ = h._take_text()
                for _p in pieces:
                    h.q.put((np.full(4, 0.25, dtype=np.float32), 24000, {"chunk_steps": 2}))
                if closed:
                    h.finish_reason = "stop"
                    h.q.put(_DONE)
                    return
                if h.cancelled:
                    h.finish_reason = "cancelled"
                    h.q.put(_DONE)
                    return
                h._wake.wait(0.01)
                h._wake.clear()

        threading.Thread(target=run, daemon=True).start()
        return h


VOICES = {"alloy": {"ref_audio": "a.wav", "ref_text": "", "language": "English"}}


def _client(backend):
    from starlette.testclient import TestClient

    from qwen3_tts_cuda_graphs_b200 import server
    return TestClient(server.create_app([backend], VOICES, None))


def test_websocket_streams_pcm_then_done():
    b = EchoBackend()
    with _client(b).websocket_connect("/v1/audio/speech/stream") as ws:
        ws.send_json({"voice": "alloy", "seed": 5, "response_format": "pcm"})
        for w in ("Hello ", "there, ", "friend."):
            ws.send_json({"text": w})
        ws.send_json({"close": True})
        chunks = [ws.receive_bytes() for _ in range(3)]
        done = ws.receive_json()
    from qwen3_tts_cuda_graphs_b200.server import to_pcm16
    assert chunks == [to_pcm16(np.full(4, 0.25, dtype=np.float32))] * 3
    assert done == {"event": "done", "finish_reason": "stop", "frames": 6}
    assert b.requests[0].seed == 5 and b.requests[0].kind == "voice_clone" and not b.requests[0].non_streaming_mode


@pytest.mark.parametrize("first,later", [
    ({"voice": "nobody", "response_format": "pcm"}, None),
    ({"voice": "alloy", "response_format": "wav"}, None),
    ({"response_format": "pcm"}, None),
    ({"voice": "alloy", "response_format": "pcm"}, {"txt": "x"}),
    ({"voice": "alloy", "response_format": "pcm"}, {"text": "x" * 1001}),
])
def test_websocket_bad_input_gets_error_and_1008(first, later):
    from starlette.websockets import WebSocketDisconnect

    b = EchoBackend()
    with _client(b).websocket_connect("/v1/audio/speech/stream") as ws:
        ws.send_json(first)
        if later is not None:
            ws.send_json(later)
        msg = ws.receive_json()
        while "event" not in msg:  # pragma: no cover - no audio precedes the error here
            msg = ws.receive_json()
        assert msg["event"] == "error" and msg["detail"]
        with pytest.raises(WebSocketDisconnect) as e:
            ws.receive_json()
        assert e.value.code == 1008
    for h in b.handles:  # a refused open request does not keep decoding
        _wait(lambda: h.cancelled or h.finish_reason is not None)


def test_websocket_disconnect_cancels_the_request():
    b = EchoBackend()
    with _client(b).websocket_connect("/v1/audio/speech/stream") as ws:
        ws.send_json({"voice": "alloy", "response_format": "pcm"})
        ws.send_json({"text": "Hello "})
        ws.receive_bytes()
    _wait(lambda: b.handles and b.handles[0].cancelled)
