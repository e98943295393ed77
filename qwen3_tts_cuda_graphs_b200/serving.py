"""Continuous-batching scheduler over the lock-step frame loop (SURVEY.md §8 row f4, "serving layer ... on top of a
continuous-batching scheduler").

The reference's servers hold ONE lock around a bs = 1 model (`examples/openai_server.py:71,181`, `demo/server.py:167,517`):
requests queue behind each other and a 10-second utterance blocks everyone for 2–3 seconds.  This engine decodes up to
`fq3_lockstep_group` (16) utterances per weight sweep and more in groups (DESIGN.md §3.5), so the serving loop is:

    admit   waiting requests take free stream slots: prompt build -> reset -> prefill (one slot at a time, between two chunks)
    launch  ONE `fq3_decode_frames(high-water slot count, chunk_frames)` for every running utterance
    emit    while that launch runs, the previous chunk's codes go through the codec on a side stream (the decode grid leaves
            20 SMs free) and out to each request's queue
    retire  a slot whose utterance hit EOS / its length cap / the cache bound / was cancelled is parked with
            `fq3_retire_stream` so the others keep going, and is free for the next admit

A request joins at the next chunk boundary (≤ chunk_frames frame-steps away) and leaves without stopping anyone.  A stream's
tokens do not depend on its neighbours (batch-invariant arithmetic, DESIGN.md §3.5): under greedy decoding every request's
codes equal its single-stream run (`tests/test_serving_gpu.py`).  By default the sampling policy is a launch argument, so
requests are batched with requests of the same policy ("cohorts"); a request with another policy waits for the running cohort
to drain.  With `mixed_policies=True` every request carries its own policy and seed into its slot (fq3_set_stream_policy):
requests of any policies share every launch, and a sampled request draws exactly what its single-stream run with the same
seed draws, whatever slot it got (`tests/test_mixed_policy_gpu.py`).

A request can also be open (`TTSRequest(text_open=True)`): its text keeps arriving through `RequestHandle.push_text` /
`close_text`.  It is admitted once its first text token is committed (text_stream.TextFeed), the pieces it received are appended
to its slot before every launch, a stream waiting for text (status.done = 4) counts as running, no launch happens while every
running stream waits, and its audio goes out in whole chunks of `chunk_frames`, so it equals the one-shot run's.  A request whose
text stays silent for `text_timeout` seconds is cancelled.

All engine calls happen on the scheduler's own thread (the engine, like the reference's model, is not thread-safe).
"""
from __future__ import annotations

import logging
import queue
import threading
import time
from dataclasses import dataclass, field
from typing import Dict, Iterator, List, Optional, Tuple

import numpy as np
import torch

from .engine import SamplingPolicy

logger = logging.getLogger(__name__)

_DONE = object()


@dataclass
class TTSRequest:
    """One utterance.  `kind`: "voice_clone" (ref_audio / ref_text / xvec_only), "custom_voice" (speaker), "voice_design"
    (instruct) — the three generate_* families of the reference API (model.py:556, :829, :1004)."""

    text: str
    kind: str = "voice_clone"
    language: str = "Auto"
    ref_audio: Optional[object] = None
    ref_text: str = ""
    speaker: Optional[str] = None
    instruct: Optional[str] = None
    xvec_only: bool = True
    non_streaming_mode: bool = True
    append_silence: bool = True
    max_new_tokens: int = 2048
    min_new_tokens: int = 2
    temperature: float = 0.9
    top_k: int = 50
    top_p: float = 1.0
    do_sample: bool = True
    repetition_penalty: float = 1.05
    seed: Optional[int] = None  # sampling seed of this request (BatchScheduler(mixed_policies=True)); None: derived from its id
    text_open: bool = False  # the text keeps arriving: `text` is its first piece, RequestHandle.push_text / close_text the rest

    def policy_key(self) -> tuple:
        return (self.do_sample, self.top_k, self.top_p, self.temperature, self.repetition_penalty, self.min_new_tokens)


class RequestHandle:
    """What `submit` returns: iterate for (audio float32, sample_rate, info) chunks as they are decoded, or `result()` for the
    whole utterance.  `codes` collects the int64 [n, 16] codec ids chunk by chunk."""

    def __init__(self, req: TTSRequest, rid: int):
        self.request, self.id = req, rid
        self.q: "queue.Queue" = queue.Queue()
        self.codes: List[torch.Tensor] = []
        self.t_submit = time.time()
        self.t_first: Optional[float] = None
        self.t_done: Optional[float] = None
        self.finish_reason: Optional[str] = None
        self.cancelled = False
        self._sr = 24000
        self._wake: Optional[threading.Event] = None  # the scheduler's: set when text arrives or the request is cancelled
        self._text_lock = threading.Lock()
        self._pieces: List[str] = [req.text] if req.text_open and req.text else []
        self._text_closed = not req.text_open
        self._t_text = time.monotonic()  # when text last arrived (TTSRequest(text_open=True): BatchScheduler's text_timeout)
        self._text_feed = None  # text_stream.TextFeed, made and used by the scheduler thread

    def cancel(self):
        self.cancelled = True
        if self._wake is not None:
            self._wake.set()

    def push_text(self, piece: str):
        """Add a piece of an open request's text (thread-safe); the scheduler commits its tokens before its next launch."""
        if not self.request.text_open:
            raise ValueError("push_text: the request's text is not open (TTSRequest(text_open=True))")
        with self._text_lock:
            if self._text_closed:
                raise ValueError("push_text after close_text")
            self._pieces.append(str(piece))
            self._t_text = time.monotonic()
        if self._wake is not None:
            self._wake.set()

    def close_text(self):
        """End an open request's text (thread-safe; a second call does nothing)."""
        if not self.request.text_open:
            raise ValueError("close_text: the request's text is not open (TTSRequest(text_open=True))")
        with self._text_lock:
            self._text_closed = True
            self._t_text = time.monotonic()
        if self._wake is not None:
            self._wake.set()

    def _take_text(self) -> Tuple[List[str], bool, float]:
        """(pieces since the last call, text closed?, when text last arrived)."""
        with self._text_lock:
            pieces, self._pieces = self._pieces, []
            return pieces, self._text_closed, self._t_text

    def chunks(self, timeout: Optional[float] = None) -> Iterator[Tuple[np.ndarray, int, dict]]:
        """The utterance's chunks as they arrive; `timeout` (seconds, for the whole utterance) raises TimeoutError and cancels
        the request, so its slot is freed at the next chunk boundary."""
        deadline = None if timeout is None else time.monotonic() + timeout
        while True:
            try:
                item = self.q.get(timeout=None if deadline is None else max(0.0, deadline - time.monotonic()))
            except queue.Empty:
                self.cancel()
                raise TimeoutError(f"request {self.id}: no result within {timeout} s") from None
            if item is _DONE:
                return
            if isinstance(item, BaseException):
                raise item
            yield item

    def __iter__(self) -> Iterator[Tuple[np.ndarray, int, dict]]:
        return self.chunks()

    def result(self, timeout: Optional[float] = None) -> Tuple[np.ndarray, int]:
        parts = [a for a, _, _ in self.chunks(timeout)]
        if not parts:
            return np.zeros(1, dtype=np.float32), self._sr  # model.py:630-632: empty generation -> one zero sample
        return np.concatenate(parts), self._sr

    @property
    def ttfa_s(self) -> Optional[float]:
        return None if self.t_first is None else self.t_first - self.t_submit


@dataclass
class _Active:
    handle: RequestHandle
    slot: int
    window: object
    emitted: int = 0
    budget: int = 0
    chunk_index: int = 0
    open_text: bool = False  # TTSRequest(text_open=True): its text rows are appended before each launch
    text_sent: int = 0       # committed text ids already in the slot (the first one is in the prompt)
    talker: object = None    # text projection of the open text's rows
    waiting: bool = False    # the stream waits for text (status.done = 4)
    gen_step: int = 0


class _StatefulAudio:
    """push(chunk) -> the chunk's samples through the slot's codec.CodecStream (same surface as model.WindowedDecode)."""

    def __init__(self, cstream, sample_rate: int):
        self.cs, self.sr = cstream, sample_rate

    def push(self, chunk: torch.Tensor):
        return self.cs.decode(chunk), self.sr


class BatchScheduler:
    """Continuous batching for one engine (= one GPU).  `tts` must have been loaded with `max_streams` >= the wanted
    concurrency (`FasterQwen3TTS.from_pretrained(..., max_streams=16)`)."""

    def __init__(self, tts, chunk_frames: int = 8, max_concurrent: Optional[int] = None, seed: int = 0, codec_lanes: int = 4,
                 codec_mode: str = "auto", codec_split_k: Optional[bool] = None, overlap_codec="auto",
                 emit_every: int = 1, mixed_policies: bool = False, text_timeout: float = 30.0):
        """codec_mode: "windowed" (default, = "auto") — the reference's 25-frame left-context re-decode (model.py:737-826): the
        audio is bit for bit what the single-stream streaming API returns for the same codes; "stateful" — one
        codec.CodecStream per slot: a chunk costs its own frames and the audio is the full non-streaming decode of the
        utterance's codes (bit for bit with codec_split_k=False, up to fp32 summation order otherwise).
        codec_lanes: CUDA streams the utterances' codec decodes of one chunk are spread over (16 windowed decodes: 23 ms on one
        stream, 11 ms on four, profiles/r02k_codec_lanes_probe.log).
        emit_every: after an utterance's first chunk (time to first audio is not touched) hand audio out every `emit_every`
        chunks: a 41-frame window per 16 new frames instead of two 33-frame windows — less codec work per second of audio, at
        the price of coarser streaming; the audio then differs from the chunk-by-chunk streaming run by the windowed policy's
        own approximation (not at all in stateful mode).
        overlap_codec: where the previous chunk's codec runs relative to the next frame-loop launch.  "host": on the GPU the
        codec lanes run first and the launch waits for them (stream events), on the host the audio is collected and handed out
        while the frame loop runs — no contention on the GPU, nothing idle on the host (16 streams: 202 audio-s/s, stable).
        "gpu": the codec runs WHILE the frame loop runs, on the 20 SMs its grid leaves free — best for one or two utterances
        (a lone request: 44 vs 41 audio-s/s), but with many the two slow each other through L2 and throughput spreads
        134–209 audio-s/s run to run.  "auto" (default): "gpu" for up to two utterances in the chunk, "host" beyond.
        "none": codec, host collection, then launch.
        (The first "gpu" runs exposed a missing dependency in the wide frame program — fixed, DESIGN.md §3.5 "pass 0a -> 0b";
        profiles/r02k_serving_overlap_fault.log, r02k_overlap_stress_after_fix.log.)
        mixed_policies: no cohorts — requests take free slots first come, first served whatever their sampling policy; each
        admitted request's policy and seed (`TTSRequest.seed`, or one derived from `seed` and the request id) become its slot's
        own policy before its prefill, and every launch passes one fixed launch-wide policy that no live stream uses.  Off by
        default: then a request that carries a `seed` is refused (the cohort shares the scheduler's `seed`).
        text_timeout: an open request (TTSRequest(text_open=True)) whose text has not ended and that receives no text for this many
        seconds is cancelled (finish_reason "text_timeout"), so a slow client does not hold a slot for ever."""
        self.tts = tts
        self.emit_every = max(1, int(emit_every))
        self.codec_lanes = max(1, int(codec_lanes))
        self.overlap_codec = {True: "gpu", False: "none"}.get(overlap_codec, overlap_codec)
        if self.overlap_codec not in ("auto", "host", "gpu", "none"):
            raise ValueError(f"overlap_codec {overlap_codec!r}: auto | host | gpu | none")
        causal = getattr(tts.model.model.speech_tokenizer.decoder.cfg, "trans_conv_trim", "") == "right"
        if codec_mode == "auto":
            codec_mode = "windowed"
        if codec_mode not in ("stateful", "windowed") or (codec_mode == "stateful" and not causal):
            raise ValueError(f"codec_mode {codec_mode!r} is not available for this decoder")
        self.codec_mode, self.codec_split_k = codec_mode, codec_split_k
        self._cstreams: Dict[int, object] = {}  # slot -> codec.CodecStream (stateful mode)
        self._draining: set = set()  # slots whose last chunk still waits for the codec: their codec state is not reusable yet
        self.eng = tts.model.engine
        self.chunk_frames = int(chunk_frames)
        cap = self.eng.max_streams
        if self.eng.lockstep_group <= 4:  # 1.7B dims: no wide program, the frame loop takes four streams per launch
            cap = min(cap, 4)
        self.max_concurrent = min(cap, max_concurrent or cap)
        self.seed = seed
        self.mixed_policies = bool(mixed_policies)
        self.text_timeout = float(text_timeout)
        self._pending: "queue.Queue[RequestHandle]" = queue.Queue()
        self._deferred: List[RequestHandle] = []   # waiting for the running cohort's policy to drain
        self._active: Dict[int, _Active] = {}
        self._cohort: Optional[tuple] = None
        self._thread: Optional[threading.Thread] = None
        self._stop = threading.Event()
        self._wake = threading.Event()
        self._next_id = 0
        self._submit_lock = threading.Lock()  # submit() is the one method other threads call
        self._lanes: List[tuple] = []  # (CUDA stream, speech tokenizer with its own launch plans) per codec lane
        self._backlog: List[tuple] = []  # (active, codes chunk, final?, reason) of the chunk that just finished
        self._failure: Optional[BaseException] = None  # what stopped the loop (device fault, ...): submit() refuses from then on
        # seconds per part of the loop: admit (prompt build + prefill), launch (host side of fq3_decode_frames), emit (codec lanes +
        # D2H + hand-out of the previous chunk), wait (blocked on the running launch)
        self.stats = {"launches": 0, "frames": 0, "requests": 0, "max_batch": 0, "t_admit": 0.0, "t_launch": 0.0, "t_emit": 0.0, "t_wait": 0.0}

    # ---- public ----
    def start(self):
        if self._thread is None:
            self._thread = threading.Thread(target=self._run, name="fq3-scheduler", daemon=True)
            self._thread.start()
        return self

    def stop(self, timeout: float = 30.0):
        self._stop.set()
        self._wake.set()
        if self._thread is not None:
            self._thread.join(timeout)
            if self._thread.is_alive():  # still inside a launch: keep the handle, a second start() must not run beside it
                logger.warning("fq3 scheduler thread did not stop within %.0f s", timeout)
                return
            self._thread = None
        self._stop.clear()

    @property
    def healthy(self) -> bool:
        """False once the loop has died of an exception (a device fault is sticky: the engine has to be rebuilt or
        `fq3_clear_fault`-ed): the HTTP front then routes around this replica (server.Dispatcher) and /health says so."""
        return self._failure is None

    def __enter__(self):
        return self.start()

    def __exit__(self, *exc):
        self.stop()

    def submit(self, req: TTSRequest) -> RequestHandle:
        if req.kind not in ("voice_clone", "custom_voice", "voice_design"):
            raise ValueError(f"unknown request kind {req.kind!r}")
        if self._failure is not None:  # nobody would ever answer: say so now instead of letting the caller wait for ever
            raise RuntimeError(f"scheduler stopped after a failure: {self._failure!r}")
        if self.mixed_policies:
            self._policy(req.policy_key(), 0 if req.seed is None else req.seed).validate()
        elif req.seed is not None:
            raise ValueError("a per-request seed needs BatchScheduler(mixed_policies=True): "
                             "in cohort mode the requests of a launch share the scheduler's seed")
        if req.text_open and req.kind == "voice_clone" and not req.xvec_only:
            raise ValueError("open text: an ICL voice clone sums the text into the reference-code rows; use xvec_only=True")
        if req.text_open and req.kind == "voice_clone" and req.non_streaming_mode:
            raise ValueError("open text needs non_streaming_mode=False (the whole text is in the prompt otherwise)")
        with self._submit_lock:
            h = RequestHandle(req, self._next_id)
            self._next_id += 1
        h._sr = self.tts.sample_rate
        h._wake = self._wake
        self._pending.put(h)
        self._wake.set()
        return h

    # ---- scheduler thread ----
    def _prepare(self, r: TTSRequest, text: Optional[str] = None):
        """Prompt embeddings exactly as the matching generate_* method builds them (model.py:202-330); `text`: the text received
        so far of an open request."""
        t = self.tts
        text = r.text if text is None else text
        if r.kind == "voice_clone":
            m, _, _, tie, tam, tth, tpe, ref_codes = t._prepare_generation(
                text, r.ref_audio, r.ref_text, language=r.language, xvec_only=r.xvec_only,
                non_streaming_mode=r.non_streaming_mode, append_silence=r.append_silence, instruct=r.instruct)
            return m, tie, tam, tth, tpe, ref_codes
        if r.kind == "custom_voice":
            t._check_custom(r.language, r.speaker)
            instruct = None if t.model.model.tts_model_size in "0b6" else r.instruct  # model.py:849-850
            m, _, _, tie, tam, tth, tpe = t._prepare_generation_custom(text, r.language, r.speaker, instruct)
        else:
            t._check_design(r.language)
            m, _, _, tie, tam, tth, tpe = t._prepare_generation_custom(text, r.language, None, r.instruct)
        return m, tie, tam, tth, tpe, None

    def _policy(self, key: tuple, seed: Optional[int] = None) -> SamplingPolicy:
        do_sample, top_k, top_p, temperature, rep, min_new = key
        return SamplingPolicy(do_sample=do_sample, top_k=top_k, top_p=top_p, temperature=temperature, repetition_penalty=rep,
                              min_new_tokens=min_new, suppress_tail=1024, seed=self.seed if seed is None else seed)

    def request_seed(self, h: RequestHandle) -> int:
        """Mixed mode: the request's own seed, else one derived from the scheduler's seed and the request id (splitmix64), so
        that it does not depend on the slot the request gets."""
        if h.request.seed is not None:
            return int(h.request.seed)
        x = (int(self.seed) * 0x9E3779B97F4A7C15 + h.id + 1) & 0xFFFFFFFFFFFFFFFF
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        return x ^ (x >> 31)

    def _launch_policy(self) -> SamplingPolicy:
        """The policy argument of a launch: the cohort's, or in mixed mode a fixed one that no live stream uses (every live stream
        has its own)."""
        if self.mixed_policies:
            return SamplingPolicy(do_sample=False, seed=self.seed)
        return self._policy(self._cohort)

    def _release(self, slot: int):
        """Retire a slot; in mixed mode also forget its policy, so that a later user of the engine's slot (slot 0: the
        single-stream API) samples with its own arguments again."""
        self.eng.retire_stream(slot)
        if self.mixed_policies:
            self.eng.set_stream_policy(slot, None)

    def _admit(self):
        """Move waiting requests into free slots (prefill runs here, between two chunk launches)."""
        from .generate import _left_pads
        from .model import WindowedDecode

        waiting = self._deferred
        self._deferred = []
        while True:
            try:
                waiting.append(self._pending.get_nowait())
            except queue.Empty:
                break
        blocked = False  # FIFO: once a request waits for another policy's cohort to drain, nothing behind it overtakes it
        for h in waiting:
            if h.cancelled:
                self._finish(h, "cancelled")
                continue
            if h.request.text_open:  # admitted once its first text token is committed; until then it holds no place in line
                try:
                    timed_out = self._pull_text(h)
                except ValueError as e:  # e.g. the text closed empty
                    h.q.put(e)
                    self._finish(h, "error")
                    continue
                if not h._text_feed.ids:
                    if timed_out:
                        self._finish(h, "text_timeout")
                    else:
                        self._deferred.append(h)
                    continue
            key = h.request.policy_key()
            if self.mixed_policies:
                self._cohort = key  # no cohorts: whatever the policy, the request only waits for a free slot
            elif self._cohort is None and not self._active:
                self._cohort = key
            free = [s for s in range(self.max_concurrent) if s not in self._active and s not in self._draining]
            if blocked or key != self._cohort or not free:
                blocked = blocked or key != self._cohort
                self._deferred.append(h)
                continue
            slot = free[0]
            feed = h._text_feed
            try:
                m, tie, tam, tth, tpe, ref_codes = self._prepare(h.request, None if feed is None else feed.text)
                if tie.shape[1] > self.eng.max_seq_len:
                    raise RuntimeError(  # talker_graph.py:163-167
                        f"Input is too long: prefill has {tie.shape[1]} tokens but max_seq_len={self.eng.max_seq_len}. "
                        "Use shorter text or shorter reference audio.")
                if feed is None:
                    self.eng.set_text_conditioning(slot, tth[0], tpe)
                else:  # the prompt holds the first text token; the rest arrive as trailing rows (text_stream.py)
                    self.eng.open_text(slot, tpe)
                if self.mixed_policies:
                    self.eng.set_stream_policy(slot, self._policy(key, self.request_seed(h)))
                    self.eng.prefill(slot, tie[0], _left_pads(tam), self._launch_policy())
                else:
                    self.eng.prefill(slot, tie[0], _left_pads(tam), self._policy(key))
            except Exception as e:  # a bad request must not take the loop down
                try:
                    self._release(slot)  # whatever the failed prefill left in the slot must not decode
                except Exception:
                    pass
                h.q.put(e)
                self._finish(h, "error")
                continue
            lane_stream, lane_tok = self._lane(slot, m.speech_tokenizer)
            if self.codec_mode == "stateful":
                cs = self._cstreams.get(slot)
                if cs is None:
                    cs = self._cstreams[slot] = lane_tok.decoder.open_stream(max(self.chunk_frames, 8), self.codec_split_k)
                with self._on(lane_stream):  # ordered behind the slot's previous utterance on the same lane
                    cs.reset()
                    if ref_codes is not None:  # ICL: the reference clip's codes are acoustic context, decoded for their state only
                        cs.decode(ref_codes.to(self.eng.device))
                window = _StatefulAudio(cs, lane_tok.sample_rate)
            else:
                window = WindowedDecode(lane_tok, ref_codes, self.chunk_frames)
            a = self._active[slot] = _Active(h, slot, window, budget=min(h.request.max_new_tokens, self.eng.max_frames))
            if feed is not None:
                a.open_text, a.talker, a.text_sent, a.waiting = True, m.talker, 1, True  # prefilled without a second token
                self._append_text(a)
            self.stats["requests"] += 1

    def _pull_text(self, h: RequestHandle) -> bool:
        """Commit the pieces an open request received since the last call (text_stream.TextFeed); returns whether its text
        has been silent for text_timeout seconds without being closed."""
        from .text_stream import TextFeed

        if h._text_feed is None:
            h._text_feed = TextFeed(self.tts.model.tokenizer.assistant, self.tts.model.model.config.tts_eos_token_id)
        pieces, closed, t_text = h._take_text()
        for p in pieces:
            h._text_feed.push(p)
        if closed:
            h._text_feed.close()
        return not closed and time.monotonic() - t_text > self.text_timeout

    def _append_text(self, a: _Active):
        """The committed text of an open slot that is not on the device yet (and the close)."""
        from .text_stream import text_rows

        feed = a.handle._text_feed
        new = feed.ids[a.text_sent:]
        if new:  # a close always commits the tts_eos id, so it travels with rows
            self.eng.append_text(a.slot, text_rows(a.talker, new), close=feed.closed)
            a.text_sent = len(feed.ids)
        rows = a.text_sent - 1  # trailing rows: the first committed token is in the prompt
        a.waiting = a.waiting and not (feed.closed or rows > a.gen_step)

    def _service_open(self):
        """Before a launch: append what every open slot received; cancel a cancelled or silent one (its slot is free again)."""
        for slot in sorted(self._active):
            a = self._active[slot]
            if not a.open_text:
                continue
            reason = "cancelled" if a.handle.cancelled else None
            if reason is None:
                try:
                    timed_out = self._pull_text(a.handle)
                except ValueError as e:
                    a.handle.q.put(e)
                    timed_out, reason = False, "error"
                if timed_out:
                    reason = "text_timeout"
                elif reason is None:
                    self._append_text(a)
            if reason is not None:
                self._finish(a.handle, reason)
                self._release(slot)
                del self._active[slot]

    def _finish(self, h: RequestHandle, reason: str):
        h.finish_reason = reason
        h.t_done = time.time()
        h.q.put(_DONE)

    @staticmethod
    def _on(stream):
        """Context of a codec lane's CUDA stream (a no-op for the host-only doubles of tests/test_serving_cpu.py)."""
        import contextlib

        return torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()

    def _lane(self, slot: int, tok):
        """Codec lane of a slot.  A windowed decode of one utterance is a chain of ~150 small launches (1.4 ms, latency-bound),
        so the utterances of a chunk are spread over a few CUDA streams, each with its own copy of the decoder's launch plans
        (the packed weights are shared); together they fill the SMs the frame loop leaves free."""
        import copy

        from .codec import SpeechTokenizer

        if not self._lanes:
            # the lanes (and the launch plans / CUDA graphs they have built) belong to the model, not to one scheduler object
            cache = self.tts.__dict__.setdefault("_serving_lanes", {})
            self._lanes = cache.setdefault(self.codec_lanes, [])
        if not self._lanes:
            for i in range(self.codec_lanes):
                dec = copy.copy(tok.decoder)
                dec._plans = {}
                stream = torch.cuda.Stream(device=self.eng.device) if torch.device(self.eng.device).type == "cuda" else None
                self._lanes.append((stream, SpeechTokenizer(dec)))
        return self._lanes[slot % len(self._lanes)]

    def _emit_enqueue(self, work: List[tuple]) -> list:
        """Enqueue the codec decode of one chunk's codes on the codec lanes (asynchronous)."""
        staged = []
        for a, chunk, final, reason in work:
            stream = self._lanes[a.slot % len(self._lanes)][0]
            # pinned staging: a copy from pageable memory first synchronises the lane's stream, i.e. waits for the decode of the
            # utterance enqueued on that lane just before
            src = chunk.pin_memory() if stream is not None else chunk
            with self._on(stream):
                audio, sr = a.window.push(src.to(self.eng.device, non_blocking=True))
            staged.append((stream, audio, sr))
        return staged

    def _emit_collect(self, work: List[tuple], staged: list):
        """Audio to the host and out to each request's queue."""
        for (a, chunk, final, reason), (stream, audio, sr) in zip(work, staged):
            with self._on(stream):
                wav = self.tts._to_numpy(audio)  # D2H on the lane's stream, synchronises it
            h = a.handle
            if h.t_first is None:
                h.t_first = time.time()
            h.codes.append(chunk)
            info = {"chunk_index": a.chunk_index, "chunk_steps": int(chunk.shape[0]), "total_steps_so_far": a.emitted,
                    "is_final": final, "slot": a.slot}
            a.chunk_index += 1
            h.q.put((wav, sr, info))
            if final:
                self._draining.discard(a.slot)
                self._finish(h, reason)

    def _emit(self, work: List[tuple]):
        if work:
            self._emit_collect(work, self._emit_enqueue(work))

    def _lanes_before_main(self):
        """Make the engine's stream wait for everything enqueued on the codec lanes: the next frame-loop launch then starts when
        the codec is done (no contention on the GPU) while the host is already free to collect the audio."""
        if torch.device(self.eng.device).type != "cuda":
            return
        main = torch.cuda.current_stream(self.eng.device)
        for stream, _ in self._lanes:
            if stream is not None:
                ev = torch.cuda.Event()
                ev.record(stream)
                main.wait_event(ev)

    def _run(self):
        eng = self.eng
        try:
            if torch.device(eng.device).type == "cuda":
                torch.cuda.set_device(eng.device)
            with torch.inference_mode():
                for s in range(self.eng.max_streams):
                    self._release(s)  # never-used slots idle inside a launch
                self._backlog = []
                while not self._stop.is_set():
                    t0 = time.perf_counter()
                    self._admit()
                    self._service_open()
                    t1 = time.perf_counter()
                    self.stats["t_admit"] += t1 - t0
                    if self._active and all(a.waiting for a in self._active.values()):
                        self._emit(self._backlog)  # every running stream waits for text: no launch until some arrives
                        self._backlog = []
                        self._wake.wait(timeout=0.05)
                        self._wake.clear()
                        continue
                    if not self._active:
                        self._emit(self._backlog)
                        self._backlog = []
                        self._cohort = None
                        if self._deferred:
                            continue
                        self._wake.wait(timeout=0.05)
                        self._wake.clear()
                        continue
                    staged = None
                    mode = self.overlap_codec
                    if mode == "auto":
                        mode = "gpu" if len(self._backlog) <= 2 else "host"
                    if mode == "none":  # codec of the previous chunk before the next launch, host waits for it
                        self._emit(self._backlog)
                        self._backlog = []
                    elif mode == "host" and self._backlog:  # GPU: codec, then frame loop; host: collects beside the frame loop
                        staged = self._emit_enqueue(self._backlog)
                        tq = time.perf_counter()
                        self._lanes_before_main()
                        self.stats["t_enqueue"] = self.stats.get("t_enqueue", 0.0) + tq - t1
                        self.stats["t_fence"] = self.stats.get("t_fence", 0.0) + time.perf_counter() - tq
                    hi = max(self._active) + 1
                    eng.decode_frames(hi, self.chunk_frames, self._launch_policy(), self.tts.predictor_graph.policy())
                    t2 = time.perf_counter()
                    self.stats["launches"] += 1
                    self.stats["max_batch"] = max(self.stats["max_batch"], len(self._active))
                    if staged is not None:
                        self._emit_collect(self._backlog, staged)
                    else:
                        self._emit(self._backlog)  # "gpu": previous chunk's codec on the SMs the running launch leaves free
                    self._backlog = []
                    t3 = time.perf_counter()
                    self.stats["t_launch"] += t2 - t1
                    self.stats["t_emit"] += t3 - t2
                    for slot in sorted(self._active):
                        a = self._active[slot]
                        st = eng.status(slot)  # synchronises the launch (first call) and reads the slot's counters
                        if st.error:
                            raise RuntimeError(f"device fault {st.error} in slot {slot}")
                        if a.open_text:
                            a.waiting, a.gen_step = st.done == 4, st.gen_step
                        n_new = min(st.n_frames, a.budget) - a.emitted
                        reason = None
                        if a.handle.cancelled:
                            reason = "cancelled"
                        elif st.done == 1:
                            reason = "stop"          # EOS (generate.py:150)
                        elif st.done == 2:
                            reason = "cache_full"    # generate.py:175-177
                        elif st.n_frames >= a.budget:
                            reason = "length"
                        if n_new > 0 and reason is None and a.emitted > 0 and n_new < self.emit_every * self.chunk_frames:
                            # emit_every > 1: after an utterance's first chunk, hand audio out every few chunks
                            continue
                        if reason is None:  # whole chunks only (a stream that waited for text ran part of one)
                            n_new -= n_new % self.chunk_frames
                        if n_new > 0 and reason != "cancelled":
                            chunk = eng.read_codes(slot, a.emitted, n_new)
                            a.emitted += n_new
                            self.stats["frames"] += n_new
                            self._backlog.append((a, chunk, reason is not None, reason))
                            if reason is not None:
                                self._draining.add(slot)
                        elif reason is not None:
                            self._finish(a.handle, reason)
                        if reason is not None:
                            self._release(slot)
                            del self._active[slot]
                    self.stats["t_wait"] += time.perf_counter() - t3
                self._emit(self._backlog)
                for a in list(self._active.values()):  # stop() in mid-utterance: nobody may wait for ever
                    if a.handle.finish_reason is None:
                        self._finish(a.handle, "shutdown")
                    self._release(a.slot)
                self._active.clear()
                leftover = list(self._deferred)
                self._deferred = []
                while True:
                    try:
                        leftover.append(self._pending.get_nowait())
                    except queue.Empty:
                        break
                for h in leftover:
                    self._finish(h, "shutdown")
                for cs in self._cstreams.values():
                    cs.close()
                self._cstreams.clear()

        except BaseException as e:  # surface a scheduler failure to every waiter instead of hanging them
            logger.exception("fq3 scheduler stopped")
            self._failure = e
            waiters = {id(a.handle): a.handle for a in self._active.values()}
            for a, _chunk, _final, _reason in self._backlog:  # a retired slot's last chunk was still waiting for the codec
                if a.handle.finish_reason is None:
                    waiters.setdefault(id(a.handle), a.handle)
            self._active.clear()
            self._backlog = []
            for h in waiters.values():
                h.finish_reason = "error"
                h.q.put(e)
                h.q.put(_DONE)
            for h in self._deferred:
                h.finish_reason = "error"
                h.q.put(e)
                h.q.put(_DONE)
            self._deferred = []
            while True:
                try:
                    h = self._pending.get_nowait()
                except queue.Empty:
                    break
                h.finish_reason = "error"
                h.q.put(e)
                h.q.put(_DONE)
