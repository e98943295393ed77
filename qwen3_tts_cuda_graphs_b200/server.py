"""HTTP front of the serving layer (SURVEY.md §8 row f4): the reference's OpenAI-compatible endpoint
(`examples/openai_server.py:219-265`: POST /v1/audio/speech, GET /health; wav / pcm streamed chunk by chunk with an
unknown-length WAV header) and the demo's server-sent-events protocol (`demo/server.py:332-541`: POST /generate/stream ->
`data: {"type": "queued" | "chunk" | "done" | "error", ...}`; POST /generate -> one base64 WAV + metrics, `:546-662`; GET /status;
reference audio as an upload, a preset or a configured voice; the demo's text / upload size limits), on top of
`serving.BatchScheduler` instead of a global lock:
concurrent requests decode in lock-step on the same weight sweep, one scheduler per GPU, requests go to the least-loaded one
(replicas only — DESIGN.md §7).

    python -m qwen3_tts_cuda_graphs_b200.server --model <dir | synthetic://0.6B-Base> --ref-audio voice.wav --ref-text "..." \
        [--voices voices.json] [--gpus 8] [--max-concurrent 16] [--port 8000]

Text that is still arriving (an LLM's reply) goes through the WebSocket `/v1/audio/speech/stream`: a JSON `{voice, seed?,
response_format: "pcm"}`, then `{"text": ...}` messages and `{"close": true}`; PCM16 chunks come back as they are decoded, then
`{"event": "done", "finish_reason", "frames"}`.

`create_app(backends, voices, default_voice)` takes anything with the scheduler's `submit(TTSRequest) -> handle` surface, so the
HTTP layer is tested on CPU with a stand-in backend (`tests/test_server_cpu.py`).
"""
from __future__ import annotations

import argparse
import asyncio
import base64
import hashlib
import io
import json
import logging
import os
import struct
import sys
import tempfile
import threading
import time
from typing import Dict, List, Optional

import numpy as np
from fastapi import FastAPI, File, Form, HTTPException, UploadFile, WebSocket, WebSocketDisconnect  # module level: the endpoints' annotations are resolved by name
from fastapi.responses import JSONResponse, Response, StreamingResponse
from pydantic import BaseModel
from starlette.background import BackgroundTask

from .serving import TTSRequest

logger = logging.getLogger(__name__)

CONTENT_TYPES = {"wav": "audio/wav", "pcm": "audio/pcm", "mp3": "audio/mpeg"}
MAX_TEXT_CHARS = 1000                 # demo/server.py:173
MAX_AUDIO_BYTES = 10 * 1024 * 1024    # demo/server.py:175 (about one minute of 44.1 kHz stereo 16-bit WAV)
AUDIO_TOO_LARGE = ("Audio file too large ({size_mb:.1f} MB). Voice cloning works best with short clips under 1 minute — "
                   "please upload a shorter recording.")
_ref_paths: Dict[str, str] = {}
_ref_paths_lock = threading.Lock()


def cached_ref_path(content: bytes) -> str:
    """An uploaded reference clip -> a file named after its content hash (demo/server.py:201-212), so the same clip uploaded again
    is the same `ref_audio` path and hits the model's voice-prompt cache (x-vector / reference codes are encoded once per voice)."""
    digest = hashlib.sha1(content).hexdigest()
    with _ref_paths_lock:
        path = _ref_paths.get(digest)
        if path and os.path.exists(path):
            return path
        path = os.path.join(tempfile.gettempdir(), f"fq3_tts_ref_{digest}.wav")
        if not os.path.exists(path):
            with open(path, "wb") as f:
                f.write(content)
        _ref_paths[digest] = path
        return path


# ---- audio helpers (examples/openai_server.py:88-118) ------------------------------------------
def to_pcm16(pcm: np.ndarray) -> bytes:
    return np.clip(np.asarray(pcm, dtype=np.float32) * 32768.0, -32768, 32767).astype("<i2").tobytes()


def wav_header(sample_rate: int, data_len: int = 0xFFFFFFFF) -> bytes:
    """16-bit mono WAV header; data_len 0xFFFFFFFF = streamed, length unknown."""
    riff = 0xFFFFFFFF if data_len == 0xFFFFFFFF else 36 + data_len
    return (b"RIFF" + struct.pack("<I", riff) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, 1, 1, sample_rate, sample_rate * 2, 2, 16)
            + b"data" + struct.pack("<I", data_len))


def to_wav_bytes(pcm: np.ndarray, sample_rate: int) -> bytes:
    raw = to_pcm16(pcm)
    return wav_header(sample_rate, len(raw)) + raw


def mp3_encoder():
    """pydub's AudioSegment (needs ffmpeg) or the reference's 400 (examples/openai_server.py:121-130).  Asked for BEFORE the utterance
    is generated, so a server without pydub refuses at once instead of after the decode."""
    try:
        from pydub import AudioSegment
    except ImportError:
        raise HTTPException(status_code=400, detail="response_format='mp3' requires pydub: pip install pydub")
    return AudioSegment


def to_mp3_bytes(pcm: np.ndarray, sample_rate: int, segment_cls=None) -> bytes:
    segment = (segment_cls or mp3_encoder())(to_pcm16(pcm), frame_rate=sample_rate, sample_width=2, channels=1)
    buf = io.BytesIO()
    segment.export(buf, format="mp3")
    return buf.getvalue()


class SpeechRequest(BaseModel):  # examples/openai_server.py:78-83
    model: str = "tts-1"
    input: str
    voice: str = "alloy"
    response_format: str = "wav"
    speed: float = 1.0  # accepted, not applied (as in the reference)
    seed: Optional[int] = None  # sampling seed: the same seed gives the same audio (a server started with --mixed-policies)


class BackendUnavailable(RuntimeError):
    """Every replica's scheduler has stopped (HTTP 503)."""


class Dispatcher:
    """Least-loaded choice among per-GPU backends (request-parallel replicas; no exchange between them)."""

    def __init__(self, backends: List[object]):
        if not backends:
            raise ValueError("no backend")
        self.backends = list(backends)
        self.in_flight = [0] * len(self.backends)
        self._lock = threading.Lock()

    def healthy(self) -> List[bool]:
        return [bool(getattr(b, "healthy", True)) for b in self.backends]

    def submit(self, req: TTSRequest):
        with self._lock:
            live = [j for j, ok in enumerate(self.healthy()) if ok]  # a replica whose loop died (device fault) is routed around
            if not live:
                raise BackendUnavailable("no healthy backend: every replica's scheduler has stopped")
            i = min(live, key=lambda j: self.in_flight[j])
            self.in_flight[i] += 1
        try:
            h = self.backends[i].submit(req)
        except Exception:
            self.release(i)
            raise
        h._backend_index = i
        return h

    def release(self, i: int):
        with self._lock:
            self.in_flight[i] = max(0, self.in_flight[i] - 1)


def _request_for(voice_cfg: dict, text: str, overrides: Optional[dict] = None) -> TTSRequest:
    """A voices.json entry -> request.  Entries: {"ref_audio", "ref_text", "language"} (voice clone, as in the reference),
    {"speaker", "language", "instruct"} (custom voice) or {"instruct", "language"} (voice design)."""
    kw = dict(text=text, language=voice_cfg.get("language", "Auto"))
    if voice_cfg.get("speaker"):
        kw.update(kind="custom_voice", speaker=voice_cfg["speaker"], instruct=voice_cfg.get("instruct") or None)
    elif voice_cfg.get("ref_audio"):
        kw.update(kind="voice_clone", ref_audio=voice_cfg["ref_audio"], ref_text=voice_cfg.get("ref_text", ""),
                  xvec_only=bool(voice_cfg.get("xvec_only", True)), non_streaming_mode=False)
    elif voice_cfg.get("instruct"):
        kw.update(kind="voice_design", instruct=voice_cfg["instruct"])
    else:
        raise ValueError("a voice needs ref_audio, speaker or instruct")
    for k in ("max_new_tokens", "temperature", "top_k", "top_p", "repetition_penalty", "do_sample", "seed"):
        if k in voice_cfg:
            kw[k] = voice_cfg[k]
    kw.update({k: v for k, v in (overrides or {}).items() if not (k == "seed" and v is None)})
    req = TTSRequest(**kw)
    _check_sampling(req)
    return req


def _check_sampling(req: TTSRequest):
    """ValueError (HTTP 400) for sampling fields out of range (engine.SamplingPolicy.validate)."""
    from .engine import SamplingPolicy

    if req.seed is not None and (isinstance(req.seed, bool) or not isinstance(req.seed, int)):
        raise ValueError(f"seed must be an integer, got {req.seed!r}")
    SamplingPolicy(do_sample=req.do_sample, top_k=req.top_k, top_p=req.top_p, temperature=req.temperature,
                   repetition_penalty=req.repetition_penalty, min_new_tokens=req.min_new_tokens,
                   seed=0 if req.seed is None else req.seed).validate()


def create_app(backends: List[object], voices: Dict[str, dict], default_voice: Optional[str] = None, sample_rate: int = 24000,
               model_name: Optional[str] = None):
    app = FastAPI(title="qwen3-tts B200 engine: OpenAI-compatible API")
    disp = Dispatcher(backends)
    app.state.dispatcher = disp

    def resolve_voice(name: str) -> dict:  # examples/openai_server.py:146-165
        if name in voices:
            return voices[name]
        if default_voice and default_voice in voices:
            logger.warning("Voice %r not configured; falling back to default voice %r", name, default_voice)
            return voices[default_voice]
        raise HTTPException(status_code=400, detail=f"Voice {name!r} is not configured. Available voices: {list(voices.keys())}")

    def settle(handle):
        """Once per request, whichever comes first — the end of its stream, or the end of the response (a client that went away
        before the first byte never starts the stream): cancel what is still decoding (the slot is freed at the next chunk
        boundary) and give the replica's in-flight count back."""
        if getattr(handle, "_settled", False):
            return
        handle._settled = True
        if getattr(handle, "finish_reason", None) is None and hasattr(handle, "cancel"):
            handle.cancel()
        disp.release(getattr(handle, "_backend_index", 0))

    async def chunks_of(handle):
        """Pull a handle's chunks without blocking the event loop."""
        loop = asyncio.get_event_loop()
        it = iter(handle)
        try:
            while True:
                item = await loop.run_in_executor(None, lambda: next(it, None))
                if item is None:
                    return
                yield item
        finally:
            settle(handle)

    @app.get("/health")
    async def health():
        ok = disp.healthy()
        status = "ok" if all(ok) else ("degraded" if any(ok) else "down")
        return {"status": status, "model_loaded": True, "backends": len(disp.backends), "healthy": ok, "in_flight": list(disp.in_flight)}

    @app.get("/v1/voices")
    async def list_voices():
        return {"voices": sorted(voices), "default": default_voice}

    @app.post("/v1/audio/speech")
    async def create_speech(req: SpeechRequest):
        if not req.input.strip():
            raise HTTPException(status_code=400, detail="'input' text is empty")
        voice_cfg = resolve_voice(req.voice)
        fmt = req.response_format.lower()
        if fmt not in CONTENT_TYPES:
            raise HTTPException(status_code=400, detail=f"response_format {fmt!r} not supported. Use: wav, pcm, mp3")
        segment_cls = mp3_encoder() if fmt == "mp3" else None
        try:
            handle = disp.submit(_request_for(voice_cfg, req.input, {"seed": req.seed}))
        except ValueError as e:
            raise HTTPException(status_code=400, detail=str(e))
        except RuntimeError as e:  # BackendUnavailable, or the chosen replica failed between the check and the submit
            raise HTTPException(status_code=503, detail=str(e))

        if fmt == "mp3":  # the whole utterance, then one encode (examples/openai_server.py:242-259)
            parts, sr = [], sample_rate
            try:
                async for audio, sr, _info in chunks_of(handle):
                    parts.append(audio)
            except Exception as e:
                raise HTTPException(status_code=500, detail=str(e))
            audio = np.concatenate(parts) if parts else np.zeros(1, dtype=np.float32)
            return Response(content=to_mp3_bytes(audio, sr, segment_cls), media_type=CONTENT_TYPES[fmt])

        async def audio_stream():
            if fmt == "wav":
                yield wav_header(sample_rate)
            async for audio, _sr, _info in chunks_of(handle):
                yield to_pcm16(audio)

        return StreamingResponse(audio_stream(), media_type=CONTENT_TYPES[fmt], background=BackgroundTask(settle, handle))

    async def demo_request(text, language, mode, ref_text, speaker, instruct, xvec_only, temperature, top_k, repetition_penalty,
                           voice, ref_preset, ref_audio, seed=None) -> TTSRequest:
        """The demo's form (demo/server.py:332-372, :546-587) -> a request.  Reference audio: an upload, else a configured voice
        (`ref_preset` / `voice`, the demo's presets), else the default voice."""
        if not text.strip():
            raise HTTPException(status_code=400, detail="text is empty")
        if len(text) > MAX_TEXT_CHARS:
            raise HTTPException(status_code=400, detail=f"Text too long ({len(text)} chars). Maximum is {MAX_TEXT_CHARS} characters.")
        over = dict(language=language, temperature=temperature, top_k=top_k, repetition_penalty=repetition_penalty, seed=seed)
        try:
            if mode == "voice_clone":
                if ref_audio is not None and getattr(ref_audio, "filename", None):
                    content = await ref_audio.read()
                    if len(content) > MAX_AUDIO_BYTES:
                        raise HTTPException(status_code=400, detail=AUDIO_TOO_LARGE.format(size_mb=len(content) / 1024 / 1024))
                    cfg = {"ref_audio": cached_ref_path(content), "ref_text": ref_text}
                else:
                    cfg = dict(resolve_voice(ref_preset or voice or (default_voice or "")))
                    if ref_text:
                        cfg["ref_text"] = ref_text
                cfg["xvec_only"] = xvec_only
                return _request_for(cfg, text, over)
            if mode == "custom":
                return _request_for({"speaker": speaker, "instruct": instruct}, text, over)
            if mode == "voice_design":
                return _request_for({"instruct": instruct}, text, over)
            raise ValueError(f"unknown mode {mode!r}")
        except ValueError as e:
            raise HTTPException(status_code=400, detail=str(e))

    def submit_or_503(req: TTSRequest):
        try:
            return disp.submit(req)
        except ValueError as e:  # e.g. a seed sent to a server without --mixed-policies
            raise HTTPException(status_code=400, detail=str(e))
        except RuntimeError as e:
            raise HTTPException(status_code=503, detail=str(e))

    @app.get("/status")
    async def status():
        """demo/server.py:251-277, for the model(s) this server was started with (no load / unload at run time)."""
        tts = getattr(disp.backends[0], "tts", None)
        model_type, speakers, name = None, [], model_name
        if tts is not None:
            try:
                model_type = tts.model.model.tts_model_type
                speakers = list(tts.model.get_supported_speakers() or [])
            except Exception:
                speakers = []
        return {"loaded": True, "model": name, "loading": False, "model_type": model_type, "speakers": speakers,
                "transcription_available": False,
                "preset_refs": [{"id": k, "label": k, "ref_text": v.get("ref_text", "")} for k, v in voices.items() if v.get("ref_audio")],
                "queue_depth": sum(disp.in_flight), "backends": len(disp.backends), "healthy": disp.healthy()}

    @app.get("/preset_ref/{preset_id}")
    async def preset_ref(preset_id: str):
        """demo/server.py:279-290: a configured voice's reference clip, for the page's player."""
        cfg = voices.get(preset_id)
        if not cfg or not cfg.get("ref_audio"):
            raise HTTPException(status_code=404, detail="Preset not found")
        try:
            with open(cfg["ref_audio"], "rb") as f:
                audio_b64 = base64.b64encode(f.read()).decode()
        except OSError:
            raise HTTPException(status_code=404, detail="Preset audio not found")
        return {"id": preset_id, "label": preset_id, "filename": os.path.basename(str(cfg["ref_audio"])),
                "ref_text": cfg.get("ref_text", ""), "audio_b64": audio_b64}

    @app.post("/load")
    async def load_model(model_id: str = Form(...)):
        """demo/server.py:293-329 switches models at run time; here the replicas are built once at start-up (weights packed into
        per-GPU arenas, launch plans warmed), so asking for the served model succeeds and anything else says how to get it."""
        if model_name is None or model_id == model_name:
            return {"status": "already_loaded", "model": model_name or model_id}
        raise HTTPException(status_code=400, detail=f"This server serves {model_name!r}; restart it with --model {model_id} to switch.")

    @app.post("/transcribe")
    async def transcribe_audio(audio: UploadFile = File(...)):
        """demo/server.py:225-248 needs the optional nano-parakeet model; without it the reference answers 503 too."""
        raise HTTPException(status_code=503, detail="Transcription model not loaded")

    @app.post("/generate/stream")
    async def generate_stream(text: str = Form(...), language: str = Form("English"), mode: str = Form("voice_clone"),
                              ref_text: str = Form(""), speaker: str = Form(""), instruct: str = Form(""),
                              xvec_only: bool = Form(True), chunk_size: int = Form(8), temperature: float = Form(0.9),
                              top_k: int = Form(50), repetition_penalty: float = Form(1.05), voice: str = Form(""),
                              ref_preset: str = Form(""), ref_audio: UploadFile = File(None), seed: Optional[int] = Form(None)):
        """The demo's SSE protocol (demo/server.py:332-541).  `chunk_size` is accepted for compatibility: the streaming granularity
        is the scheduler's `chunk_frames` (one launch for all running utterances), set when the server starts."""
        req = await demo_request(text, language, mode, ref_text, speaker, instruct, xvec_only, temperature, top_k, repetition_penalty,
                                 voice, ref_preset, ref_audio, seed)
        ahead = sum(disp.in_flight)
        handle = submit_or_503(req)
        t0 = time.perf_counter()

        async def sse():
            if ahead > 0:  # demo/server.py:513-514: only said when somebody is ahead
                yield f"data: {json.dumps({'type': 'queued', 'position': ahead})}\n\n"
            total_audio_s, ttfa_ms = 0.0, None
            try:
                async for audio, sr, _info in chunks_of(handle):
                    now_ms = (time.perf_counter() - t0) * 1000
                    ttfa_ms = now_ms if ttfa_ms is None else ttfa_ms
                    total_audio_s += len(audio) / sr
                    payload = {"type": "chunk", "audio_b64": base64.b64encode(to_wav_bytes(audio, sr)).decode(), "sample_rate": sr,
                               "ttfa_ms": round(ttfa_ms), "rtf": round(total_audio_s / (now_ms / 1000), 3) if now_ms > 0 else 0.0,
                               "total_audio_s": round(total_audio_s, 3), "elapsed_ms": round(now_ms)}
                    yield f"data: {json.dumps(payload)}\n\n"
                total_ms = (time.perf_counter() - t0) * 1000
                done = {"type": "done", "ttfa_ms": round(ttfa_ms or 0), "total_audio_s": round(total_audio_s, 3),
                        "rtf": round(total_audio_s / (total_ms / 1000), 3) if total_ms > 0 else 0.0, "total_ms": round(total_ms)}
                yield f"data: {json.dumps(done)}\n\n"
            except Exception as e:  # generation errors travel in-band, like the demo's
                yield f"data: {json.dumps({'type': 'error', 'message': str(e)})}\n\n"

        return StreamingResponse(sse(), media_type="text/event-stream", headers={"Cache-Control": "no-cache", "X-Accel-Buffering": "no"},
                                 background=BackgroundTask(settle, handle))

    @app.websocket("/v1/audio/speech/stream")
    async def speech_stream(ws: WebSocket):
        """Text that is still arriving (an LLM's reply) in, PCM16 out.  First message: JSON {"voice", "seed"?, "response_format":
        "pcm"}; then any number of {"text": "..."} and one {"close": true}.  The server answers with binary PCM16 chunks as they
        are decoded and a final {"event": "done", "finish_reason", "frames"}; bad input gets {"event": "error", "detail"} and close
        code 1008.  MAX_TEXT_CHARS bounds the whole text.  A disconnect cancels the request (serving.TTSRequest(text_open=True))."""
        await ws.accept()
        handle, sender = None, None

        async def refuse(detail: str, code: int = 1008):
            await ws.send_json({"event": "error", "detail": detail})
            await ws.close(code=code)

        try:
            first = await ws.receive_json()
            if not isinstance(first, dict) or "voice" not in first:
                return await refuse('the first message must be a JSON object {"voice": ..., "response_format": "pcm"}')
            if str(first.get("response_format", "pcm")).lower() != "pcm":
                return await refuse("response_format must be 'pcm' on this endpoint")
            try:
                voice_cfg = resolve_voice(str(first["voice"]))
                handle = disp.submit(_request_for(voice_cfg, "", {"seed": first.get("seed"), "text_open": True}))
            except HTTPException as e:
                return await refuse(str(e.detail))
            except ValueError as e:
                return await refuse(str(e))
            except RuntimeError as e:  # no healthy backend
                return await refuse(str(e), 1011)

            async def pump():
                frames = 0
                try:
                    async for audio, _sr, info in chunks_of(handle):
                        frames += int(info.get("chunk_steps", 0))
                        await ws.send_bytes(to_pcm16(audio))
                except ValueError as e:  # e.g. the text closed empty
                    return await refuse(str(e))
                except Exception as e:
                    return await refuse(str(e), 1011)
                await ws.send_json({"event": "done", "finish_reason": handle.finish_reason, "frames": frames})
                await ws.close()

            sender = asyncio.ensure_future(pump())
            total = 0
            while True:
                recv = asyncio.ensure_future(ws.receive_json())
                done, _ = await asyncio.wait({recv, sender}, return_when=asyncio.FIRST_COMPLETED)
                if recv not in done:  # the request ended first (length cap, error): nothing more to read
                    recv.cancel()
                    return
                msg = recv.result()
                if isinstance(msg, dict) and "text" in msg and isinstance(msg["text"], str):
                    total += len(msg["text"])
                    if total > MAX_TEXT_CHARS:
                        return await refuse(f"Text too long ({total} chars). Maximum is {MAX_TEXT_CHARS} characters.")
                    handle.push_text(msg["text"])
                elif isinstance(msg, dict) and msg.get("close") is True:
                    handle.close_text()
                    break
                else:
                    return await refuse('expected {"text": "..."} or {"close": true}')
            await sender
        except WebSocketDisconnect:
            pass
        except ValueError:  # not JSON
            await refuse("messages must be JSON")
        finally:  # a disconnect or a refusal cancels what is still decoding
            if sender is not None and not sender.done():
                sender.cancel()
            if handle is not None:
                settle(handle)

    @app.post("/generate")
    async def generate_non_streaming(text: str = Form(...), language: str = Form("English"), mode: str = Form("voice_clone"),
                                     ref_text: str = Form(""), speaker: str = Form(""), instruct: str = Form(""),
                                     xvec_only: bool = Form(True), temperature: float = Form(0.9), top_k: int = Form(50),
                                     repetition_penalty: float = Form(1.05), voice: str = Form(""), ref_preset: str = Form(""),
                                     ref_audio: UploadFile = File(None), seed: Optional[int] = Form(None)):
        """The demo's one-shot endpoint (demo/server.py:546-662): the whole utterance as one base64 WAV plus metrics."""
        req = await demo_request(text, language, mode, ref_text, speaker, instruct, xvec_only, temperature, top_k, repetition_penalty,
                                 voice, ref_preset, ref_audio, seed)
        handle = submit_or_503(req)
        t0 = time.perf_counter()
        parts, sr = [], sample_rate
        try:
            async for audio, sr, _info in chunks_of(handle):
                parts.append(audio)
        except HTTPException:
            raise
        except Exception as e:
            raise HTTPException(status_code=500, detail=str(e))
        elapsed = time.perf_counter() - t0
        audio = np.concatenate(parts) if parts else np.zeros(1, dtype=np.float32)
        dur = len(audio) / sr
        return JSONResponse({"audio_b64": base64.b64encode(to_wav_bytes(audio, sr)).decode(), "sample_rate": sr,
                             "metrics": {"total_ms": round(elapsed * 1000), "audio_duration_s": round(dur, 3),
                                         "rtf": round(dur / elapsed, 3) if elapsed > 0 else 0.0}})

    return app


# ---- entry point (examples/openai_server.py:273-356) -------------------------------------------
def load_voices(args) -> (Dict[str, dict], str):
    if args.voices:
        with open(args.voices) as f:
            voices = json.load(f)
        return voices, next(iter(voices))
    if args.ref_audio:
        return {"default": {"ref_audio": args.ref_audio, "ref_text": args.ref_text, "language": args.language}}, "default"
    if args.speaker:
        return {"default": {"speaker": args.speaker, "language": args.language}}, "default"
    print("ERROR: provide --ref-audio <file>, --speaker <id> or --voices <config.json>", file=sys.stderr)
    sys.exit(1)


def replica_devices(gpus: int, device: str = "cuda") -> List[str]:
    """--gpus N -> cuda:0 .. cuda:N-1; one replica may be placed with the reference's --device flag ("cuda" = cuda:0, "cuda:3")."""
    if gpus <= 1:
        return [device if ":" in device else "cuda:0"]
    return [f"cuda:{g}" for g in range(gpus)]


def build_backends(model: str, gpus: int, max_concurrent: int, chunk_frames: int, max_seq_len: int = 2048, device: str = "cuda",
                   mixed_policies: bool = False):
    """One model replica + scheduler per GPU.  mixed_policies: requests of different sampling policies share launches, and a
    request's `seed` is honoured (serving.BatchScheduler)."""
    import torch

    from .model import FasterQwen3TTS
    from .serving import BatchScheduler

    out = []
    for dev in replica_devices(gpus, device):
        tts = FasterQwen3TTS.from_pretrained(model, device=dev, dtype=torch.bfloat16, max_seq_len=max_seq_len,
                                             max_streams=max_concurrent)
        out.append(BatchScheduler(tts, chunk_frames=chunk_frames, max_concurrent=max_concurrent, mixed_policies=mixed_policies).start())
    return out


def warm_up(backends: List[object], voices: Dict[str, dict], rounds: int = 2, frames: int = 40) -> float:
    """Run a short utterance of every configured voice through every replica before the port opens (the reference's servers call
    `_warmup` for the same reason: `demo/server.py:317,688`): the voice prompts are encoded and cached, the dense-prefill graph, the
    codec lanes' launch plans and their CUDA graphs are built — all of which would otherwise land in the first requests' latency.
    Returns the seconds it took."""
    t0 = time.perf_counter()
    for _ in range(rounds):  # a plan becomes a CUDA graph on its second use
        handles = []
        for b in backends:
            for cfg in voices.values():
                handles.append(b.submit(_request_for(cfg, "Warm up.", {"max_new_tokens": frames, "min_new_tokens": min(frames, 2)})))
        for h in handles:
            try:
                h.result()
            except Exception as e:  # a broken voice must not keep the server from starting; it will fail per request
                logger.warning("warm-up of a voice failed: %s", e)
    return time.perf_counter() - t0


def main(argv=None):
    p = argparse.ArgumentParser(description="OpenAI-compatible TTS server on the fq3 engine", formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--model", default=os.environ.get("QWEN_TTS_MODEL", "synthetic://0.6B-Base"), help="checkpoint directory, cached hub id, or synthetic://<preset>")
    p.add_argument("--voices", default=os.environ.get("QWEN_TTS_VOICES"), metavar="FILE")
    p.add_argument("--ref-audio", default=os.environ.get("QWEN_TTS_REF_AUDIO"), metavar="FILE")
    p.add_argument("--ref-text", default=os.environ.get("QWEN_TTS_REF_TEXT", ""))
    p.add_argument("--speaker", default=None, help="CustomVoice speaker id when --voices is not used")
    p.add_argument("--language", default=os.environ.get("QWEN_TTS_LANGUAGE", "Auto"))
    p.add_argument("--host", default="0.0.0.0")
    p.add_argument("--port", type=int, default=8000)
    p.add_argument("--device", default="cuda", help="Torch device of a single replica (default: cuda)")
    p.add_argument("--gpus", type=int, default=1, help="replicas, one per GPU (cuda:0 .. cuda:N-1)")
    p.add_argument("--max-concurrent", type=int, default=16, help="lock-step streams per GPU")
    p.add_argument("--chunk-frames", type=int, default=8, help="frames per launch = streaming granularity (8 frames = 0.64 s)")
    p.add_argument("--no-warmup", action="store_true", help="open the port at once; the first requests then pay for plan building")
    p.add_argument("--mixed-policies", action="store_true", dest="mixed_policies",
                   help="requests of different sampling policies share every launch, and a request's seed is honoured "
                        "(default: requests are batched with requests of the same policy and a seed is refused)")
    args = p.parse_args(argv)
    logging.basicConfig(level=logging.INFO)
    voices, default_voice = load_voices(args)
    import uvicorn

    backends = build_backends(args.model, args.gpus, args.max_concurrent, args.chunk_frames, device=args.device,
                              mixed_policies=args.mixed_policies)
    if not args.no_warmup:
        logger.info("Warm-up: %.1f s", warm_up(backends, voices))
    app = create_app(backends, voices, default_voice, sample_rate=backends[0].tts.sample_rate, model_name=args.model)
    logger.info("Server listening on http://%s:%d (%d GPU(s), %d streams each)", args.host, args.port, args.gpus, args.max_concurrent)
    try:
        uvicorn.run(app, host=args.host, port=args.port)
    finally:
        for b in backends:
            b.stop()


if __name__ == "__main__":
    main()
