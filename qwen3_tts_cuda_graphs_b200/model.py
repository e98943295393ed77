"""FasterQwen3TTS — the reference's public API (`faster_qwen3_tts/model.py`) on the B200-native fq3 engine.

Same constructor attributes, same method names, argument meaning and error behaviour as the reference
(SURVEY.md §8b): `from_pretrained`, `generate_voice_clone[_streaming]`, `generate_custom_voice[_streaming]`,
`generate_voice_design[_streaming]`, `_warmup`, `sample_rate`, `_voice_prompt_cache`.  The hot path underneath is
not a CUDA-graph replay of HF modules but the persistent weight-streaming kernel (csrc/fq3_kernel.cuh) and the
codec kernels (csrc/fq3_codec.cu).
"""
from __future__ import annotations

import contextlib
import logging
import os
import wave
from pathlib import Path
from typing import Generator, Iterable, List, Optional, Tuple, Union

import numpy as np
import torch

from .base_model import Qwen3TTSBaseModel
from .engine import SamplingPolicy
from .predictor_graph import PredictorGraph
from .sampling import set_default_engine
from .talker_graph import TalkerGraph

logger = logging.getLogger(__name__)

# sampling arguments one entry of generate_voice_clone_batch(per_request=...) may set
PER_REQUEST_KEYS = ("temperature", "top_k", "top_p", "do_sample", "repetition_penalty", "min_new_tokens", "seed")


class WindowedDecode:
    """The hybrid streaming decode policy of model.py:737-826 for ONE utterance: accumulate and re-decode everything until 25
    frames exist (that first decode also calibrates samples per frame), then decode a sliding window of 25 context frames +
    the new chunk and keep the new chunk's samples.  `push(chunk)` returns the new samples; the context part of a window is
    decoded tail-only (`skip_samples`, codec.CodecDecoder.decode).  Used by `_stream_audio` and by serving.BatchScheduler."""

    def __init__(self, tok, ref_codes, chunk_size: int, context_frames: int = 25):
        self.tok, self.ref_codes = tok, ref_codes
        self.context_frames = context_frames
        self.min_cal = max(context_frames, chunk_size)
        self.all_codes, self.prev_len, self.spf = [], 0, None

    def push(self, chunk: torch.Tensor):
        tok, ref_codes = self.tok, self.ref_codes
        self.all_codes.append(chunk)
        n_new = chunk.shape[0]
        flat = torch.cat(self.all_codes, dim=0)
        n_total = flat.shape[0]
        if self.spf is None:
            codes_in = flat if ref_codes is None else torch.cat([ref_codes.to(flat.device), flat], dim=0)
            skip = 0
            if ref_codes is not None:
                # the reference clip's part is cut off proportionally (model.py:788-795); where the decoder's length law is exact
                # (causal trim: total_upsample samples per frame) the cut is known before the decode, and the vocoder skips what
                # only those samples can see (CodecDecoder.decode: the kept samples are bit-identical to a full decode)
                dec = getattr(tok, "decoder", None)
                if dec is not None and getattr(getattr(dec, "cfg", None), "trans_conv_trim", "") == "right":
                    skip = int(ref_codes.shape[0] / max(codes_in.shape[0], 1) * dec.n_samples(int(codes_in.shape[0])))
            audio_list, sr = tok.decode({"audio_codes": codes_in.unsqueeze(0), "skip_samples": skip} if skip else {"audio_codes": codes_in.unsqueeze(0)})
            audio = audio_list[0].flatten()
            if ref_codes is not None:
                audio = audio[int(ref_codes.shape[0] / max(codes_in.shape[0], 1) * len(audio)):]
            new_audio = audio[self.prev_len:]
            self.prev_len = len(audio)
            if n_total >= self.min_cal:
                self.spf = len(audio) / n_total
            return new_audio, sr
        start = max(0, n_total - n_new - self.context_frames)
        window = flat[start:]
        n_ctx = window.shape[0] - n_new
        cut = int(round(n_ctx * self.spf)) if n_ctx > 0 else 0
        # the context frames are decoded for their state only: tell the decoder which samples will be thrown away
        audio_list, sr = tok.decode({"audio_codes": window.unsqueeze(0), "skip_samples": cut})
        audio = audio_list[0].flatten()
        return (audio[cut:] if n_ctx > 0 else audio), sr


class FasterQwen3TTS:
    def __init__(self, base_model, predictor_graph, talker_graph, device: str = "cuda",
                 dtype: torch.dtype = torch.bfloat16, max_seq_len: int = 2048):
        self.model = base_model
        self.predictor_graph = predictor_graph
        self.talker_graph = talker_graph
        self.device = device
        self.dtype = dtype
        self.max_seq_len = max_seq_len
        self.sample_rate = self._infer_sample_rate(base_model)
        self._warmed_up = False
        self._codec_stream = None  # side stream of the overlapped streaming decode (FQ3_OVERLAP_CODEC)
        self._codec_streams = {}   # chunk_size -> codec.CodecStream (FQ3_STATEFUL_CODEC)
        self._voice_prompt_cache = {}

    @staticmethod
    def _infer_sample_rate(base_model) -> int:
        """model.py:49-69: speech_tokenizer.sample_rate -> base_model.sample_rate -> 24000."""
        rate = None
        tok = getattr(getattr(base_model, "model", None), "speech_tokenizer", None)
        if tok is not None:
            rate = getattr(tok, "sample_rate", None)
        if rate is None:
            rate = getattr(base_model, "sample_rate", None)
        if rate is None:
            logger.warning("Could not infer sample rate from base model; defaulting to 24000 Hz.")
            return 24000
        return int(rate)

    @classmethod
    def from_pretrained(cls, model_name: str, device: str = "cuda", dtype: Union[str, torch.dtype] = torch.bfloat16,
                        attn_implementation: str = "sdpa", max_seq_len: int = 2048, **synthetic_kwargs):
        if isinstance(dtype, str):
            dtype = getattr(torch, dtype)
        if not device.startswith("cuda") or not torch.cuda.is_available():
            raise ValueError("CUDA graphs require CUDA device")  # same message as model.py:96-97
        logger.info(f"Loading Qwen3-TTS model: {model_name}")
        base = Qwen3TTSBaseModel.from_pretrained(model_name, device_map=device, torch_dtype=dtype,
                                                 attn_implementation=attn_implementation, max_seq_len=max_seq_len,
                                                 **synthetic_kwargs)
        eng = base.engine
        predictor_graph = PredictorGraph(eng, do_sample=True, top_k=50, temperature=0.9)  # model.py:124-133
        talker_graph = TalkerGraph(eng)
        set_default_engine(eng)
        return cls(base, predictor_graph, talker_graph, device=device, dtype=dtype, max_seq_len=max_seq_len)

    def _warmup(self, prefill_len: int):
        """model.py:154-163.  Nothing is captured lazily; kept because servers call it explicitly."""
        if self._warmed_up:
            return
        self.predictor_graph.capture(num_warmup=3)
        self.talker_graph.capture(prefill_len=prefill_len, num_warmup=3)
        self._warmed_up = True

    def generate(self, text: str, language: str = "English", max_new_tokens: int = 2048, temperature: float = 0.9,
                 top_k: int = 50, do_sample: bool = True, repetition_penalty: float = 1.05):
        raise NotImplementedError(
            "Default voice generation not yet implemented. Use generate_voice_clone() with reference audio."
        )

    # ---- prompt preparation ----------------------------------------------------------------------
    def _load_ref_audio_with_silence(self, ref_audio, silence_secs: float = 0.5) -> Tuple[np.ndarray, int]:
        """model.py:185-200 (`sf.read` + mono mix-down; soundfile is not in this image: frontend.load_audio)."""
        from .frontend import load_audio

        audio, sr = load_audio(str(ref_audio))
        if silence_secs > 0:
            audio = np.concatenate([audio, np.zeros(int(silence_secs * sr), dtype=np.float32)])
        return audio, sr

    def _prepare_generation(self, text, ref_audio, ref_text, language, xvec_only=True, non_streaming_mode=False,
                            append_silence=True, instruct=None):
        """model.py:202-292."""
        input_ids = self.model._tokenize_texts([self.model._build_assistant_text(text)])
        instruct_ids = [None]
        if instruct:
            instruct_ids = [self.model._tokenize_texts([self.model._build_instruct_text(instruct)])[0]]
        key = (str(ref_audio), ref_text, xvec_only, append_silence)
        if key in self._voice_prompt_cache:
            vcp, ref_ids = self._voice_prompt_cache[key]
        elif xvec_only:
            items = self.model.create_voice_clone_prompt(ref_audio=str(ref_audio), ref_text="", x_vector_only_mode=True)
            vcp = dict(ref_code=[None], ref_spk_embedding=[items[0].ref_spk_embedding], x_vector_only_mode=[True], icl_mode=[False])
            ref_ids = [None] * len(input_ids)
            self._voice_prompt_cache[key] = (vcp, ref_ids)
        else:
            try:
                audio_in = self._load_ref_audio_with_silence(ref_audio, silence_secs=0.5 if append_silence else 0.0)
            except (FileNotFoundError, wave.Error, EOFError, ValueError):
                if self.model.frontend is not None:
                    raise
                audio_in = str(ref_audio)  # synthetic presets fingerprint the path instead
            items = self.model.create_voice_clone_prompt(ref_audio=audio_in, ref_text=ref_text)
            vcp = self.model._prompt_items_to_voice_clone_prompt(items)
            rt = items[0].ref_text
            ref_ids = [self.model._tokenize_texts([self.model._build_ref_text(rt)])[0] if rt else None]
            self._voice_prompt_cache[key] = (vcp, ref_ids)
        m = self.model.model
        tie, tam, tth, tpe = self._build_talker_inputs_local(
            m=m, input_ids=input_ids, ref_ids=ref_ids, voice_clone_prompt=vcp,
            languages=[language] if language is not None else ["Auto"], speakers=None,
            non_streaming_mode=non_streaming_mode, instruct_ids=instruct_ids,
        )
        if not self._warmed_up:
            self._warmup(tie.shape[1])
        talker = m.talker
        talker.rope_deltas = None
        ref_codes = None
        if not xvec_only and vcp.get("ref_code") and vcp["ref_code"][0] is not None:
            ref_codes = vcp["ref_code"][0]
        return m, talker, m.config.talker_config, tie, tam, tth, tpe, ref_codes

    def _prepare_generation_custom(self, text, language, speaker, instruct=None):
        """model.py:294-329."""
        input_ids = self.model._tokenize_texts([self.model._build_assistant_text(text)])
        instruct_ids = [None if not instruct else self.model._tokenize_texts([self.model._build_instruct_text(instruct)])[0]]
        m = self.model.model
        tie, tam, tth, tpe = self._build_talker_inputs_local(
            m=m, input_ids=input_ids, ref_ids=[None], voice_clone_prompt=None,
            languages=[language] if language is not None else ["Auto"], speakers=[speaker],
            non_streaming_mode=False, instruct_ids=instruct_ids,
        )
        if not self._warmed_up:
            self._warmup(tie.shape[1])
        m.talker.rope_deltas = None
        return m, m.talker, m.config.talker_config, tie, tam, tth, tpe

    def _build_talker_inputs_local(self, m, input_ids, ref_ids, voice_clone_prompt, languages, speakers,
                                   non_streaming_mode: bool, instruct_ids=None):
        """Prompt layout of model.py:331-553.  Default: the layout is worked out on the host as one descriptor per row and the rows
        are produced by ONE text_projection call over every text token of the prompt plus one assembly kernel
        (fq3_assemble_prompt); FQ3_PROMPT_FUSED=0 keeps the op-by-op mirror of the reference (`_build_talker_inputs_eager`,
        about sixty small launches), which the parity tests hold the fused path against."""
        eng = getattr(self.talker_graph, "engine", None) or getattr(m.talker, "engine", None)
        if os.environ.get("FQ3_PROMPT_FUSED", "1") == "0" or eng is None:
            return self._build_talker_inputs_eager(m, input_ids, ref_ids, voice_clone_prompt, languages, speakers,
                                                   non_streaming_mode, instruct_ids)
        t, tc, cfg = m.talker, m.config.talker_config, m.config
        dev = t.device
        H = tc.hidden_size
        tok: List[int] = [cfg.tts_bos_token_id, cfg.tts_eos_token_id, cfg.tts_pad_token_id]  # every text token whose projection is needed
        BOS, EOS, PAD = 0, 1, 2

        def host(ids) -> List[int]:
            h = getattr(ids, "_host_ids", None)
            return list(h) if h is not None else [int(x) for x in ids.reshape(-1).tolist()]

        def tp(ids) -> List[int]:  # indices of the projected rows of these token ids
            ids = host(ids) if hasattr(ids, "reshape") else [int(x) for x in ids]
            base = len(tok)
            tok.extend(ids)
            return list(range(base, base + len(ids)))

        spk_rows = m.generate_speaker_prompt(voice_clone_prompt) if voice_clone_prompt is not None else None
        speakers = speakers if speakers is not None else [None] * len(input_ids)
        spk_table: List[torch.Tensor] = []
        ref_tables: List[torch.Tensor] = []
        n_ref = 0
        NONE, CE, SPK, ICL = 0, 1, 2, 3
        seqs, trailing = [], []
        for i, (ids, language, speaker) in enumerate(zip(input_ids, languages, speakers)):
            rows: List[tuple] = []  # (text row index | -1, codec kind, codec index)
            if instruct_ids is not None and instruct_ids[i] is not None:
                rows += [(k, NONE, 0) for k in tp(instruct_ids[i])]
            if spk_rows is None:
                if speaker in ("", None):
                    spk = None
                else:
                    if speaker.lower() not in tc.spk_id:
                        raise NotImplementedError(f"Speaker {speaker} not implemented")
                    spk = (CE, tc.spk_id[speaker.lower()])
            else:
                use = voice_clone_prompt["x_vector_only_mode"][i] or voice_clone_prompt["icl_mode"][i]
                spk = None
                if use:
                    spk = (SPK, len(spk_table))
                    spk_table.append(spk_rows[i].reshape(1, -1))
            assert language is not None
            if language.lower() == "auto":
                lang_id = None
            else:
                if language.lower() not in tc.codec_language_id:
                    raise NotImplementedError(f"Language {language} not implemented")
                lang_id = tc.codec_language_id[language.lower()]
            if language.lower() in ("chinese", "auto") and speaker not in ("", None) and tc.spk_is_dialect.get(speaker.lower()):
                lang_id = tc.codec_language_id[tc.spk_is_dialect[speaker.lower()]]
            prefix = ([tc.codec_nothink_id, tc.codec_think_bos_id, tc.codec_think_eos_id] if lang_id is None else
                      [tc.codec_think_id, tc.codec_think_bos_id, lang_id, tc.codec_think_eos_id])
            codec = [(CE, c) for c in prefix] + ([spk] if spk is not None else []) + [(CE, tc.codec_pad_id), (CE, tc.codec_bos_id)]
            n = len(codec)
            ids_l = host(ids)
            rows += [(k, NONE, 0) for k in tp(ids_l[:3])]  # role tokens
            rows += [(PAD if k < n - 2 else BOS, codec[k][0], codec[k][1]) for k in range(n - 1)]
            icl = (voice_clone_prompt is not None and voice_clone_prompt.get("ref_code") is not None
                   and voice_clone_prompt["icl_mode"][i])
            if icl:
                # generate_icl_prompt (base_model.py): text = TP(ref ++ text) ++ eos, codec = CE(bos) ++ 16-codebook sums of the ref frames
                ref_code = voice_clone_prompt["ref_code"][i]
                text = tp(host(ref_ids[i])[3:-2] + ids_l[3:-5]) + [EOS]
                cod = [(CE, tc.codec_bos_id)] + [(ICL, n_ref + f) for f in range(ref_code.shape[0])]
                ref_tables.append(ref_code.to(torch.int32))
                n_ref += ref_code.shape[0]
                Lt, Lc = len(text), len(cod)
                if non_streaming_mode:
                    rows += [(k, CE, tc.codec_pad_id) for k in text] + [(PAD, ck, ci) for ck, ci in cod]
                    trail = [PAD]
                elif Lt >= Lc:
                    rows += [(text[k], cod[k][0], cod[k][1]) for k in range(Lc)]
                    trail = text[Lc:] if Lt > Lc else [PAD]
                else:
                    rows += [(text[k] if k < Lt else PAD, cod[k][0], cod[k][1]) for k in range(Lc)]
                    trail = [PAD]
            elif non_streaming_mode:
                rows += [(k, CE, tc.codec_pad_id) for k in tp(ids_l[3:-5]) + [EOS]]
                rows.append((PAD, CE, tc.codec_bos_id))
                trail = [PAD]
            else:
                rows.append((tp(ids_l[3:4])[0], codec[-1][0], codec[-1][1]))
                trail = tp(ids_l[4:-5]) + [EOS]
            seqs.append(rows)
            trailing.append(trail)
        # left-pad the batch, right-pad the trailing rows with the tts_pad vector (model.py:519-551); one more row: pad_e itself
        B = len(seqs)
        lens = [len(r) for r in seqs]
        T = max(lens)
        R = max(len(x) for x in trailing)
        desc = torch.zeros(B * T + B * R + 1, 4, dtype=torch.int32)
        desc[:, 0] = -1
        tam = torch.zeros(B, T, dtype=torch.long)
        for b_, rows in enumerate(seqs):
            if rows:
                desc[b_ * T + T - lens[b_]:(b_ + 1) * T, :3] = torch.tensor(rows, dtype=torch.int32)
            tam[b_, T - lens[b_]:] = 1
        for b_, tr in enumerate(trailing):
            base = B * T + b_ * R
            desc[base:base + R, 0] = PAD
            desc[base:base + len(tr), 0] = torch.tensor(tr, dtype=torch.int32)
        desc[-1, 0] = PAD
        tok_dev = torch.tensor(tok, dtype=torch.long).to(dev, non_blocking=True)
        tp_rows = t.text_projection(t.get_text_embeddings()(tok_dev)).contiguous()
        spk_dev = torch.cat(spk_table, 0).to(dev, torch.bfloat16).contiguous() if spk_table else None
        ref_dev = torch.cat(ref_tables, 0).to(dev).contiguous() if ref_tables else None
        out = torch.empty(desc.shape[0], H, dtype=torch.bfloat16, device=dev)
        eng.assemble_prompt(tp_rows, desc.to(dev, non_blocking=True), spk_dev, ref_dev, out)
        tie = out[:B * T].view(B, T, H)
        tth = out[B * T:B * T + B * R].view(B, R, H)
        pad_e = out[-1].view(1, 1, H)
        return tie, tam.to(dev), tth, pad_e

    def _build_talker_inputs_eager(self, m, input_ids, ref_ids, voice_clone_prompt, languages, speakers,
                                   non_streaming_mode: bool, instruct_ids=None):
        """Op-by-op mirror of model.py:331-553 (SURVEY.md Appendix A5).  TP = text_projection(text_embedding(ids)),
        CE = talker codec embedding."""
        t, tc, cfg = m.talker, m.config.talker_config, m.config
        dev = t.device
        TP = lambda ids: t.text_projection(t.get_text_embeddings()(ids))
        CE = lambda ids: t.get_input_embeddings()(torch.tensor(ids, device=dev, dtype=torch.long))
        spk_rows = m.generate_speaker_prompt(voice_clone_prompt) if voice_clone_prompt is not None else None
        speakers = speakers if speakers is not None else [None] * len(input_ids)
        seqs, trailing = [], []
        pad_e = None
        for i, (ids, language, speaker) in enumerate(zip(input_ids, languages, speakers)):
            parts = []
            if instruct_ids is not None and instruct_ids[i] is not None:
                parts.append(TP(instruct_ids[i]))
            # speaker row
            if spk_rows is None:
                if speaker in ("", None):
                    spk = None
                else:
                    if speaker.lower() not in tc.spk_id:
                        raise NotImplementedError(f"Speaker {speaker} not implemented")
                    spk = CE([tc.spk_id[speaker.lower()]]).view(-1)
            else:
                use = voice_clone_prompt["x_vector_only_mode"][i] or voice_clone_prompt["icl_mode"][i]
                spk = spk_rows[i] if use else None
            # language id (dialect speakers override it)
            assert language is not None
            if language.lower() == "auto":
                lang_id = None
            else:
                if language.lower() not in tc.codec_language_id:
                    raise NotImplementedError(f"Language {language} not implemented")
                lang_id = tc.codec_language_id[language.lower()]
            if language.lower() in ("chinese", "auto") and speaker not in ("", None) and tc.spk_is_dialect.get(speaker.lower()):
                lang_id = tc.codec_language_id[tc.spk_is_dialect[speaker.lower()]]
            bos_e, eos_e, pad_e = TP(torch.tensor([[cfg.tts_bos_token_id, cfg.tts_eos_token_id, cfg.tts_pad_token_id]],
                                                  device=dev)).chunk(3, dim=1)
            prefix = ([tc.codec_nothink_id, tc.codec_think_bos_id, tc.codec_think_eos_id] if lang_id is None else
                      [tc.codec_think_id, tc.codec_think_bos_id, lang_id, tc.codec_think_eos_id])
            codec = [CE(prefix).unsqueeze(0)]
            if spk is not None:
                codec.append(spk.view(1, 1, -1))
            codec.append(CE([tc.codec_pad_id, tc.codec_bos_id]).unsqueeze(0))
            codec = torch.cat(codec, dim=1)
            n = codec.shape[1]
            parts.append(TP(ids[:, :3]))  # role tokens
            parts.append(torch.cat([pad_e.expand(-1, n - 2, -1), bos_e], dim=1) + codec[:, :-1])
            icl = (voice_clone_prompt is not None and voice_clone_prompt.get("ref_code") is not None
                   and voice_clone_prompt["icl_mode"][i])
            if icl:
                icl_embed, trail = m.generate_icl_prompt(
                    text_id=ids[:, 3:-5], ref_id=ref_ids[i][:, 3:-2],
                    ref_code=voice_clone_prompt["ref_code"][i].to(dev).clone(), tts_pad_embed=pad_e, tts_eos_embed=eos_e,
                    non_streaming_mode=non_streaming_mode)
                parts.append(icl_embed)
            elif non_streaming_mode:
                n_text = ids[:, 3:-5].shape[1]
                parts.append(torch.cat([TP(ids[:, 3:-5]), eos_e], dim=1) + CE([tc.codec_pad_id] * (n_text + 1)).unsqueeze(0))
                parts.append(pad_e + CE([tc.codec_bos_id]).unsqueeze(0))
                trail = pad_e
            else:
                parts.append(TP(ids[:, 3:4]) + codec[:, -1:])
                trail = torch.cat([TP(ids[:, 4:-5]), eos_e], dim=1)
            seqs.append(torch.cat(parts, dim=1).squeeze(0))
            trailing.append(trail.squeeze(0))
        # left-pad the batch, right-pad trailing hiddens with the tts_pad vector (model.py:519-551)
        lens = [s.shape[0] for s in seqs]
        T = max(lens)
        H = seqs[0].shape[-1]
        tie = torch.zeros(len(seqs), T, H, dtype=seqs[0].dtype, device=dev)
        tam = torch.zeros(len(seqs), T, dtype=torch.long, device=dev)
        for b, s in enumerate(seqs):
            tie[b, T - lens[b]:] = s
            tam[b, T - lens[b]:] = 1
        R = max(x.shape[0] for x in trailing)
        tth = pad_e.reshape(1, 1, H).expand(len(seqs), R, H).clone()
        for b, x in enumerate(trailing):
            tth[b, : x.shape[0]] = x
        return tie, tam, tth, pad_e

    # ---- audio helpers ------------------------------------------------------------------------
    @staticmethod
    def _to_numpy(a) -> np.ndarray:
        if hasattr(a, "cpu"):
            return a.flatten().float().cpu().numpy()
        return a.flatten() if hasattr(a, "flatten") else a

    def _decode_full(self, m, codec_ids, ref_codes=None) -> Tuple[List[np.ndarray], int]:
        """model.py:634-656: prepend ICL ref codes, decode, cut the reference part proportionally."""
        codes = codec_ids if ref_codes is None else torch.cat([ref_codes.to(codec_ids.device), codec_ids], dim=0)
        ref_len = 0 if ref_codes is None else ref_codes.shape[0]
        inputs = {"audio_codes": codes.unsqueeze(0)}
        dec = getattr(m.speech_tokenizer, "decoder", None)
        if ref_len > 0 and dec is not None and getattr(getattr(dec, "cfg", None), "trans_conv_trim", "") == "right":
            # the samples of the reference part are thrown away below: the vocoder need not compute them (WindowedDecode.push)
            inputs["skip_samples"] = int(ref_len / max(codes.shape[0], 1) * dec.n_samples(int(codes.shape[0])))
        audio_list, sr = m.speech_tokenizer.decode(inputs)
        out = []
        for a in audio_list:
            a = self._to_numpy(a)
            if ref_len > 0:
                a = a[int(ref_len / max(codes.shape[0], 1) * len(a)):]
            out.append(a)
        return out, sr

    def _log_rtf(self, timing):
        n = timing["steps"]
        total = timing["prefill_ms"] / 1000 + timing["decode_s"]
        if total > 0:
            logger.info(f"Generated {n / 12.5:.2f}s audio in {total:.2f}s ({timing['ms_per_step']:.1f}ms/step, "
                        f"RTF: {n * 0.08 / total:.2f})")

    def _stream_audio(self, m, stream, ref_codes, chunk_size, to_host: bool = True):
        """Hybrid streaming decode policy of model.py:737-826 (accumulate until 25 frames, then a 25-frame
        left-context sliding window).  to_host=False keeps each chunk as a device tensor (bench.py's
        device-resident leg); the public generators always yield host numpy like the reference."""
        tok = m.speech_tokenizer
        window = WindowedDecode(tok, ref_codes, chunk_size)
        # Opt-in (FQ3_STATEFUL_CODEC=1): stateful incremental decode instead of the windowed re-decode — every chunk costs its own
        # frames only and the audio equals the full non-streaming decode (codec.CodecStream).  The windowed policy below stays
        # the default because it is the reference's.
        cstream = None
        if os.environ.get("FQ3_STATEFUL_CODEC", "0") == "1" and getattr(tok.decoder.cfg, "trans_conv_trim", "") == "right":
            cstream = self._codec_streams.get(chunk_size)
            if cstream is None:
                cstream = self._codec_streams[chunk_size] = tok.decoder.open_stream(max(chunk_size, 8))
        first = True
        for chunk, timing in stream:
            # FQ3_OVERLAP_CODEC (streaming.py): the next chunk is already running on the main stream, so everything below — the
            # window gather and the codec decode — goes to a side stream that only waits for THIS chunk's codes
            ready = timing.get("codes_ready") if isinstance(timing, dict) else None
            if ready is not None:
                if self._codec_stream is None:
                    self._codec_stream = torch.cuda.Stream(device=chunk.device)
                self._codec_stream.wait_event(ready)
            with (torch.cuda.stream(self._codec_stream) if ready is not None else contextlib.nullcontext()):
                if cstream is not None:
                    if first:
                        cstream.reset()
                        if ref_codes is not None:  # ICL: the reference audio's codes are acoustic context, decoded for their state only
                            cstream.decode(ref_codes.to(chunk.device))
                        first = False
                    new_audio, sr = cstream.decode(chunk), tok.sample_rate
                else:
                    new_audio, sr = window.push(chunk)
            if ready is not None:
                self._codec_stream.synchronize()
            yield (self._to_numpy(new_audio) if to_host else new_audio), sr, timing

    def _gen_kwargs(self, max_new_tokens, min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty):
        return dict(max_new_tokens=max_new_tokens, min_new_tokens=min_new_tokens, temperature=temperature, top_k=top_k,
                    top_p=top_p, do_sample=do_sample, repetition_penalty=repetition_penalty,
                    predictor_graph=self.predictor_graph, talker_graph=self.talker_graph)

    # ---- streaming text ------------------------------------------------------------------------
    def _prepare_custom_open(self, text, language, speaker, instruct):
        _, talker, _, tie, tam, _, tpe = self._prepare_generation_custom(text, language, speaker, instruct)
        return tie, tam, tpe, talker

    def _generate_open_text(self, pieces, prepare, chunk_size, max_new_tokens, min_new_tokens, temperature, top_k, top_p,
                            do_sample, repetition_penalty):
        """The `*_streaming` generators with `text` an iterable of str pieces (an LLM's token stream, say): speech starts after
        the first committed text token and the stream waits on the device whenever its next text token has not arrived
        (text_stream.py).  Codes and audio equal the `str` call's on the whole text (text_stream.py: up to ~120 text tokens)."""
        from .generate import _fresh_seed, is_fused
        from .text_stream import TextFeed, generate_open

        m = self.model.model
        if not is_fused(m.talker, self.predictor_graph, self.talker_graph):
            raise ValueError("streaming text runs on the fused engine path only, not on the operator-at-a-time path")
        feed = TextFeed(self.model.tokenizer.assistant, m.config.tts_eos_token_id)

        def make_policy():
            return SamplingPolicy(do_sample=do_sample, top_k=top_k, top_p=top_p, temperature=temperature,
                                  repetition_penalty=repetition_penalty, min_new_tokens=min_new_tokens, suppress_tail=1024,
                                  seed=_fresh_seed())

        stream = generate_open(self.talker_graph, self.predictor_graph, prepare, feed, pieces, make_policy, max_new_tokens,
                               chunk_size)
        yield from self._stream_audio(m, stream, None, chunk_size)

    # ---- voice clone ---------------------------------------------------------------------------
    @torch.inference_mode()
    def generate_voice_clone(self, text: str, language: str, ref_audio, ref_text: str, max_new_tokens: int = 2048,
                             min_new_tokens: int = 2, temperature: float = 0.9, top_k: int = 50, top_p: float = 1.0,
                             do_sample: bool = True, repetition_penalty: float = 1.05, xvec_only: bool = True,
                             non_streaming_mode: bool = True, append_silence: bool = True,
                             instruct: Optional[str] = None) -> Tuple[list, int]:
        from .generate import fast_generate

        m, talker, config, tie, tam, tth, tpe, ref_codes = self._prepare_generation(
            text, ref_audio, ref_text, language=language, xvec_only=xvec_only, non_streaming_mode=non_streaming_mode,
            append_silence=append_silence, instruct=instruct)
        codec_ids, timing = fast_generate(
            talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth, tts_pad_embed=tpe,
            config=config, **self._gen_kwargs(max_new_tokens, min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty))
        if codec_ids is None:
            logger.warning("Generation returned no tokens")
            return [np.zeros(1, dtype=np.float32)], self.sample_rate
        audio, sr = self._decode_full(m, codec_ids, ref_codes)
        self._log_rtf(timing)
        return audio, sr

    @torch.inference_mode()
    def generate_voice_clone_batch(self, texts: List[str], language: str, ref_audio, ref_text: str, max_new_tokens: int = 2048,
                                   min_new_tokens: int = 2, temperature: float = 0.9, top_k: int = 50, top_p: float = 1.0,
                                   do_sample: bool = True, repetition_penalty: float = 1.05, xvec_only: bool = True,
                                   non_streaming_mode: bool = True, append_silence: bool = True,
                                   per_request: Optional[List[dict]] = None) -> Tuple[List[np.ndarray], int]:
        """Several texts in one voice, decoded `max_streams` at a time in lock-step (load the model with
        `from_pretrained(..., max_streams=4)`).  An extension over the reference's bs = 1 API; returns one waveform per text.
        per_request: one dict of sampling arguments per text (keys of PER_REQUEST_KEYS; a key a dict leaves out takes the scalar
        argument, a missing `seed` a fresh one): the texts still share every launch, and each one is sampled exactly as
        generate_voice_clone with those arguments and seed would sample it."""
        from .generate import _fresh_seed, fast_generate_batch

        policies = None
        if per_request is not None:
            if len(per_request) != len(texts):
                raise ValueError(f"per_request: {len(per_request)} entries for {len(texts)} texts")
            scalar = dict(temperature=temperature, top_k=top_k, top_p=top_p, do_sample=do_sample,
                          repetition_penalty=repetition_penalty, min_new_tokens=min_new_tokens)
            policies = []
            for d in per_request:
                unknown = set(d) - set(PER_REQUEST_KEYS)
                if unknown:
                    raise ValueError(f"per_request: unknown key(s) {sorted(unknown)}; allowed: {list(PER_REQUEST_KEYS)}")
                kw = {**scalar, **{k: v for k, v in d.items() if k != "seed"}}
                seed = d.get("seed")
                policies.append(SamplingPolicy(suppress_tail=1024, seed=_fresh_seed() if seed is None else int(seed), **kw).validate())
        reqs, metas = [], []
        for text in texts:
            m, talker, config, tie, tam, tth, tpe, ref_codes = self._prepare_generation(
                text, ref_audio, ref_text, language=language, xvec_only=xvec_only, non_streaming_mode=non_streaming_mode,
                append_silence=append_silence)
            reqs.append((tie, tam, tth, tpe))
            metas.append((m, ref_codes))
        codes, timing = fast_generate_batch(self.talker_graph, self.predictor_graph, reqs, max_new_tokens=max_new_tokens,
                                            min_new_tokens=min_new_tokens, temperature=temperature, top_k=top_k, top_p=top_p,
                                            do_sample=do_sample, repetition_penalty=repetition_penalty, policies=policies)
        audio = []
        for c, (m, ref_codes) in zip(codes, metas):
            if c is None:
                audio.append(np.zeros(1, dtype=np.float32))
            else:
                a, _ = self._decode_full(m, c, ref_codes)
                audio.append(a[0])
        logger.info(f"batch of {len(texts)}: {timing['frames']} frames in {timing['total_s']:.2f}s "
                    f"({timing['audio_s_per_s']:.1f} audio-s/s before the codec)")
        return audio, self.sample_rate

    @torch.inference_mode()
    def generate_voice_clone_streaming(self, text: Union[str, Iterable[str]], language: str, ref_audio, ref_text: str,
                                       max_new_tokens: int = 2048, min_new_tokens: int = 2, temperature: float = 0.9,
                                       top_k: int = 50, top_p: float = 1.0, do_sample: bool = True,
                                       repetition_penalty: float = 1.05, chunk_size: int = 12, xvec_only: bool = True,
                                       non_streaming_mode: bool = True, append_silence: bool = True, parity_mode: bool = False,
                                       instruct: Optional[str] = None) -> Generator[Tuple[np.ndarray, int, dict], None, None]:
        from .streaming import fast_generate_streaming

        if parity_mode:
            raise NotImplementedError("parity_mode runs upstream qwen_tts with a dynamic cache (streaming.py:192-359); not part of this engine")
        if not isinstance(text, str):
            if not xvec_only:
                raise ValueError("streaming text: an ICL voice clone sums the text into the reference-code rows; use xvec_only=True")
            if non_streaming_mode:
                raise ValueError("streaming text needs non_streaming_mode=False (the whole text is in the prompt otherwise)")

            def prepare(s):
                m, talker, _, tie, tam, _, tpe, _ = self._prepare_generation(
                    s, ref_audio, ref_text, language=language, xvec_only=True, non_streaming_mode=False,
                    append_silence=append_silence, instruct=instruct)
                return tie, tam, tpe, talker

            yield from self._generate_open_text(text, prepare, chunk_size, max_new_tokens, min_new_tokens, temperature, top_k, top_p,
                                                do_sample, repetition_penalty)
            return
        m, talker, config, tie, tam, tth, tpe, ref_codes = self._prepare_generation(
            text, ref_audio, ref_text, language=language, xvec_only=xvec_only, non_streaming_mode=non_streaming_mode,
            append_silence=append_silence, instruct=instruct)
        stream = fast_generate_streaming(
            talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth, tts_pad_embed=tpe,
            config=config, chunk_size=chunk_size,
            **self._gen_kwargs(max_new_tokens, min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty))
        yield from self._stream_audio(m, stream, ref_codes, chunk_size)

    # ---- custom voice --------------------------------------------------------------------------
    def _check_custom(self, language, speaker):
        if self.model.model.tts_model_type != "custom_voice":
            raise ValueError("Loaded model does not support custom voice generation")
        self.model._validate_languages([language])
        self.model._validate_speakers([speaker])

    @torch.inference_mode()
    def generate_custom_voice(self, text: str, speaker: str, language: str, instruct: Optional[str] = None,
                              max_new_tokens: int = 2048, min_new_tokens: int = 2, temperature: float = 0.9, top_k: int = 50,
                              top_p: float = 1.0, do_sample: bool = True, repetition_penalty: float = 1.05) -> Tuple[list, int]:
        from .generate import fast_generate

        self._check_custom(language, speaker)
        if self.model.model.tts_model_size in "0b6":  # model.py:849-850
            instruct = None
        m, talker, config, tie, tam, tth, tpe = self._prepare_generation_custom(text, language, speaker, instruct)
        codec_ids, timing = fast_generate(
            talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth, tts_pad_embed=tpe,
            config=config, **self._gen_kwargs(max_new_tokens, min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty))
        if codec_ids is None:
            logger.warning("Generation returned no tokens")
            return [np.zeros(1, dtype=np.float32)], self.sample_rate
        audio, sr = self._decode_full(m, codec_ids)
        self._log_rtf(timing)
        return audio, sr

    @torch.inference_mode()
    def generate_custom_voice_streaming(self, text: Union[str, Iterable[str]], speaker: str, language: str, instruct: Optional[str] = None,
                                        max_new_tokens: int = 2048, min_new_tokens: int = 2, temperature: float = 0.9,
                                        top_k: int = 50, top_p: float = 1.0, do_sample: bool = True,
                                        repetition_penalty: float = 1.05, chunk_size: int = 12):
        from .streaming import fast_generate_streaming

        self._check_custom(language, speaker)
        if self.model.model.tts_model_size in "0b6":
            instruct = None
        if not isinstance(text, str):
            yield from self._generate_open_text(
                text, lambda s: self._prepare_custom_open(s, language, speaker, instruct), chunk_size, max_new_tokens,
                min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty)
            return
        m, talker, config, tie, tam, tth, tpe = self._prepare_generation_custom(text, language, speaker, instruct)
        stream = fast_generate_streaming(
            talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth, tts_pad_embed=tpe,
            config=config, chunk_size=chunk_size,
            **self._gen_kwargs(max_new_tokens, min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty))
        yield from self._stream_audio(m, stream, None, chunk_size)

    # ---- voice design --------------------------------------------------------------------------
    def _check_design(self, language):
        if self.model.model.tts_model_type != "voice_design":
            raise ValueError("Loaded model does not support voice design generation")
        self.model._validate_languages([language])

    @torch.inference_mode()
    def generate_voice_design(self, text: str, instruct: str, language: str, max_new_tokens: int = 2048,
                              min_new_tokens: int = 2, temperature: float = 0.9, top_k: int = 50, top_p: float = 1.0,
                              do_sample: bool = True, repetition_penalty: float = 1.05) -> Tuple[list, int]:
        from .generate import fast_generate

        self._check_design(language)
        m, talker, config, tie, tam, tth, tpe = self._prepare_generation_custom(text, language, None, instruct)
        codec_ids, timing = fast_generate(
            talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth, tts_pad_embed=tpe,
            config=config, **self._gen_kwargs(max_new_tokens, min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty))
        if codec_ids is None:
            logger.warning("Generation returned no tokens")
            return [np.zeros(1, dtype=np.float32)], self.sample_rate
        audio, sr = self._decode_full(m, codec_ids)
        self._log_rtf(timing)
        return audio, sr

    @torch.inference_mode()
    def generate_voice_design_streaming(self, text: Union[str, Iterable[str]], instruct: str, language: str, max_new_tokens: int = 2048,
                                        min_new_tokens: int = 2, temperature: float = 0.9, top_k: int = 50,
                                        top_p: float = 1.0, do_sample: bool = True, repetition_penalty: float = 1.05,
                                        chunk_size: int = 12):
        from .streaming import fast_generate_streaming

        self._check_design(language)
        if not isinstance(text, str):
            yield from self._generate_open_text(
                text, lambda s: self._prepare_custom_open(s, language, None, instruct), chunk_size, max_new_tokens,
                min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty)
            return
        m, talker, config, tie, tam, tth, tpe = self._prepare_generation_custom(text, language, None, instruct)
        stream = fast_generate_streaming(
            talker=talker, talker_input_embeds=tie, attention_mask=tam, trailing_text_hiddens=tth, tts_pad_embed=tpe,
            config=config, chunk_size=chunk_size,
            **self._gen_kwargs(max_new_tokens, min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty))
        yield from self._stream_audio(m, stream, None, chunk_size)
