"""fast_generate — non-streaming generation (`faster_qwen3_tts/generate.py:16-215`) on the fq3 engine.

Two paths behind the reference's signature:

* fused (default): when `talker_graph` / `predictor_graph` are the engine-backed operators of this
  package, prefill and the ENTIRE frame loop run on the device — one prefill launch per <=8 prompt rows
  and one persistent-kernel launch for all frames; the host synchronises once at the end.  This removes the
  >=3 device->host syncs per frame of generate.py:150-197.
* operator-at-a-time: any duck-typed pair exposing the reference's operator seam
  (`tests/test_sampling.py:79-93` doubles) is driven frame by frame with this package's CUDA sampler.

Loop semantics (EOS test before append, min_new_tokens, suppress mask, 16-row embedding sum,
max_seq_len-1 stop) are the ones in SURVEY.md Appendix A1 in both paths.
"""
from __future__ import annotations

import time
from typing import Optional, Sequence, Tuple

import torch

from .engine import SamplingPolicy
from .predictor_graph import PredictorGraph
from .sampling import apply_repetition_penalty, sample_logits
from .talker_graph import TalkerGraph


def _fresh_seed() -> int:
    # honour torch.manual_seed like the reference's torch.multinomial does
    return int(torch.randint(0, 2**62, (1,)).item())


def _left_pads(attention_mask: Optional[torch.Tensor]) -> int:
    if attention_mask is None:
        return 0
    return int((attention_mask.reshape(attention_mask.shape[0], -1)[0] == 0).sum().item())


def is_fused(talker, predictor_graph, talker_graph) -> bool:
    return (
        isinstance(talker_graph, TalkerGraph)
        and isinstance(predictor_graph, PredictorGraph)
        and talker_graph.engine is predictor_graph.engine
        and getattr(talker, "engine", None) is talker_graph.engine
    )


def fused_prefill(talker_graph: TalkerGraph, predictor_graph: PredictorGraph, tie, tam, tth, tpe, policy: SamplingPolicy):
    """Prompt pass + first-token sample on the device; returns the engine and stream index."""
    eng, idx = talker_graph.engine, talker_graph.stream_idx
    T = tie.shape[1]
    if T > eng.max_seq_len:
        raise RuntimeError(
            f"Input is too long: prefill has {T} tokens but max_seq_len={eng.max_seq_len}. "
            "Use shorter text or shorter reference audio."
        )
    eng.set_text_conditioning(idx, tth[0], tpe)
    eng.prefill(idx, tie[0], _left_pads(tam), policy)
    return eng, idx


@torch.inference_mode()
def fast_generate(
    talker,
    talker_input_embeds: torch.Tensor,
    attention_mask: torch.Tensor,
    trailing_text_hiddens: torch.Tensor,
    tts_pad_embed: torch.Tensor,
    config,
    predictor_graph,
    talker_graph,
    max_new_tokens: int = 2048,
    min_new_tokens: int = 2,
    temperature: float = 0.9,
    top_k: int = 50,
    top_p: float = 1.0,
    do_sample: bool = True,
    repetition_penalty: float = 1.05,
    subtalker_dosample: Optional[bool] = None,
    subtalker_top_k: Optional[int] = None,
    subtalker_top_p: Optional[float] = None,
    subtalker_temperature: Optional[float] = None,
    parity_mode: bool = False,
    seed: Optional[int] = None,
) -> Tuple[Optional[torch.Tensor], dict]:
    """Returns (codec_ids int64 [T,16] | None, timing) exactly like generate.py:213-215."""
    if parity_mode:
        raise NotImplementedError(
            "parity_mode drives upstream qwen_tts.talker.generate (generate.py:52-97), which is not part of this engine"
        )
    if is_fused(talker, predictor_graph, talker_graph):
        policy = SamplingPolicy(
            do_sample=do_sample, top_k=top_k, top_p=top_p, temperature=temperature,
            repetition_penalty=repetition_penalty, min_new_tokens=min_new_tokens, suppress_tail=1024,
            seed=_fresh_seed() if seed is None else seed,
        )
        torch.cuda.synchronize()
        t0 = time.time()
        eng, idx = fused_prefill(talker_graph, predictor_graph, talker_input_embeds, attention_mask,
                                 trailing_text_hiddens, tts_pad_embed, policy)
        torch.cuda.synchronize()
        t_prefill = time.time() - t0
        t1 = time.time()
        eng.decode_frames(1, min(max_new_tokens, eng.max_frames), policy, predictor_graph.policy())
        st = eng.status(idx)  # the only synchronisation of the decode loop
        t_decode = time.time() - t1
        n = st.n_frames
        timing = {
            "prefill_ms": t_prefill * 1000, "decode_s": t_decode, "steps": n,
            "ms_per_step": (t_decode / n * 1000) if n > 0 else 0, "steps_per_s": (n / t_decode) if t_decode > 0 else 0,
        }
        if n == 0:
            return None, timing
        return eng.read_codes(idx, 0, n).to(talker_input_embeds.device), timing
    return _generate_with_operators(
        talker, talker_input_embeds, attention_mask, trailing_text_hiddens, tts_pad_embed, config, predictor_graph,
        talker_graph, max_new_tokens, min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty, seed,
    )


@torch.inference_mode()
def fast_generate_batch(talker_graph, predictor_graph, requests, max_new_tokens: int = 2048, min_new_tokens: int = 2,
                        temperature: float = 0.9, top_k: int = 50, top_p: float = 1.0, do_sample: bool = True,
                        repetition_penalty: float = 1.05, seed: Optional[int] = None,
                        policies: Optional[Sequence[SamplingPolicy]] = None):
    """Request-parallel generation (BASELINE configs[3] / [4]; no counterpart in the reference, which is bs = 1): up to
    `engine.max_streams` independent utterances per call; lock-step groups of up to `engine.lockstep_group` (16) of them share
    every weight sweep of the persistent kernel (a stream that hit EOS idles until its group is done; more streams than one
    group run group after group).  `requests` = list of (talker_input_embeds, attention_mask,
    trailing_text_hiddens, tts_pad_embed) as built for fast_generate.  Returns ([codec_ids | None per request], timing).
    Each stream draws from its own Philox stream (seed ^ slot), so a request's tokens do not depend on its neighbours.
    `policies`: one SamplingPolicy per request (seed included), set as the stream's own policy for its prefill and frame loop
    (fq3.h: fq3_set_stream_policy) — requests of different policies share the launches, and each one draws exactly what a
    single-stream run with that policy and seed draws; the scalar arguments then only make the launch-wide policy no stream uses."""
    eng = talker_graph.engine
    if policies is not None:
        policies = list(policies)
        if len(policies) != len(requests):
            raise ValueError(f"policies: {len(policies)} for {len(requests)} requests")
        if not all(isinstance(p, SamplingPolicy) for p in policies):
            raise ValueError("policies: one SamplingPolicy per request")
    policy = SamplingPolicy(
        do_sample=do_sample, top_k=top_k, top_p=top_p, temperature=temperature, repetition_penalty=repetition_penalty,
        min_new_tokens=min_new_tokens, suppress_tail=1024, seed=_fresh_seed() if seed is None else seed,
    )
    sub = predictor_graph.policy()
    out = [None] * len(requests)
    frames = 0
    torch.cuda.synchronize()
    t0 = time.time()
    # one call per engine-full of requests when the wide frame program is available (it forms its own lock-step groups of up to
    # 16); otherwise (1.7B dims) groups of four through the reference-shaped program
    per_call = eng.max_streams if eng.lockstep_group > 4 else min(eng.max_streams, 4)
    for g0 in range(0, len(requests), per_call):
        group = requests[g0:g0 + per_call]
        try:
            for s, (tie, tam, tth, tpe) in enumerate(group):
                if tie.shape[1] > eng.max_seq_len:
                    raise RuntimeError(
                        f"Input is too long: prefill has {tie.shape[1]} tokens but max_seq_len={eng.max_seq_len}. "
                        "Use shorter text or shorter reference audio."
                    )
                eng.set_text_conditioning(s, tth[0], tpe)
                if policies is not None:
                    eng.set_stream_policy(s, policies[g0 + s])
                eng.prefill(s, tie[0], _left_pads(tam), policy)
            eng.decode_frames(len(group), min(max_new_tokens, eng.max_frames), policy, sub)
        finally:
            if policies is not None:  # a later caller of these slots (slot 0: the single-stream API) gets the launch's policy again
                for s in range(len(group)):
                    eng.set_stream_policy(s, None)
        for s in range(len(group)):
            n = eng.status(s).n_frames
            frames += n
            if n > 0:
                out[g0 + s] = eng.read_codes(s, 0, n).to(group[s][0].device)
    torch.cuda.synchronize()
    dt = time.time() - t0
    return out, {"total_s": dt, "frames": frames, "audio_s_per_s": frames * 0.08 / dt if dt > 0 else 0.0}


def suppress_mask_for(config, device) -> torch.Tensor:
    """generate.py:46-50 without the 1024 single-element writes."""
    V, eos = config.vocab_size, config.codec_eos_token_id
    m = torch.zeros(V, dtype=torch.bool, device=device)
    m[max(0, V - 1024):] = True
    if 0 <= eos < V:
        m[eos] = False
    return m


def operator_frames(talker, tie, tam, tth, tpe, config, predictor_graph, talker_graph, max_new_tokens, min_new_tokens,
                    temperature, top_k, top_p, do_sample, repetition_penalty, seed, timing_out: dict):
    """Frame generator over the duck-typed operator seam (one frame per iteration)."""
    eos = config.codec_eos_token_id
    n_groups = config.num_code_groups
    dev = tie.device
    smask = suppress_mask_for(config, dev)
    seed = _fresh_seed() if seed is None else seed
    kw = dict(temperature=temperature, top_k=top_k, top_p=top_p, do_sample=do_sample, suppress_mask=smask, seed=seed)
    embed0 = talker.get_input_embeddings()
    head = talker.codec_head
    embeds = talker.code_predictor.get_input_embeddings()

    t0 = time.time()
    out = talker.forward(
        inputs_embeds=tie, attention_mask=tam, use_cache=True, output_hidden_states=True, return_dict=True,
        trailing_text_hidden=tth, tts_pad_embed=tpe, generation_step=None, past_hidden=None, past_key_values=None,
    )
    past_hidden, gen_step = out.past_hidden, out.generation_step
    token = sample_logits(out.logits[:, -1, :], suppress_tokens=[eos] if min_new_tokens > 0 else None, draw_index=0, **kw)
    prefill_len = talker_graph.prefill_kv(out.past_key_values)
    talker_graph.set_generation_state(tam, getattr(talker, "rope_deltas", None))
    torch.cuda.synchronize()
    timing_out["prefill_s"] = time.time() - t0

    firsts = []
    for step in range(max_new_tokens):
        if token.item() == eos:
            return
        cur = embed0(token.unsqueeze(1))
        codes = predictor_graph.run(torch.cat((past_hidden, cur), dim=1))
        firsts.append(token.view(()))
        rows = [cur] + [embeds[i](codes[i].view(1, 1)) for i in range(n_groups - 1)]
        x = torch.cat(rows, dim=1).sum(1, keepdim=True)
        x = x + (tth[:, gen_step].unsqueeze(1) if gen_step < tth.shape[1] else tpe)
        yield torch.cat([token.view(1), codes])
        pos = prefill_len + step
        if pos >= talker_graph.max_seq_len - 1:
            return
        hidden = talker_graph.run(x, position=pos)
        logits = head(hidden[:, -1, :]).unsqueeze(0)
        if repetition_penalty != 1.0:
            logits = apply_repetition_penalty(logits, torch.stack(firsts), repetition_penalty)
        token = sample_logits(logits.squeeze(0), suppress_tokens=[eos] if len(firsts) < min_new_tokens else None,
                              draw_index=step + 1, **kw)
        past_hidden = hidden[:, -1:, :].clone()
        gen_step += 1


def _generate_with_operators(talker, tie, tam, tth, tpe, config, predictor_graph, talker_graph, max_new_tokens,
                             min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty, seed):
    tinfo: dict = {}
    t0 = time.time()
    frames = list(operator_frames(talker, tie, tam, tth, tpe, config, predictor_graph, talker_graph, max_new_tokens,
                                  min_new_tokens, temperature, top_k, top_p, do_sample, repetition_penalty, seed, tinfo))
    torch.cuda.synchronize()
    total = time.time() - t0
    t_decode = total - tinfo.get("prefill_s", 0.0)
    n = len(frames)
    timing = {
        "prefill_ms": tinfo.get("prefill_s", 0.0) * 1000, "decode_s": t_decode, "steps": n,
        "ms_per_step": (t_decode / n * 1000) if n > 0 else 0, "steps_per_s": (n / t_decode) if t_decode > 0 else 0,
    }
    return (torch.stack(frames) if frames else None), timing
