"""Incremental text input: decode speech while the text is still arriving (fq3.h: fq3_open_text / fq3_append_text).

Qwen3-TTS reads its text one token per frame: the prompt holds the first text token and frame g adds trailing text row g.  An
open stream therefore needs text row g only when frame g is built, and a stream whose row has not arrived waits on the device
(status.done = 4) without changing its state.  Waits change no arithmetic and no draw, so an open stream's codes equal the codes
of the same stream with the whole text given up front, whatever the arrival schedule.

* `TextFeed` turns `str` pieces (an LLM's token stream, say) into committed text-token ids: ids that no later text can change.
* `text_rows` projects committed ids into trailing text rows exactly as the one-shot prompt builder does.
* `generate_open` is the streaming generator behind `FasterQwen3TTS.generate_*_streaming(text=<iterable of str>)`.

Bit-exactness of the rows.  The one-shot prompt builder projects every text token of a prompt in one
`text_projection(text_embedding(ids))` call; here the ids arrive in pieces and are projected in calls of at most
`MAX_PROJECTION_ROWS` rows.  In the projection's GEMM (fq3_codec.cu, fq3c_run) the split-K partition, and with it the order in
which a row's fp32 products are summed, depends on the row count M only through ceil(M / 128) (the split count also has to fit
the plan's workspace, which codec.attach_splitk_workspace sizes for eight splits of these shapes); the N-tile width also changes
at M = 128, but it only decides which columns a CTA computes, not how an element's K sum is ordered.  So a row's bits are the same in
every call of at most 128 rows.  The open path's rows equal the one-shot path's whenever both calls that produce them stay within
128 rows: the one-shot prompt's call (3 special rows, the instruct ids, 3 role ids and the text, so up to about 120 text tokens),
and here the prompt built at the first commit, which projects every token received by then.  A first piece of more than about
120 tokens, or a longer text on the one-shot side, differs from the other path in the fp32 summation order only.
"""
from __future__ import annotations

import time
from typing import Callable, Iterable, Iterator, List, Sequence

import torch

MAX_PROJECTION_ROWS = 128


class TextFeed:
    """Committed text-token ids of a text that arrives in pieces.

    `tokenize(text)` is the one-shot path's call: the ids of the assistant template around `text` (3 role ids + text + 5 trailer
    ids); the text's ids are `tokenize(text)[3:-5]`.  After every piece the received text is re-tokenized whole, and the feed
    commits ids that (a) come from the text before its last whitespace, where a byte-level BPE no longer merges across, and (b) are
    a prefix of the current full encoding.  Committed ids never change.  `close()` commits the rest of the final encoding and then
    `eos_id` (the tts_eos row that ends the trailing text, model.py:298)."""

    def __init__(self, tokenize: Callable[[str], Sequence[int]], eos_id: int):
        self._tokenize = tokenize
        self.eos_id = int(eos_id)
        self.text = ""
        self.ids: List[int] = []
        self.closed = False

    def _encode(self, text: str) -> List[int]:
        return [int(i) for i in self._tokenize(text)][3:-5]

    def _commit(self, ids: Sequence[int]) -> List[int]:
        if list(ids[:len(self.ids)]) != self.ids:
            raise RuntimeError("the tokenizer changed ids the text feed had already committed")
        new = [int(i) for i in ids[len(self.ids):]]
        self.ids.extend(new)
        return new

    def push(self, piece: str) -> List[int]:
        """Add a piece of text; returns the ids it commits (possibly none)."""
        if self.closed:
            raise ValueError("the text is closed")
        self.text += str(piece)
        cut = len(self.text)
        while cut > 0 and not self.text[cut - 1].isspace():
            cut -= 1
        while cut > 0 and self.text[cut - 1].isspace():
            cut -= 1
        if cut == 0:
            return []
        stable, full = self._encode(self.text[:cut]), self._encode(self.text)
        n = 0
        while n < min(len(stable), len(full)) and stable[n] == full[n]:
            n += 1
        if n <= len(self.ids):
            return []
        return self._commit(full[:n])

    def close(self) -> List[int]:
        """End the text; returns the ids it commits, the final eos_id included."""
        if self.closed:
            return []
        if not self.text.strip():
            raise ValueError("the text is empty")
        self.closed = True
        new = self._commit(self._encode(self.text))
        self.ids.append(self.eos_id)
        return new + [self.eos_id]


def text_rows(talker, ids: Sequence[int]) -> torch.Tensor:
    """bf16 [len(ids), H_t]: text_projection(text_embedding(ids)) in calls of at most MAX_PROJECTION_ROWS rows."""
    dev = talker.device
    out = []
    for i in range(0, len(ids), MAX_PROJECTION_ROWS):
        t = torch.tensor([int(x) for x in ids[i:i + MAX_PROJECTION_ROWS]], dtype=torch.long, device=dev)
        out.append(talker.text_projection(talker.get_text_embeddings()(t)).reshape(t.shape[0], -1))
    if not out:
        return torch.empty(0, talker.config.hidden_size, dtype=torch.bfloat16, device=dev)
    return torch.cat(out, 0)


def generate_open(talker_graph, predictor_graph, prepare: Callable[[str], tuple], feed: TextFeed, pieces: Iterable[str],
                  make_policy: Callable[[], object], max_new_tokens: int, chunk_size: int) -> Iterator[tuple]:
    """Streaming generation of one open-text stream in the engine's slot.  Yields `(codec_chunk int64 [<=chunk_size, 16], info)`
    like streaming.fast_generate_streaming; every chunk has exactly chunk_size frames except the last, so a windowed codec cuts
    the audio where the `str` call cuts it.

    `prepare(text)` builds (tie, tam, tpe, talker) for the received text; the prompt holds the text's first token only, so it is
    built as soon as one id is committed.  `make_policy()` is called after it, where the `str` path draws its seed.  Before
    each launch the generator pulls pieces until the text is chunk_size rows ahead of the stream's generation step or the pieces
    end; when the stream waits for text it blocks on the next piece and launches nothing."""
    from .generate import _left_pads

    eng, idx = talker_graph.engine, talker_graph.stream_idx
    sub = predictor_graph.policy()
    it = iter(pieces)
    t0 = time.time()

    def pull() -> List[int]:
        """The ids one more piece commits (the rest and eos when the pieces end)."""
        try:
            return feed.push(next(it))
        except StopIteration:
            return feed.close()

    pending: List[int] = []
    while not feed.ids and not feed.closed:
        pending += pull()
    tie, tam, tpe, talker = prepare(feed.text)
    policy = make_policy()
    T = tie.shape[1]
    if T > eng.max_seq_len:
        raise RuntimeError(f"Input is too long: prefill has {T} tokens but max_seq_len={eng.max_seq_len}. "
                           "Use shorter text or shorter reference audio.")
    eng.open_text(idx, tpe)
    eng.prefill(idx, tie[0], _left_pads(tam), policy)
    pending = pending[1:]  # the first text token is in the prompt
    rows = 0

    def append(ids: List[int]):
        nonlocal rows
        if ids or feed.closed:
            eng.append_text(idx, text_rows(talker, ids), close=feed.closed)
            rows += len(ids)

    append(pending)
    t_prefill = time.time() - t0
    st = eng.status(idx)
    budget = min(max_new_tokens, eng.max_frames)
    emitted, chunk_idx, buf, t1 = 0, 0, 0, time.time()
    while emitted + buf < budget:
        while not feed.closed and rows < st.gen_step + chunk_size:
            append(pull())
        while st.done == 4 and not feed.closed and rows <= st.gen_step:  # waiting: block on the text
            append(pull())
        eng.decode_frames(1, min(chunk_size - buf, budget - emitted - buf), policy, sub)
        st = eng.status(idx)
        buf = st.n_frames - emitted
        final = st.done in (1, 2, 3) or st.n_frames >= budget
        if buf == chunk_size or (final and buf > 0):
            chunk = eng.read_codes(idx, emitted, buf).to(tie.device)
            emitted += buf
            info = {"chunk_index": chunk_idx, "chunk_steps": buf, "prefill_ms": t_prefill * 1000 if chunk_idx == 0 else 0,
                    "decode_ms": (time.time() - t1) * 1000, "total_steps_so_far": emitted, "is_final": final}
            chunk_idx, buf, t1 = chunk_idx + 1, 0, time.time()
            yield chunk, info
        if final:
            break
