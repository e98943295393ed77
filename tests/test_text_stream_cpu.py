"""TextFeed (text_stream.py): committed ids stay a prefix of the final encoding whatever the split of the text into pieces, and
after close they equal the one-shot path's ids assistant(text)[3:-5] followed by tts_eos."""
import random

import pytest

from qwen3_tts_cuda_graphs_b200.text_stream import TextFeed

TEXTS = [
    "the quick brown fox jumps over the lazy dog.",
    "Hello, world! This is a streaming   test, with  double spaces\nand a newline.",
    "speak slowly, calm voice? reference clip says this!",
    "unbelievably antidisestablishmentarianism tokenization re-merges words",
]
EOS = 502


def _random_splits(text, rng):
    cuts = sorted(set(rng.randrange(1, len(text)) for _ in range(rng.randrange(0, len(text)))))
    return [text[a:b] for a, b in zip([0] + cuts, cuts + [len(text)])]


def _check(tokenize, text, pieces):
    feed = TextFeed(tokenize, EOS)
    final = list(tokenize(text))[3:-5]
    seen = []
    for p in pieces:
        seen += feed.push(p)
        assert feed.ids == seen
        assert final[:len(feed.ids)] == feed.ids  # committed ids never change
    seen += feed.close()
    assert feed.ids == seen == final + [EOS]
    assert feed.closed and feed.close() == []


def _tokenizers(tmp_path):
    from helpers import write_tiny_tokenizer
    from qwen3_tts_cuda_graphs_b200.base_model import HFTokenizer, SyntheticTokenizer
    from qwen3_tts_cuda_graphs_b200.config import preset

    cfg = preset("tiny")
    write_tiny_tokenizer(str(tmp_path / "tiny"), cfg)
    yield "synthetic", SyntheticTokenizer(cfg).assistant
    yield "tiny_wordlevel", HFTokenizer(str(tmp_path / "tiny")).assistant
    yield "byte_level_bpe", _byte_bpe(tmp_path / "bpe").assistant


def _byte_bpe(path):
    """A byte-level BPE trained here (offline) with the chat-template special tokens, like the checkpoints' tokenizer.json."""
    from tokenizers import Tokenizer, decoders, models, pre_tokenizers, trainers

    from qwen3_tts_cuda_graphs_b200.base_model import HFTokenizer

    tok = Tokenizer(models.BPE())
    tok.pre_tokenizer = pre_tokenizers.ByteLevel(add_prefix_space=False)
    tok.decoder = decoders.ByteLevel()
    trainer = trainers.BpeTrainer(vocab_size=600, special_tokens=["<|im_start|>", "<|im_end|>"],
                                  initial_alphabet=pre_tokenizers.ByteLevel.alphabet())
    corpus = [t * 3 for t in TEXTS] + ["assistant\n", "streaming text arrives word by word while speech is decoded"] * 20
    tok.train_from_iterator(corpus, trainer)
    path.mkdir(parents=True, exist_ok=True)
    tok.save(str(path / "tokenizer.json"))
    t = HFTokenizer(str(path))
    ids = t.assistant("hello")
    assert len(ids) >= 9 and ids[0] == tok.token_to_id("<|im_start|>")
    return t


@pytest.mark.parametrize("seed", range(6))
def test_text_feed_commit_rule_under_random_splits(tmp_path, seed):
    rng = random.Random(seed)
    for name, tokenize in _tokenizers(tmp_path):
        for text in TEXTS:
            if name == "byte_level_bpe":
                # the template's role ids must stay 3 and the trailer 5 for [3:-5] to be the text: true when the text does not
                # merge with the newline before it or <|im_end|> after it (the special tokens are split off whole)
                assert list(tokenize(text))[:3] == list(tokenize("x"))[:3]
            _check(tokenize, text, _random_splits(text, rng))
            _check(tokenize, text, list(text))
            _check(tokenize, text, [text])


def test_text_feed_commits_nothing_inside_the_last_word():
    from qwen3_tts_cuda_graphs_b200.base_model import SyntheticTokenizer
    from qwen3_tts_cuda_graphs_b200.config import preset

    tok = SyntheticTokenizer(preset("tiny")).assistant
    feed = TextFeed(tok, EOS)
    assert feed.push("hel") == [] and feed.push("lo") == []
    got = feed.push(" wor")
    assert got == tok("hello")[3:-5]
    assert feed.push("ld") == []
    assert feed.close() == tok("hello world")[3:-5][1:] + [EOS]
    with pytest.raises(ValueError):
        feed.push("more")


def test_text_feed_refuses_an_empty_text():
    from qwen3_tts_cuda_graphs_b200.base_model import SyntheticTokenizer
    from qwen3_tts_cuda_graphs_b200.config import preset

    feed = TextFeed(SyntheticTokenizer(preset("tiny")).assistant, EOS)
    feed.push("   ")
    with pytest.raises(ValueError):
        feed.close()
