"""CLIP BPE tokenizer (SURVEY 8(f)-1) pinned against transformers.CLIPTokenizer on a vocabulary learned here (the real
vocab.json / merges.txt are not available offline): against its ids stored in tests/golden, and against transformers itself where
it is installed."""
import collections
import os
import zlib

import numpy as np
import pytest

from fast_image_editing_with_generative_models_b200.tokenizer import BOS, EOS, CLIPBPETokenizer, byte_alphabet
from tests.util import GOLDEN

CORPUS = ("a photo of a cat sitting on a wooden bench in the park . a watercolor painting of mountains at sunset , highly detailed . "
          "the quick brown fox jumps over the lazy dog's back ; it's raining cats and dogs ! we've got 2 apples , 37 oranges and 1000 grapes . "
          "a man riding a horse on the beach , cinematic lighting , 4k . an oil painting of a sunflower field . portrait of a woman wearing a red hat . "
          "change the cat to a dog . make it snow . turn the sky purple . a café in zürich . 東京 tower at night . naïve résumé").lower()


def _learn(n_merges=300):
    """A plain BPE trainer: byte alphabet + </w> variants, then the n most frequent pair merges of the corpus."""
    table = byte_alphabet()
    chars = [table[b] for b in range(256)]
    vocab = {c: i for i, c in enumerate(chars)}
    for c in chars:
        vocab[c + "</w>"] = len(vocab)
    words = collections.Counter()
    for w in CORPUS.split():
        enc = [table[b] for b in w.encode("utf-8")]
        enc[-1] += "</w>"
        words[tuple(enc)] += 1
    merges = []
    for _ in range(n_merges):
        pairs = collections.Counter()
        for w, c in words.items():
            for a, b in zip(w, w[1:]):
                pairs[(a, b)] += c
        if not pairs:
            break
        (a, b), _cnt = max(pairs.items(), key=lambda kv: (kv[1], kv[0]))
        merges.append((a, b))
        vocab[a + b] = len(vocab)
        new = collections.Counter()
        for w, c in words.items():
            out, i = [], 0
            while i < len(w):
                if i < len(w) - 1 and w[i] == a and w[i + 1] == b:
                    out.append(a + b); i += 2
                else:
                    out.append(w[i]); i += 1
            new[tuple(out)] += c
        words = new
    vocab[BOS] = len(vocab)
    vocab[EOS] = len(vocab)
    return vocab, merges


PROMPTS = ["", "a photo of a cat", "A Photo   of\ta CAT!!", "it's raining; we've got 37 oranges & 1000 grapes...", "naïve café in Zürich — 東京 tower", "don't you'll I'm they'd he's we're",
           "x" * 300, " ".join(["a watercolor painting of mountains at sunset , highly detailed"] * 12), "<|endoftext|> mid <|startoftext|>", "emoji 🙂 test", "tabs\nand\r\nnewlines",
           "éclair (decomposed accent)", "under_score #hash @at 3.14 1,000"]


@pytest.fixture(scope="module")
def toks():
    """(this tokenizer, transformers.CLIPTokenizer or None where transformers is not installed, vocabulary)."""
    vocab, merges = _learn()
    try:
        import transformers
    except ImportError:
        return CLIPBPETokenizer(vocab, merges), None, vocab
    try:
        ref = transformers.CLIPTokenizer(vocab=vocab, merges=[tuple(m) for m in merges])
    except Exception:
        ref = transformers.CLIPTokenizer(vocab=vocab, merges=[" ".join(m) for m in merges])
    return CLIPBPETokenizer(vocab, merges), ref, vocab


@pytest.fixture(scope="module")
def transformers_ids():
    """transformers' ids of PROMPTS, stored by tests/golden/make_tokenizer_golden.py."""
    z = np.load(os.path.join(GOLDEN, "clip_tokenizer_golden.npz"))
    assert [zlib.crc32(p.encode("utf-8")) for p in PROMPTS] == z["prompt_crc"].tolist(), "PROMPTS changed: regenerate the fixture"
    return z["ids"].tolist()


def test_byte_alphabet_is_a_bijection_on_printables():
    t = byte_alphabet()
    assert len(set(t.values())) == 256 and t[ord("a")] == "a" and t[ord(" ")] == "Ġ" and all(not c.isspace() for c in t.values())


@pytest.mark.parametrize("i", range(len(PROMPTS)))
def test_ids_match_transformers(toks, transformers_ids, i):
    mine, ref, _ = toks
    want = transformers_ids[i]
    if ref is not None:
        assert list(ref(PROMPTS[i], padding="max_length", max_length=77, truncation=True).input_ids) == want
    got = mine(PROMPTS[i])[0]
    assert len(got) == 77 and got == want, (PROMPTS[i], got[:20], want[:20])


def test_batch_and_pad_token(toks):
    mine, ref, vocab = toks
    rows = mine(PROMPTS[:4])
    assert [len(r) for r in rows] == [77] * 4 and rows[0][:2] == [vocab[BOS], vocab[EOS]] and rows[0][2:] == [vocab[EOS]] * 75
    bang = CLIPBPETokenizer(vocab, [], pad_token="!")            # tokenizer_2 of SDXL pads with "!" (id 0 in the real vocabulary)
    assert bang("")[0][2:] == [vocab["!"]] * 75


def test_from_files_roundtrip(toks, tmp_path):
    import json
    mine, _, vocab = toks
    (tmp_path / "vocab.json").write_text(json.dumps(vocab), encoding="utf-8")
    (tmp_path / "merges.txt").write_text("#version: 0.2\n" + "\n".join(" ".join(m) for m in sorted(mine.ranks, key=mine.ranks.get)) + "\n", encoding="utf-8")
    (tmp_path / "special_tokens_map.json").write_text(json.dumps({"pad_token": {"content": "!"}}))
    again = CLIPBPETokenizer.from_files(str(tmp_path))
    assert again.pad_id == vocab["!"] and again.tokenize_ids(PROMPTS[3]) == mine.tokenize_ids(PROMPTS[3])
