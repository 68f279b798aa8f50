"""Generates tests/golden/clip_tokenizer_golden.npz from the REAL transformers.CLIPTokenizer (5.5.0): the ids of every prompt of
tests/test_tokenizer_cpu.py (padding="max_length", max_length=77, truncation=True) on the vocabulary that test learns, with a CRC32
of each prompt so that a changed prompt list is caught.

    python tests/golden/make_tokenizer_golden.py"""
import os
import sys
import zlib

import numpy as np
import transformers

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests.test_tokenizer_cpu import PROMPTS, _learn  # noqa: E402

if __name__ == "__main__":
    vocab, merges = _learn()
    ref = transformers.CLIPTokenizer(vocab=vocab, merges=[tuple(m) for m in merges])
    ids = np.array([ref(p, padding="max_length", max_length=77, truncation=True).input_ids for p in PROMPTS], np.int64)
    crc = np.array([zlib.crc32(p.encode("utf-8")) for p in PROMPTS], np.int64)
    np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "clip_tokenizer_golden.npz"), ids=ids, prompt_crc=crc)
