"""TEST INFRASTRUCTURE ONLY — golden for the caption tokenizer (tests/test_tokenizer_cpu.py), from the reference's
`SimpleTokenizer` and its vocabulary file (see oracle/ref_harness.py for where the reference is imported from):

    python -m oracle.make_golden_tokenizer

The full vocabulary (1.3 MB) is not stored.  The corpus is tokenized with it once while recording every merge that
fires; tests/golden/tokenizer_bpe.txt.gz keeps only those merges, in file order.  BPE fires the lowest-ranked merge
present in a word at each step, and dropping merges that never fire on a word cannot change that choice, so the
reduced vocabulary splits the corpus into the same token strings (checked below; the ids differ, being ranks in the
smaller file).  The reference tokenizer built on the reduced file then gives the stored ids, decodes and vocabulary
layout (tokenizer.json + tokenizer.npz)."""
from __future__ import annotations

import gzip
import hashlib
import importlib.util
import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
VOCAB = os.path.join(OUT, "tokenizer_bpe.txt.gz")

CORPUS = [
    "a photo of a cat", "A Photo of a CAT!!!", "  multiple   spaces\tand\nnewlines ",
    "it's the dog's ball, they've won; I'm here, we'll go, he'd say, don't", "'s't're've'm'll'd", "''''",
    "naïve café déjà vu — “quotes” ‘single’ … ellipsis", "日本語のテキスト と 中文文本 and한국어", "emoji 😀😃 🤖👍🏽 flags 🇩🇪",
    "numbers 1234567890 3.14159 1e-5 ½ ²", "&amp;lt;b&amp;gt; html &amp; entities &lt;i&gt; &#39;x&#39;",
    "<start_of_text> literal specials <end_of_text> inside", "<START_OF_TEXT> upper special", "", "   ", "x", "a" * 300,
    "word " * 200, "supercalifragilisticexpialidocious antidisestablishmentarianism",
    "e-mail: someone@example.com, http://example.com/path?query=1&b=2", "tabs\tand\x00control\x07chars",
    "mixed123abc456 under_score-dash", "ÀÉÎÕÜ ßẞ ǅ İi", "𝔘𝔫𝔦𝔠𝔬𝔡𝔢 math 𝟘𝟙𝟚", "！？。、", "á combining ë",
]
EXTRA = ["Keep CASE <mask> <Mask> <start_of_text>"]     # for the case-keeping tokenizer with an extra special token
LENGTHS = (None, 8, 16, 77, 200)                        # padding, exact fit, truncation (last slot = end token)


def corpus():
    rng = random.Random(0)
    alphabet = "abcdefghijklmnopqrstuvwxyz  ABC.,!?'0123456789-éüñ日本😀"
    return CORPUS + ["".join(rng.choice(alphabet) for _ in range(rng.randint(1, 120))) for _ in range(400)]


class _Recording(dict):
    """bpe_ranks that remembers every pair the merge loop finds in it: the loop asks `in` only of the pair it is
    about to merge."""

    def __init__(self, d):
        super().__init__(d)
        self.fired = set()

    def __contains__(self, k):
        hit = dict.__contains__(self, k)
        if hit:
            self.fired.add(k)
        return hit


def digest(obj) -> str:
    """sha256 of a JSON-able value (lists of ids, sorted vocabulary items, strings)."""
    return hashlib.sha256(json.dumps(obj, ensure_ascii=False).encode("utf-8")).hexdigest()


def main():
    root = rh.REF_ROOT
    spec = importlib.util.spec_from_file_location("_ref_text_tokenizer", os.path.join(root, "vtp", "tokenizers", "text_tokenizer.py"))
    ref_mod = importlib.util.module_from_spec(spec)       # by path: `import vtp` needs omegaconf
    spec.loader.exec_module(ref_mod)
    full_path = os.path.join(root, "tools", "bpe_simple_vocab_16e6.txt.gz")
    texts = corpus()
    extra = texts + EXTRA
    full = ref_mod.SimpleTokenizer(full_path)
    full2 = ref_mod.SimpleTokenizer(full_path, clean="whitespace", additional_special_tokens=["<mask>"])
    full.bpe_ranks, full2.bpe_ranks = _Recording(full.bpe_ranks), _Recording(full2.bpe_ranks)
    strings = lambda tok, t: [tok.decoder[i] for i in tok.encode(t)]
    want = [strings(full, t) for t in texts + ["one caption", "a cat"]]
    want2 = [strings(full2, t) for t in extra]
    fired = full.bpe_ranks.fired | full2.bpe_ranks.fired

    lines = gzip.open(full_path).read().decode("utf-8").split("\n")
    kept = [ln for ln in lines[1:49152 - 256 - 2 + 1] if tuple(ln.split()) in fired]
    with open(VOCAB, "wb") as f:                          # fixed header time: the file is byte-for-byte reproducible
        with gzip.GzipFile(fileobj=f, mode="wb", mtime=0) as z:
            z.write("\n".join([lines[0]] + kept).encode("utf-8"))

    ref = ref_mod.SimpleTokenizer(VOCAB)
    ref2 = ref_mod.SimpleTokenizer(VOCAB, clean="whitespace", additional_special_tokens=["<mask>"])
    assert [strings(ref, t) for t in texts + ["one caption", "a cat"]] == want
    assert [strings(ref2, t) for t in extra] == want2

    ids = [ref.encode(t) for t in texts]
    meta = {"corpus_sha256": digest(texts), "vocab_size": ref.vocab_size, "sot_token_id": ref.sot_token_id,
            "eot_token_id": ref.eot_token_id, "all_special_ids": ref.all_special_ids, "context_length": ref.context_length,
            "vocab_size_extra_special": ref2.vocab_size, "merges_kept": len(kept),
            "sha256": {"encoder": digest(sorted(ref.encoder.items())), "decoder": digest(sorted(ref.decoder.items())),
                       "byte_decoder": digest(sorted(ref.byte_decoder.items())),
                       "decoded": digest([ref.decode(i) for i in ids]),
                       "one_caption": digest(ref("one caption").tolist()),
                       "extra_special": digest(ref2(extra).tolist()),
                       **{f"batch_{L}": digest(ref(texts, L).tolist()) for L in LENGTHS}}}
    with open(os.path.join(OUT, "tokenizer.json"), "w") as f:
        json.dump(meta, f, indent=1)
    np.savez_compressed(os.path.join(OUT, "tokenizer.npz"), ids_flat=np.array([i for row in ids for i in row], dtype=np.int16),
                        ids_len=np.array([len(row) for row in ids], dtype=np.int16))
    print("tokenizer: kept", len(kept), "merges of", 49152 - 256 - 2, "vocab", ref.vocab_size)


if __name__ == "__main__":
    main()
