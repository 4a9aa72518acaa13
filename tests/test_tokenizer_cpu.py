"""Caption tokenizer (vtp_b200/text_tokenizer.py, SURVEY.md §8(f)4) — CPU tests.

  * against the reference `SimpleTokenizer` (vtp/tokenizers/text_tokenizer.py:144-295), recorded by
    oracle/make_golden_tokenizer.py on a corpus built to hit the pattern's branches: identical vocabulary, identical ids
    for every caption, identical truncation and decoding.  The vocabulary is the reference's data file reduced to the
    merges that corpus uses (tests/golden/tokenizer_bpe.txt.gz; the reduction leaves every caption's split unchanged);
  * self-contained cases on a tiny synthetic vocabulary (written to a temp dir): merge order, end-of-word variants,
    special tokens, truncation rule, errors."""
import gzip
import os

import pytest
import torch

from oracle.make_golden_tokenizer import EXTRA, LENGTHS, VOCAB, corpus, digest
from tests.util import load_golden
from vtp_b200.text_tokenizer import BPETokenizer, find_bpe_file, get_tokenizer


def test_token_ids_equal_the_live_reference():
    meta, g = load_golden("tokenizer")
    h = meta["sha256"]
    texts = corpus()
    assert digest(texts) == meta["corpus_sha256"]
    ours = BPETokenizer(VOCAB)
    assert digest(sorted(ours.encoder.items())) == h["encoder"] and digest(sorted(ours.decoder.items())) == h["decoder"]
    assert digest(sorted(ours.byte_decoder.items())) == h["byte_decoder"]
    assert [ours.vocab_size, ours.sot_token_id, ours.eot_token_id, ours.all_special_ids, ours.context_length] == \
           [meta[k] for k in ("vocab_size", "sot_token_id", "eot_token_id", "all_special_ids", "context_length")]
    ref_ids = torch.split(g["ids_flat"].long(), g["ids_len"].tolist())
    ids = [ours.encode(text) for text in texts]
    for text, a, b in zip(texts, ids, ref_ids):
        assert a == b.tolist(), text
    assert digest([ours.decode(a) for a in ids]) == h["decoded"]
    for L in LENGTHS:                           # padding, exact fit, truncation (last slot becomes <end_of_text>)
        x = ours(texts, L)
        assert x.dtype == torch.long and digest(x.tolist()) == h[f"batch_{L}"], L
    assert digest(ours("one caption").tolist()) == h["one_caption"]
    # second call: served from the caption cache, same ids
    assert digest(ours(texts).tolist()) == h["batch_None"]
    # no lower-casing + an extra special token (case-sensitive cache hit of specials, as upstream)
    o2 = BPETokenizer(VOCAB, clean="whitespace", additional_special_tokens=["<mask>"])
    assert digest(o2(texts + EXTRA).tolist()) == h["extra_special"]
    assert o2.vocab_size == meta["vocab_size_extra_special"] == ours.vocab_size + 1
    # get_tokenizer mirrors the factory
    assert get_tokenizer(bpe_path=VOCAB, context_length=32)("a cat").shape == (1, 32)


def _tiny_vocab(tmp_path):
    """header line + five merges: 't h', 'th e</w>', 'c a', 'ca t</w>', 'a t</w>' (the last can never apply after 'c a')."""
    p = tmp_path / "tiny_bpe.txt.gz"
    with gzip.open(p, "wb") as f:
        f.write('"version"\nt h\nth e</w>\nc a\nca t</w>\na t</w>\n'.encode("utf-8"))
    return str(p)


def test_merge_order_and_layout_on_a_synthetic_vocabulary(tmp_path):
    tok = BPETokenizer(_tiny_vocab(tmp_path), context_length=8)
    # layout: 256 byte symbols, 256 end-of-word variants, merges in file order (a trailing empty line yields one more,
    # empty, entry exactly as upstream's split('\n')), then the two special tokens
    assert tok.encoder["th"] == 512 and tok.encoder["the</w>"] == 513 and tok.encoder["cat</w>"] == 515
    assert tok.sot_token_id == tok.vocab_size - 2 and tok.eot_token_id == tok.vocab_size - 1
    b = lambda ch: tok.encoder[ch]
    assert tok.encode("the") == [513]                                   # t h -> th ; th e</w> -> the</w>
    assert tok.encode("The  cat") == [513, 515]                         # lower-cased, whitespace collapsed
    assert tok.encode("that") == [512, tok.encoder["at</w>"]]           # 't h' (rank 0) before 'a t</w>' (rank 4)
    assert tok.encode("tht") == [512, b("t</w>")]                       # no merge for (th, t</w>)
    assert tok.encode("ththe") == [512, 513]                            # every occurrence of the best pair merges per round
    assert tok.encode("é") == [b("Ã"), b("©") + 256]                    # two UTF-8 bytes, the last one end-of-word
    assert tok.encode("<end_of_text>") == [tok.eot_token_id]
    assert tok.decode(tok.encode("the cat é")) == "the cat é "
    out = tok(["the", "the cat the cat the cat the cat", ""])
    sot, eot = tok.sot_token_id, tok.eot_token_id
    assert out.tolist() == [[sot, 513, eot, 0, 0, 0, 0, 0],
                            [sot, 513, 515, 513, 515, 513, 515, eot],    # cut to 8, last slot = end token
                            [sot, eot, 0, 0, 0, 0, 0, 0]]
    assert tok(["the"], context_length=2).tolist() == [[sot, eot]]


def test_vocabulary_lookup_and_errors(tmp_path, monkeypatch):
    with pytest.raises(FileNotFoundError):
        BPETokenizer(str(tmp_path / "missing.txt.gz"))
    monkeypatch.setenv("VTP_BPE_PATH", _tiny_vocab(tmp_path))
    assert find_bpe_file() == os.path.abspath(_tiny_vocab(tmp_path))
    assert BPETokenizer().encode("the") == [513]
    with pytest.raises(AssertionError):
        BPETokenizer(context_length=None)("x")
