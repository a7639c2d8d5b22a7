"""Tokenisation parity (north_star: "tokenisation ... must be bit-exact"): polus_b200.tokenization against the Rust
`tokenizers` library -- the engine behind the BertTokenizerFast the reference calls (polus/models.py:275-284) -- on
random vocabularies, Unicode text, sentence pairs, truncation and fixed-length padding.  Sentences of the reference's own
tests (tests/test_models.py:16, tests/test_data.py:374-376) are included.  The library's encodings of these seeded
inputs are stored in tests/golden/wordpiece_tokenizers.npz (generator: tests/golden/make_tokenizer_golden.py), so the
comparison needs no tokenizer package."""
import hashlib
import os
import random

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "wordpiece_tokenizers.npz")
MAX_LENGTH = 50

REFERENCE_SENTENCES = [
    "Hello, my dog is cute",
    "The quick brown fox jumps over the lazy dog.",
    "Chemical compounds such as 2-acetylaminofluorene (AAF) and N-hydroxy-AAF were tested.",
]
LATIN = list("abcdefghijklmnopqrstuvwxyz0123456789")
ACCENTED = [chr(c) for c in (0xE9, 0xFC, 0xF1, 0xE7, 0xE5, 0xF8, 0xDF, 0x130, 0x131, 0x1E9E, 0x1C5)]
CJK = [chr(c) for c in (0x4E2D, 0x6587, 0x5B57, 0x65E5, 0x672C, 0x8A9E)]
GREEK = [chr(c) for c in (0x3B1, 0x3B2, 0x3B3, 0x3B4)]
ALPHABET = LATIN + ACCENTED + CJK + GREEK + ["'", "-"]
PUNCT = list(".,;:!?()[]{}\"/\\%$#@&*+=<>~^`|_") + [chr(c) for c in (0x2014, 0x2026, 0xAB, 0xBB, 0xBF, 0xB7)]
SPACES = [" ", "  ", "\t", "\n", "\r\n"] + [chr(c) for c in (0xA0, 0x2003, 0x2009, 0x3000, 0x2028)]
WEIRD = [chr(c) for c in (0x00, 0xFFFD, 0x200B, 0x301, 0xAD, 0x07, 0x0B, 0x85, 0x202E)]


def make_vocab(rng):
    words = set()
    while len(words) < 400:
        n = rng.randint(1, 6)
        words.add("".join(rng.choice(LATIN + CJK + GREEK) for _ in range(n)))
    pieces = {"##" + "".join(rng.choice(LATIN) for _ in range(rng.randint(1, 3))) for _ in range(300)}
    singles = set(LATIN) | set(CJK) | set(PUNCT[:20]) | {"##" + c for c in LATIN}
    singles -= set("qxz") | {"##q", "##x"}  # some letters missing: words that need them become [UNK]
    vocab = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + sorted(words | pieces | singles)
    return {t: i for i, t in enumerate(dict.fromkeys(vocab))}


def make_text(rng, vocab_words):
    parts = []
    for _ in range(rng.randint(0, 40)):
        r = rng.random()
        if r < 0.45:
            parts.append(rng.choice(vocab_words))
        elif r < 0.65:
            parts.append("".join(rng.choice(ALPHABET) for _ in range(rng.randint(1, 12))))
        elif r < 0.80:
            parts.append(rng.choice(PUNCT))
        elif r < 0.85:
            parts.append(rng.choice(WEIRD))
        elif r < 0.88:
            parts.append(rng.choice(["[SEP]", "[MASK]", "[CLS]", "[UNK]"]))
        elif r < 0.90:
            parts.append("a" * rng.randint(95, 105))
        else:
            parts.append(rng.choice(vocab_words).upper())
        if rng.random() < 0.8:
            parts.append(rng.choice(SPACES))
    return "".join(parts)


def seeded_inputs(lowercase):
    """The vocabulary, texts and sentence pairs the golden encodings were made from."""
    rng = random.Random(1234 + lowercase)
    vocab = make_vocab(rng)
    words = [w for w in vocab if not w.startswith("##") and not w.startswith("[")]
    texts = REFERENCE_SENTENCES + [make_text(rng, words) for _ in range(400)]
    pairs = [(make_text(rng, words), make_text(rng, words)) for _ in range(200)]  # query / document (polus.ir cross-encoder)
    return vocab, texts, pairs


def inputs_digest(texts, pairs):
    return hashlib.sha256("\x1f".join(texts + [s for p in pairs for s in p]).encode("utf-8")).hexdigest()


def golden_key(lowercase):
    return "lower" if lowercase else "cased"


def padded(ids, n_first, vocab):
    """(input_ids, token_type_ids, attention_mask) padded to MAX_LENGTH from the unpadded ids and the first segment's length."""
    n, pad = len(ids), MAX_LENGTH - len(ids)
    return list(ids) + [vocab["[PAD]"]] * pad, [0] * n_first + [1] * (n - n_first) + [0] * pad, [1] * n + [0] * pad


def golden_encodings(z, key, kind, vocab):
    ids, lens, first = (z[f"{key}_{kind}_{f}"].astype(np.int64) for f in ("ids", "len", "first"))
    ends = np.cumsum(lens)
    return [padded(ids[e - n:e].tolist(), int(n0), vocab) for e, n, n0 in zip(ends, lens, first)]


@pytest.mark.parametrize("lowercase", [True, False])
def test_wordpiece_bit_exact_against_tokenizers(lowercase):
    from polus_b200.tokenization import BertWordPieceTokenizer
    vocab, texts, pairs = seeded_inputs(lowercase)
    key = golden_key(lowercase)
    with np.load(GOLDEN) as z:
        assert inputs_digest(texts, pairs) == str(z[f"{key}_inputs_sha256"]), "seeded inputs differ from the golden file's"
        singles, doubles = golden_encodings(z, key, "single", vocab), golden_encodings(z, key, "pair", vocab)
    assert len(singles) == len(texts) and len(doubles) == len(pairs)
    ours = BertWordPieceTokenizer(vocab, lowercase=lowercase)
    for t, e in zip(texts, singles):
        o = ours(t, max_length=MAX_LENGTH, padding="max_length", truncation=True)
        assert (o["input_ids"], o["token_type_ids"], o["attention_mask"]) == e, repr(t)
    for (a, b), e in zip(pairs, doubles):
        o = ours(a, b, max_length=MAX_LENGTH, padding="max_length", truncation=True)
        assert (o["input_ids"], o["token_type_ids"], o["attention_mask"]) == e, (a, b)


def test_batch_call_shape_matches_reference_usage():
    """tests/test_models.py:18-25 call shape: fixed-length int32 arrays for input_ids / token_type_ids / attention_mask."""
    from polus_b200.tokenization import BertWordPieceTokenizer
    rng = random.Random(7)
    vocab = make_vocab(rng)
    tok = BertWordPieceTokenizer(vocab)
    out = tok(REFERENCE_SENTENCES, max_length=64, padding="max_length", truncation=True, return_token_type_ids=True,
              return_attention_mask=True, return_tensors="np")
    for k in ("input_ids", "token_type_ids", "attention_mask"):
        assert out[k].shape == (3, 64) and out[k].dtype == np.int32
    assert (out["input_ids"][:, 0] == vocab["[CLS]"]).all()
    lens = out["attention_mask"].sum(1)
    assert all(out["input_ids"][i, lens[i] - 1] == vocab["[SEP]"] for i in range(3))
