"""Generates tests/golden/wordpiece_tokenizers.npz: what the Rust `tokenizers` library (the engine behind the
BertTokenizerFast the reference calls, polus/models.py:275-284) encodes for the seeded vocabularies, texts and sentence
pairs of tests/test_tokenization_cpu.py.  Needs the `tokenizers` package, and pytest (the test module it takes the
inputs from imports it):  python tests/golden/make_tokenizer_golden.py

Stored per casing ("lower" / "cased"): the unpadded token ids of every encoding (concatenated, with their lengths), the
length of the first segment of every pair, and a SHA-256 of the inputs.  The padded ids, token types and attention
mask the test compares against follow from those; main() checks that against the library's own padded output."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from tests.test_tokenization_cpu import MAX_LENGTH, golden_key, inputs_digest, padded, seeded_inputs  # noqa: E402


def library_tokenizer(vocab, lowercase, max_length):
    from tokenizers import Tokenizer, models, normalizers, pre_tokenizers, processors
    tok = Tokenizer(models.WordPiece(vocab, unk_token="[UNK]", max_input_chars_per_word=100))
    tok.add_special_tokens(["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"])
    tok.normalizer = normalizers.BertNormalizer(clean_text=True, handle_chinese_chars=True, strip_accents=None, lowercase=lowercase)
    tok.pre_tokenizer = pre_tokenizers.BertPreTokenizer()
    tok.post_processor = processors.BertProcessing(("[SEP]", vocab["[SEP]"]), ("[CLS]", vocab["[CLS]"]))
    tok.enable_truncation(max_length=max_length, strategy="longest_first")
    tok.enable_padding(length=max_length, pad_id=vocab["[PAD]"], pad_token="[PAD]", pad_type_id=0)
    return tok


def main():
    out = {}
    for lowercase in (True, False):
        vocab, texts, pairs = seeded_inputs(lowercase)
        ref = library_tokenizer(vocab, lowercase, MAX_LENGTH)
        key = golden_key(lowercase)
        for kind, encs in (("single", [ref.encode(t) for t in texts]), ("pair", [ref.encode(a, b) for a, b in pairs])):
            ids, lens, first = [], [], []
            for e in encs:
                n = sum(e.attention_mask)
                n0 = e.type_ids.index(1) if 1 in e.type_ids else n
                assert padded(e.ids[:n], n0, vocab) == (e.ids, e.type_ids, e.attention_mask)
                ids += e.ids[:n]
                lens.append(n)
                first.append(n0)
            out[f"{key}_{kind}_ids"] = np.asarray(ids, np.int16)
            out[f"{key}_{kind}_len"] = np.asarray(lens, np.int16)
            out[f"{key}_{kind}_first"] = np.asarray(first, np.int16)
        out[f"{key}_inputs_sha256"] = np.asarray(inputs_digest(texts, pairs))
    np.savez_compressed(os.path.join(HERE, "wordpiece_tokenizers.npz"), **out)
    print("wrote wordpiece_tokenizers.npz:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
