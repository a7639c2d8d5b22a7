"""RoBERTa-family support without a GPU: the position-id rule of tests/roberta_ref.py against HuggingFace's own; its
embeddings + the oracle's encoder layers against HF torch RoBERTa blocks (tests/golden/roberta_hf_torch.npz, generator
tests/golden/make_roberta_golden.py); and the HF config.json fields that select RoBERTa semantics."""
import json
import os

import numpy as np
import pytest

from oracle import numpy_ref as R
from tests import roberta_ref as RR

HERE = os.path.dirname(os.path.abspath(__file__))


def _padded_rows(rng, B, S, pad, vocab=50):
    """Right-, left- and mid-padded rows, plus an all-pad row and an all-real row."""
    ids = rng.integers(0, vocab, (B, S))
    ids[ids == pad] = pad + 2                     # real tokens are never the pad id unless placed below
    for b in range(B):
        kind, L = b % 5, int(rng.integers(0, S + 1))
        if kind == 0:
            ids[b, L:] = pad
        elif kind == 1:
            ids[b, :S - L] = pad
        elif kind == 2:
            ids[b, rng.random(S) < 0.3] = pad
        elif kind == 3:
            ids[b] = pad
    return ids


@pytest.mark.parametrize("pad", [0, 1])
def test_reference_position_ids_equal_transformers(pad):
    import torch
    from transformers.models.roberta.modeling_roberta import RobertaEmbeddings
    rng = np.random.default_rng(pad)
    for B, S in [(10, 1), (10, 7), (15, 64), (5, 512)]:
        ids = _padded_rows(rng, B, S, pad)
        want = RobertaEmbeddings.create_position_ids_from_input_ids(torch.from_numpy(ids), pad).numpy()
        got = RR.roberta_position_ids(ids, pad)
        np.testing.assert_array_equal(got, want)
        assert (got[ids == pad] == pad).all() and (got[ids != pad] > pad).all()


def _golden():
    z = np.load(os.path.join(HERE, "golden", "roberta_hf_torch.npz"))
    tree = lambda tag: {"emb": {k: z[f"{tag}/emb/{k}"].astype(np.float64) for k in ("word", "pos", "type", "emb_ln_g", "emb_ln_b")},
                        "layers": [{k: z[f"{tag}/layers/{i}/{k}"].astype(np.float64) for k in
                                    ("Wqkv", "bqkv", "Wo", "bo", "ln1_g", "ln1_b", "W1", "b1", "W2", "b2", "ln2_g", "ln2_b")}
                                   for i in range(2)]}
    return z, tree("w"), tree("g")


def test_golden_covers_the_padding_cases():
    z, _, g = _golden()
    ids, pad = z["ids"], int(z["pad"])
    assert (ids == pad).all(axis=1).any()                          # an all-pad row
    assert any((r == pad).any() and (r[(r == pad).argmax():] != pad).any() for r in ids)   # a pad id mid-sequence
    np.testing.assert_array_equal(z["pos_ids"], RR.roberta_position_ids(ids, pad))
    assert np.abs(g["emb"]["pos"][pad]).max() > 0 and np.abs(g["emb"]["word"][pad]).max() > 0   # TF: pad rows get gradients


def test_roberta_forward_matches_hf_torch():
    z, w, _ = _golden()
    pos_ids = RR.roberta_position_ids(z["ids"], int(z["pad"]))
    h, _ = RR.embeddings_fwd(z["ids"], z["tt"], w["emb"], pos_ids)
    np.testing.assert_allclose(h, z["h0"], rtol=1e-9, atol=1e-10)
    add = R.attention_mask_additive(z["mask"]).astype(np.float64)
    for i, lp in enumerate(w["layers"]):
        h, _ = R.bert_layer_fwd(h, add, lp, nh=1, eps=1e-5)
        np.testing.assert_allclose(h, z[f"h{i + 1}"], rtol=1e-8, atol=1e-9)


def test_roberta_backward_matches_torch_autograd():
    z, w, g = _golden()
    pos_ids = RR.roberta_position_ids(z["ids"], int(z["pad"]))
    h, ec = RR.embeddings_fwd(z["ids"], z["tt"], w["emb"], pos_ids)
    add = R.attention_mask_additive(z["mask"]).astype(np.float64)
    caches = []
    for lp in w["layers"]:
        h, c = R.bert_layer_fwd(h, add, lp, nh=1, eps=1e-5)
        caches.append(c)
    assert abs((h * z["R"]).sum() - z["loss"]) < 1e-8
    dh = z["R"]
    for i in (1, 0):
        dh, gl = R.bert_layer_bwd(dh, caches[i], w["layers"][i])
        for k, v in gl.items():
            np.testing.assert_allclose(v, g["layers"][i][k], rtol=1e-7, atol=1e-9, err_msg=f"layer {i} {k}")
    ge = RR.embeddings_bwd(dh, ec, w["emb"])
    for k, v in ge.items():
        np.testing.assert_allclose(v, g["emb"][k], rtol=1e-7, atol=1e-9, err_msg=k)


# the config.json of a HuggingFace RoBERTa-base snapshot
ROBERTA_BASE_CONFIG = {
    "architectures": ["RobertaForMaskedLM"], "attention_probs_dropout_prob": 0.1, "bos_token_id": 0, "eos_token_id": 2,
    "hidden_act": "gelu", "hidden_dropout_prob": 0.1, "hidden_size": 768, "initializer_range": 0.02,
    "intermediate_size": 3072, "layer_norm_eps": 1e-05, "max_position_embeddings": 514, "model_type": "roberta",
    "num_attention_heads": 12, "num_hidden_layers": 12, "pad_token_id": 1, "type_vocab_size": 1, "vocab_size": 50265}


def test_roberta_config_json_populates_bert_config(tmp_path):
    from polus_b200.nn import BertConfig
    path = tmp_path / "config.json"
    path.write_text(json.dumps(ROBERTA_BASE_CONFIG))
    cfg = BertConfig(**json.loads(path.read_text()))
    assert (cfg.model_type, cfg.pad_token_id, cfg.layer_norm_eps) == ("roberta", 1, 1e-5)
    assert (cfg.vocab_size, cfg.max_position_embeddings, cfg.type_vocab_size) == (50265, 514, 1)
    assert cfg.roberta_positions
    for model_type in ("xlm-roberta", "camembert"):
        assert BertConfig(model_type=model_type).roberta_positions
    bert = BertConfig()
    assert (bert.model_type, bert.pad_token_id, bert.roberta_positions) == ("bert", 0, False)
