"""Generates tests/golden/mlm_hf_torch.npz: the masked-LM head of HuggingFace `transformers` (torch) BertForMaskedLM and
RobertaForMaskedLM in fp64 -- the independent implementation that pins the head and loss of tests/mlm_ref.py.

Run in the build container (needs torch + transformers, CPU only):  python tests/golden/make_mlm_golden.py

Per family: a 2-layer model at H = 16 with an odd vocabulary (V = 61), weights rounded to float16 values and stored as
float16 (the passes themselves run in fp64).  Stored: the encoder output h [B,S,H], masked_lm_positions / ids /
weights [B,P] (0/1 weights, padding slots at position 0), the head's weights, the logits at the masked positions, HF's
MLM loss (mean over labelled positions), and the gradients of the loss with respect to h and the head's parameters,
the tied decoder included (taken with h as a leaf, so the word-embedding gradient is the decoder's part only).
"""
import os

import numpy as np
import torch
import transformers as tf

HERE = os.path.dirname(os.path.abspath(__file__))
B, S, P, V, H = 3, 10, 4, 61, 16


def one(family, seed):
    torch.manual_seed(seed)
    kw = dict(vocab_size=V, hidden_size=H, num_hidden_layers=2, num_attention_heads=2, intermediate_size=32,
              hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, max_position_embeddings=S + 2)
    if family == "roberta":
        net = tf.RobertaForMaskedLM(tf.RobertaConfig(**kw, type_vocab_size=1, layer_norm_eps=1e-5, pad_token_id=1))
        enc, head, names = net.roberta, net.lm_head, ("dense", "layer_norm")
    else:
        net = tf.BertForMaskedLM(tf.BertConfig(**kw))
        enc, head, names = net.bert, net.cls.predictions, ("transform.dense", "transform.LayerNorm")
    net = net.double()
    with torch.no_grad():
        for p in net.parameters():
            p.copy_((p + 0.1 * torch.randn_like(p)).to(torch.float16).to(torch.float64))
    rng = np.random.default_rng(seed)
    ids = torch.from_numpy(rng.integers(4, V, (B, S)))
    pos = np.zeros((B, P), np.int32)
    w = np.zeros((B, P), np.float32)
    for b, n in enumerate((4, 2, 3)):
        pos[b, :n] = np.sort(rng.choice(np.arange(1, S), n, replace=False))
        w[b, :n] = 1.0
    lab = np.where(w > 0, rng.integers(0, V, (B, P)), 0).astype(np.int32)
    h = enc(input_ids=ids).last_hidden_state.detach().requires_grad_(True)
    dense = head.get_submodule(names[0])
    ln = head.get_submodule(names[1])
    sel = h[torch.arange(B)[:, None], torch.from_numpy(pos).long()].reshape(B * P, H)
    logits = head(sel)                                                  # dense -> gelu -> LN -> tied decoder + bias
    labels = torch.from_numpy(np.where(w > 0, lab, -100).reshape(-1)).long()
    loss = torch.nn.functional.cross_entropy(logits, labels)
    loss.backward()
    word = head.decoder.weight
    g = lambda t: t.grad.detach().numpy()
    f16 = lambda t: t.detach().numpy().astype(np.float16)
    p = f"{family}/"
    return {p + "h": h.detach().numpy(), p + "pos": pos, p + "lab": lab, p + "w": w,
            p + "W_dense": f16(dense.weight.T), p + "b_dense": f16(dense.bias), p + "ln_g": f16(ln.weight),
            p + "ln_b": f16(ln.bias), p + "bias": f16(head.bias), p + "word": f16(word), p + "eps": np.float64(ln.eps),
            p + "logits": logits.detach().numpy(), p + "loss": np.float64(loss.item()), p + "g_h": g(h),
            p + "g_W_dense": g(dense.weight).T, p + "g_b_dense": g(dense.bias), p + "g_ln_g": g(ln.weight),
            p + "g_ln_b": g(ln.bias), p + "g_bias": g(head.bias), p + "g_word": g(word)}


def main():
    out = {}
    out.update(one("bert", 0))
    out.update(one("roberta", 1))
    np.savez_compressed(os.path.join(HERE, "mlm_hf_torch.npz"), **out)


if __name__ == "__main__":
    main()
