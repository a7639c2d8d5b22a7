"""Generates tests/golden/roberta_hf_torch.npz: inputs, weights, outputs and gradients of HuggingFace `transformers`
(torch) RoBERTa blocks -- RobertaEmbeddings + 2 RobertaLayers in fp64 -- the independent implementation that pins the
RoBERTa reference of tests/roberta_ref.py.

Run in the build container (needs torch + transformers, CPU only):  python tests/golden/make_roberta_golden.py

Configuration of the RoBERTa family: pad_token_id 1, type_vocab_size 1, layer_norm_eps 1e-5.  The batch holds right-
padded rows, one row with the pad id in mid-sequence (it takes position padding_idx and does not advance the count) and
one all-pad row.  The model is small (H = 16, one head of 16, I = 32) and the weights are rounded to float16 values and
stored as float16, so the file stays small; the forward and backward passes themselves run in fp64.

Gradient semantics: torch's nn.Embedding(padding_idx=...) drops the gradient of the padding row; TensorFlow's embedding
lookup, which the reference runs (TFRobertaEmbeddings), does not.  `padding_idx` is therefore removed from the word and
the position embedding modules before the forward pass, so the stored gradients follow TF: the padding rows collect the
gradients of pad tokens.  The position ids themselves still come from RobertaEmbeddings.padding_idx (= pad_token_id).
"""
import os

import numpy as np
import torch
from transformers import RobertaConfig
from transformers.models.roberta.modeling_roberta import RobertaEmbeddings, RobertaLayer

HERE = os.path.dirname(os.path.abspath(__file__))
PAD = 1


def main():
    torch.manual_seed(0)
    torch.set_grad_enabled(True)
    cfg = RobertaConfig(vocab_size=24, hidden_size=16, num_hidden_layers=2, num_attention_heads=1, intermediate_size=32,
                        max_position_embeddings=16, type_vocab_size=1, hidden_dropout_prob=0.0,
                        attention_probs_dropout_prob=0.0, layer_norm_eps=1e-5, pad_token_id=PAD)
    cfg._attn_implementation = "eager"
    emb = RobertaEmbeddings(cfg).double()
    emb.word_embeddings.padding_idx = None      # TF semantics for the gradients (module docstring)
    emb.position_embeddings.padding_idx = None
    layers = [RobertaLayer(cfg).double() for _ in range(2)]
    for m in [emb] + layers:
        for name, p in m.named_parameters():
            with torch.no_grad():
                if "LayerNorm.weight" in name:
                    p.copy_(1 + 0.1 * torch.randn_like(p))
                elif name.endswith("bias"):
                    p.copy_(0.05 * torch.randn_like(p))
                else:
                    p.copy_(0.1 * torch.randn_like(p))
                p.copy_(p.half().double())          # exactly representable in the float16 the file stores
    B, S = 4, 8
    g = torch.Generator().manual_seed(1)
    ids = torch.randint(3, 24, (B, S), generator=g)
    lens = [8, 5, 7, 0]
    for b, L in enumerate(lens):
        ids[b, L:] = PAD
    ids[2, 3] = PAD                               # a pad id inside the real tokens of row 2
    tt = torch.zeros(B, S, dtype=torch.long)
    mask = (torch.arange(S)[None, :] < torch.tensor(lens)[:, None]).long()
    add_mask = (1.0 - mask.double())[:, None, None, :] * -10000.0
    pos_ids = RobertaEmbeddings.create_position_ids_from_input_ids(ids, PAD)
    h = emb(input_ids=ids, token_type_ids=tt)
    hs = [h]
    for l in layers:
        h = l(h, attention_mask=add_mask)
        h = h[0] if isinstance(h, tuple) else h
        hs.append(h)
    R = torch.randn(h.shape, generator=g, dtype=torch.double)
    loss = (h * R).sum()
    loss.backward()
    out = {"ids": ids.numpy(), "tt": tt.numpy(), "mask": mask.numpy(), "pos_ids": pos_ids.numpy(), "R": R.numpy(),
           "loss": np.float64(loss.item()), "pad": np.int64(PAD)}
    for i, t in enumerate(hs):
        out[f"h{i}"] = t.detach().numpy()
    n = lambda p: p.detach().numpy()
    e = emb
    for tag, f in (("w", lambda p: n(p).astype(np.float16)), ("g", lambda p: n(p.grad))):
        out[f"{tag}/emb/word"] = f(e.word_embeddings.weight)
        out[f"{tag}/emb/pos"] = f(e.position_embeddings.weight)
        out[f"{tag}/emb/type"] = f(e.token_type_embeddings.weight)
        out[f"{tag}/emb/emb_ln_g"] = f(e.LayerNorm.weight)
        out[f"{tag}/emb/emb_ln_b"] = f(e.LayerNorm.bias)
        for i, l in enumerate(layers):
            a, o = l.attention.self, l.attention.output
            # torch Linear stores [out,in]; Keras kernels are [in,out]
            out[f"{tag}/layers/{i}/Wqkv"] = np.concatenate([f(a.query.weight).T, f(a.key.weight).T, f(a.value.weight).T], 1)
            out[f"{tag}/layers/{i}/bqkv"] = np.concatenate([f(a.query.bias), f(a.key.bias), f(a.value.bias)])
            out[f"{tag}/layers/{i}/Wo"] = f(o.dense.weight).T
            out[f"{tag}/layers/{i}/bo"] = f(o.dense.bias)
            out[f"{tag}/layers/{i}/ln1_g"] = f(o.LayerNorm.weight)
            out[f"{tag}/layers/{i}/ln1_b"] = f(o.LayerNorm.bias)
            out[f"{tag}/layers/{i}/W1"] = f(l.intermediate.dense.weight).T
            out[f"{tag}/layers/{i}/b1"] = f(l.intermediate.dense.bias)
            out[f"{tag}/layers/{i}/W2"] = f(l.output.dense.weight).T
            out[f"{tag}/layers/{i}/b2"] = f(l.output.dense.bias)
            out[f"{tag}/layers/{i}/ln2_g"] = f(l.output.LayerNorm.weight)
            out[f"{tag}/layers/{i}/ln2_b"] = f(l.output.LayerNorm.bias)
    np.savez_compressed(os.path.join(HERE, "roberta_hf_torch.npz"), **{k: np.asarray(v) for k, v in out.items()})
    print("wrote roberta_hf_torch.npz:", len(out), "arrays, loss", loss.item())


if __name__ == "__main__":
    main()
