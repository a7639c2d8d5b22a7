"""RoBERTa-family pieces of the CPU references -- TEST INFRASTRUCTURE ONLY.

The encoder layers, LayerNorm, NER head and CRF are oracle/numpy_ref.py's; what RoBERTa adds is its position ids and an
embedding block that reads one position row per token.  Pinned against HF torch RobertaEmbeddings + RobertaLayer by
tests/golden/roberta_hf_torch.npz (generator tests/golden/make_roberta_golden.py, check tests/test_roberta_cpu.py).
"""
import numpy as np

from oracle import numpy_ref as R


def roberta_position_ids(ids, pad):
    """HF RobertaEmbeddings.create_position_ids_from_input_ids: pad + cumsum(ids != pad) * (ids != pad)."""
    mask = (np.asarray(ids) != pad).astype(np.int64)
    return np.cumsum(mask, axis=1) * mask + pad


def embeddings_fwd(ids, tt, p, pos_ids, drop_mask=None, eps=1e-5):
    """TFRobertaEmbeddings: LN(word[ids] + pos[pos_ids] + type[tt]) then dropout (same sum order as the BERT oracle)."""
    z = p["word"][ids] + p["pos"][pos_ids] + p["type"][tt]
    y, c = R.layer_norm(z, p["emb_ln_g"], p["emb_ln_b"], eps)
    if drop_mask is not None:
        y = y * drop_mask
    return y, dict(ids=ids, tt=tt, pos_ids=pos_ids, ln=c, drop_mask=drop_mask)


def embeddings_bwd(dy, c, p):
    """Gradients of every table row a token read, as TF's embedding lookup gives them: the padding rows collect the
    gradients of pad tokens (torch's nn.Embedding(padding_idx=...) would zero them)."""
    if c["drop_mask"] is not None:
        dy = dy * c["drop_mask"]
    dz, gg, gb = R.layer_norm_bwd(dy, c["ln"], p["emb_ln_g"])
    H = dz.shape[-1]
    g = {"emb_ln_g": gg, "emb_ln_b": gb}
    for name, index in (("word", c["ids"]), ("pos", c["pos_ids"]), ("type", c["tt"])):
        g[name] = np.zeros_like(p[name])
        np.add.at(g[name], np.asarray(index).reshape(-1), dz.reshape(-1, H))
    return g


def ner_loss_and_grads(params, ids, mask, tt, tags, nh, pad, eps=1e-5):
    """oracle/ner_model.loss_and_grads for a RoBERTa-family encoder (derived position ids, LayerNorm epsilon)."""
    h, ec = embeddings_fwd(ids, tt, params["emb"], roberta_position_ids(ids, pad), eps=eps)
    add = R.attention_mask_additive(mask).astype(np.float64)
    caches = []
    for lp in params["layers"]:
        h, c = R.bert_layer_fwd(h, add, lp, nh, eps=eps)
        caches.append(c)
    e, hc = R.ner_head_fwd(h, params["head"], "swish")
    B, S, _ = e.shape
    _, loss, ge, gtrans = R.crf_nll_with_grads(e, tags, np.full(B, S), params["trans"])
    dh, ghead = R.ner_head_bwd(ge, hc, params["head"])
    glayers = []
    for lp, lc in zip(reversed(params["layers"]), reversed(caches)):
        dh, g = R.bert_layer_bwd(dh, lc, lp)
        glayers.append(g)
    glayers.reverse()
    return loss, e, dict(emb=embeddings_bwd(dh, ec, params["emb"]), layers=glayers, head=ghead, trans=gtrans)


def build_torch_roberta(vocab, max_pos, pad, hidden=768, heads=12, **kw):
    """oracle/torch_ref.build's fp32 NER+CRF network with HF RobertaEmbeddings (one token type, position ids from
    input_ids and pad) and LayerNorm epsilon 1e-5.  RobertaLayer is BertLayer, so the encoder layers are kept.
    padding_idx is removed from the embedding modules: the padding rows get the pad tokens' gradients, as under TF."""
    import torch
    from transformers import RobertaConfig
    from transformers.models.roberta.modeling_roberta import RobertaEmbeddings
    from oracle import torch_ref
    net = torch_ref.build(hidden=hidden, heads=heads, vocab=vocab, max_pos=max_pos, **kw)
    cfg = RobertaConfig(vocab_size=vocab, hidden_size=hidden, num_attention_heads=heads, max_position_embeddings=max_pos,
                        type_vocab_size=1, layer_norm_eps=1e-5, pad_token_id=pad, hidden_dropout_prob=kw.get("dropout", 0.1))
    net.emb = RobertaEmbeddings(cfg)
    net.emb.word_embeddings.padding_idx = None
    net.emb.position_embeddings.padding_idx = None
    for m in net.layers.modules():
        if isinstance(m, torch.nn.LayerNorm):
            m.eps = 1e-5
    return net
