"""fp64 numpy reference of the masked-LM head and loss (HF BertForMaskedLM / RobertaForMaskedLM at TF BERT's
masked_lm_positions), on top of the oracle's GELU and LayerNorm; pinned to HF torch by tests/golden/mlm_hf_torch.npz
(tests/test_mlm_cpu.py).  Weights in the Keras layout of polus_b200.nn.BertLMPredictionHead: W_dense [H, H] (in, out),
word [V, H] (the tied embedding table)."""
import numpy as np

from oracle import numpy_ref as R


def head_fwd(h, pos, p, eps):
    """h [B,S,H] -> logits [B*P, V] at the masked positions, and the cache for head_bwd."""
    Bsz, _, H = h.shape
    sel = h[np.arange(Bsz)[:, None], pos].reshape(-1, H)
    z = sel @ p["W_dense"] + p["b_dense"]
    a = R.gelu(z)
    t, ln_cache = R.layer_norm(a, p["ln_g"], p["ln_b"], eps)
    logits = t @ p["word"].T + p["bias"]
    return logits, (sel, z, t, ln_cache)


def loss_fwd(logits, lab, w):
    """sum_r w_r (lse_r - x_r[y_r]) / sum_r w_r (0 when every weight is 0) and d loss / d logits."""
    lab, w = lab.reshape(-1), w.reshape(-1).astype(np.float64)
    m = logits.max(-1, keepdims=True)
    lse = (m + np.log(np.exp(logits - m).sum(-1, keepdims=True)))[:, 0]
    nll = lse - logits[np.arange(len(lab)), lab]
    W = w.sum()
    if W == 0:
        return 0.0, np.zeros_like(logits)
    g = np.exp(logits - lse[:, None])
    g[np.arange(len(lab)), lab] -= 1.0
    return float((w * nll).sum() / W), g * (w / W)[:, None]


def head_bwd(dlogits, cache, p, h_shape, pos):
    """Gradients of the head's parameters, of the tied table (the decoder's part) and of h."""
    sel, z, t, ln_cache = cache
    g = {"bias": dlogits.sum(0), "word": dlogits.T @ t}
    dt = dlogits @ p["word"]
    da, g["ln_g"], g["ln_b"] = R.layer_norm_bwd(dt, ln_cache, p["ln_g"])
    dz = da * R.gelu_grad(z)
    g["W_dense"], g["b_dense"] = sel.T @ dz, dz.sum(0)
    dsel = dz @ p["W_dense"].T
    Bsz, S, H = h_shape
    dh = np.zeros(h_shape)
    P = pos.shape[1]
    np.add.at(dh, (np.repeat(np.arange(Bsz), P), pos.reshape(-1)), dsel)
    g["h"] = dh
    return g
