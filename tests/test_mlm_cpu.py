"""Masked-LM pieces that need no GPU: host masking (polus_b200.mlm.mask_tokens), the argument checks of the new entry
points (made before any CUDA call), and which vocabulary GEMMs polus_gemm_tc accepts."""
import ctypes as C

import numpy as np
import pytest

SPECIAL = (0, 101, 102, 103)   # [PAD], [CLS], [SEP], [MASK] of the BERT vocabulary
MASK_ID, V = 103, 30522


def _batch(rng, B, S):
    ids = rng.integers(1000, V, (B, S)).astype(np.int32)
    lens = rng.integers(0, S + 1, B)
    mask = (np.arange(S)[None, :] < lens[:, None]).astype(np.int32)
    ids[:, 0] = 101
    ids[np.arange(B), np.maximum(lens - 1, 0)] = 102
    ids[mask == 0] = 0
    return ids, mask


def _mask(ids, mask, P, seed, p=0.15):
    from polus_b200.mlm import mask_tokens
    return mask_tokens(ids, mask, vocab_size=V, mask_token_id=MASK_ID, special_token_ids=SPECIAL, max_predictions=P,
                       mlm_probability=p, rng=np.random.default_rng(seed))


def test_mask_tokens_rules():
    rng = np.random.default_rng(0)
    B, S, P = 64, 128, 20
    ids, mask = _batch(rng, B, S)
    out, pos, lab, w = _mask(ids, mask, P, 1)
    assert out.shape == ids.shape and pos.shape == lab.shape == w.shape == (B, P)
    assert pos.dtype == lab.dtype == np.int32 and w.dtype == np.float32
    cand = (mask != 0) & ~np.isin(ids, SPECIAL)
    n_cand = cand.sum(1)
    n_expect = np.where(n_cand == 0, 0, np.minimum(P, np.maximum(1, np.rint(0.15 * n_cand))))
    for b in range(B):
        n = int(w[b].sum())
        assert n == n_expect[b]
        assert np.all(w[b, :n] == 1) and np.all(w[b, n:] == 0)
        sel = pos[b, :n]
        assert np.all(np.diff(sel) > 0)                                  # sorted, without replacement
        assert np.all(cand[b, sel])                                      # never special or pad tokens
        assert np.array_equal(lab[b, :n], ids[b, sel])
        assert np.all(pos[b, n:] == 0) and np.all(lab[b, n:] == 0)
        untouched = np.ones(S, bool)
        untouched[sel] = False
        assert np.array_equal(out[b, untouched], ids[b, untouched])
    capped = _mask(ids, mask, 3, 1)[3].sum(1)                            # max_predictions caps n
    assert np.all(capped == np.minimum(3, n_expect))


def test_mask_tokens_split_and_determinism():
    rng = np.random.default_rng(2)
    B, S, P = 2048, 128, 20
    ids, mask = _batch(rng, B, S)
    mask[:] = 1
    out, pos, lab, w = _mask(ids, mask, P, 7)
    sel = w > 0
    rows = np.nonzero(sel)[0]
    new = out[rows, pos[sel]]
    n = sel.sum()
    is_mask = new == MASK_ID
    kept = (new == lab[sel]) & ~is_mask
    # binomial bounds at 6 sigma; a random replacement equals the original with probability 1/V
    for frac, count in ((0.8, is_mask.sum()), (0.1 + 0.1 / V, kept.sum())):
        sd = np.sqrt(n * frac * (1 - frac))
        assert abs(count - n * frac) < 6 * sd, (frac, count, n)
    again = _mask(ids, mask, P, 7)
    for a, b in zip(again, (out, pos, lab, w)):
        assert np.array_equal(a, b)
    assert not np.array_equal(_mask(ids, mask, P, 8)[1], pos)


def test_mask_tokens_argument_errors():
    ids = np.zeros((2, 4), np.int32)
    with pytest.raises(ValueError):
        _mask(ids, np.zeros((2, 5), np.int32), 2, 0)
    with pytest.raises(ValueError):
        _mask(ids, np.ones((2, 4), np.int32), 0, 0)
    with pytest.raises(ValueError):
        _mask(ids, np.ones((2, 4), np.int32), 2, 0, p=0.0)
    out, pos, lab, w = _mask(ids, np.zeros((2, 4), np.int32), 3, 0)     # nothing to mask
    assert not w.any() and not pos.any() and np.array_equal(out, ids)


def test_entry_point_argument_errors():
    from polus_b200 import _lib
    fake = C.c_void_p(256)
    with pytest.raises(ValueError, match="H must be a positive multiple of 8"):
        _lib.call("polus_gather_positions", fake, fake, 2, 4, 12, 3, fake, None)
    with pytest.raises(ValueError, match="S must be >= 1"):
        _lib.call("polus_gather_positions", fake, fake, 2, 0, 16, 3, fake, None)
    with pytest.raises(ValueError, match="H must be a positive multiple of 8"):
        _lib.call("polus_scatter_positions_add", fake, fake, 2, 4, 0, 3, fake, None)
    with pytest.raises(ValueError, match="P must be <= 12288"):
        _lib.call("polus_scatter_positions_add", fake, fake, 2, 4, 16, 12289, fake, None)
    with pytest.raises(ValueError, match="B and P must be >= 0"):
        _lib.call("polus_scatter_positions_add", fake, fake, 2, 4, 16, -1, fake, None)
    with pytest.raises(ValueError, match="V must be >= 1"):
        _lib.call("polus_vocab_xent", fake, 4, 0, 8, fake, fake, fake, fake, fake, None)
    with pytest.raises(ValueError, match="ldl must be >= V and a multiple of 8"):
        _lib.call("polus_vocab_xent", fake, 4, 997, 997, fake, fake, fake, fake, fake, None)
    with pytest.raises(ValueError, match="ldl must be >= V"):
        _lib.call("polus_vocab_xent", fake, 4, 997, 992, fake, fake, fake, fake, fake, None)
    with pytest.raises(ValueError, match="labels need weights"):
        _lib.call("polus_vocab_xent", fake, 4, 997, 1000, fake, None, fake, fake, fake, None)
    with pytest.raises(ValueError, match="needs d_argmax"):
        _lib.call("polus_vocab_xent", fake, 4, 997, 1000, None, None, None, None, None, None)
    with pytest.raises(ValueError, match="ld must be >= N"):
        _lib.call("polus_colsum_bf16", fake, 4, 997, 996, fake, None)
    with pytest.raises(ValueError, match="need R >= 0 and N >= 1"):
        _lib.call("polus_colsum_bf16", fake, 4, 0, 8, fake, None)
    # accepted shapes with nothing to do return before any launch
    _lib.call("polus_gather_positions", fake, fake, 0, 4, 16, 3, fake, None)
    _lib.call("polus_colsum_bf16", fake, 0, 997, 1000, fake, None)
    assert _lib.call("polus_version") >= 103


def _gemm(N, **kw):
    from polus_b200 import _lib
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = 512, N, 768, 1, 1
    g.A = _lib.Operand(4096, 768, 0, 0, 0, _lib.BF16)
    g.B = _lib.Operand(8192, 768, 0, 0, kw.get("b_mn", 0), _lib.BF16)
    if kw.get("b_mn"):
        g.B.ld = (N + 7) // 8 * 8
    g.C, g.ldc, g.c_dtype = 16384, (N + 7) // 8 * 8, _lib.BF16
    g.bias = kw.get("bias")
    g.act = kw.get("act", 0)
    g.alpha, g.split_k = 1.0, 1
    g.colsum = kw.get("colsum")
    g.C2 = kw.get("c2")
    return _lib.call("polus_gemm_tc_supported", C.byref(g))


def test_gemm_accepts_vocabulary_widths():
    """N % 8 != 0 is taken for plain and bias-only problems with a K-major B; anything needing whole 8-column groups
    still goes elsewhere."""
    for N in (30522, 50265, 250002, 997, 1):
        assert _gemm(N) == 1 and _gemm(N, bias=32768) == 1, N
        assert _gemm(N, b_mn=1) == 0
        assert _gemm(N, act=1) == 0
        assert _gemm(N, colsum=32768) == 0
        assert _gemm(N, c2=65536, act=1) == 0
    assert _gemm(30528, b_mn=1) == 1 and _gemm(30528, act=1) == 1   # multiples of 8 keep every option


@pytest.mark.parametrize("family", ["bert", "roberta"])
def test_reference_head_matches_hf_torch_golden(family):
    """tests/mlm_ref.py against HF torch fp64 (tests/golden/mlm_hf_torch.npz): logits, loss and every gradient of the
    head, the tied decoder's part of the word-embedding gradient and d loss / d h, to the 1e-8 pin of the BERT oracle."""
    import os
    from tests import mlm_ref
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "mlm_hf_torch.npz"))
    g = lambda k: z[f"{family}/{k}"].astype(np.float64)
    p = {k: g(k) for k in ("W_dense", "b_dense", "ln_g", "ln_b", "bias", "word")}
    h, pos = g("h"), z[f"{family}/pos"].astype(np.int64)
    logits, cache = mlm_ref.head_fwd(h, pos, p, float(g("eps")))
    np.testing.assert_allclose(logits, g("logits"), rtol=1e-8, atol=1e-8)
    loss, dlogits = mlm_ref.loss_fwd(logits, z[f"{family}/lab"], z[f"{family}/w"])
    assert abs(loss - float(g("loss"))) <= 1e-8 * abs(float(g("loss")))
    grads = mlm_ref.head_bwd(dlogits, cache, p, h.shape, pos)
    for k in ("W_dense", "b_dense", "ln_g", "ln_b", "bias", "word", "h"):
        ref = g("g_" + k)
        np.testing.assert_allclose(grads[k], ref, rtol=1e-8, atol=1e-8 * (np.abs(ref).max() + 1e-30), err_msg=k)
    assert mlm_ref.loss_fwd(logits, z[f"{family}/lab"], np.zeros_like(z[f"{family}/w"]))[0] == 0.0
