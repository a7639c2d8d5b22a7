"""Masked-LM training on the device: the position gather / scatter, the vocabulary cross-entropy with its in-place
gradient, the tcgen05 GEMM at vocabulary widths (N not a multiple of 8), the tied head against HF torch
BertForMaskedLM / RobertaForMaskedLM, graph replay, and HF checkpoint import / export."""
import ctypes as C
import json

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BF16_EPS = 2.0 ** -8
_KEEP = []


@pytest.fixture(scope="module")
def dev():
    from polus_b200 import device
    device.init(0)
    return device


@pytest.fixture(autouse=True)
def _keepalive():
    yield
    _KEEP.clear()


def T(arr, dtype=None):
    from polus_b200.tensor import Tensor
    t = Tensor.from_numpy(arr, dtype)
    _KEEP.append(t)
    return t


def new(shape, dtype):
    from polus_b200.tensor import Tensor
    t = Tensor(shape, dtype, zero=True)
    _KEEP.append(t)
    return t


def call(name, *a):
    from polus_b200 import _lib
    return _lib.call(name, *a)


def st():
    from polus_b200 import device
    return device.stream()


def _xent_ref(x, y, w):
    """fp64 loss, per-row nll and gradient of sum_r w_r nll_r / sum w over float logits x [R,V]."""
    x = x.astype(np.float64)
    m = x.max(1, keepdims=True)
    lse = (m + np.log(np.exp(x - m).sum(1, keepdims=True)))[:, 0]
    nll = lse - x[np.arange(len(y)), y]
    W = w.astype(np.float64).sum()
    loss = float((w * nll).sum() / W) if W > 0 else 0.0
    g = np.exp(x - lse[:, None])
    g[np.arange(len(y)), y] -= 1.0
    g *= (w / W if W > 0 else 0.0 * w)[:, None]
    return loss, nll, g


CASES = [(V, R) for V in (1, 7, 997, 28996, 30522) for R in (1, 3, 10240)] + [(V, R) for V in (50265, 250002) for R in (1, 3, 160)]


@pytest.mark.parametrize("V,R", CASES)
def test_vocab_xent_matches_fp64(dev, V, R):
    """Loss rel 1e-5, gradient within bf16 rounding of the fp64 value, argmax bit-exact (ties included), ldl > V,
    zero and fractional weights; the same logits with labels NULL give the same argmax and stay untouched.  R = 10240 is
    the B = 256, P = 40 batch; at V >= 50265 the host reference limits R to 160 rows."""
    from polus_b200.tensor import BF16, F32, I32
    rng = np.random.default_rng(V * 7 + R)
    ldl = (V + 7) // 8 * 8 + 8
    x = dev.bf16_round((rng.standard_normal((R, V)) * 3).astype(np.float32))
    if V > 1:
        top = rng.integers(0, V, R)
        x[np.arange(R), top] = 20.0
        dup = np.minimum(top + rng.integers(1, 4, R), V - 1)           # a tie at a higher index: the lower one wins
        x[np.arange(R), dup] = np.where(dup != top, 20.0, x[np.arange(R), dup])
    y = rng.integers(0, V, R).astype(np.int32)
    w = rng.choice(np.array([0.0, 1.0, 0.25, 2.0], np.float32), R)
    if R > 1:
        w[0] = 1.0
    buf = np.full((R, ldl), 7.0, np.float32)
    buf[:, :V] = x
    for weights in (w, np.zeros(R, np.float32)):
        lg = T(buf, BF16)
        nll, amax, loss = new((R,), F32), new((R,), I32), new((), F32)
        call("polus_vocab_xent", lg.ptr, R, V, ldl, T(y, I32).ptr, T(weights, F32).ptr, nll.ptr, amax.ptr, loss.ptr, st())
        loss_r, nll_r, g_r = _xent_ref(x, y, weights)
        got = lg.numpy()
        np.testing.assert_array_equal(amax.numpy(), np.argmax(x, 1))
        np.testing.assert_array_equal(got[:, V:], 7.0)                 # the padding columns are not written
        if weights.any():
            assert abs(float(loss) - loss_r) <= 1e-5 * abs(loss_r), (float(loss), loss_r)
            np.testing.assert_allclose(nll.numpy(), nll_r, rtol=1e-5, atol=1e-5)
            scale = (weights / weights.sum())[:, None]
            assert np.all(np.abs(got[:, :V] - g_r) <= BF16_EPS * np.abs(g_r) + 1e-6 * scale + 1e-30)
        else:
            assert float(loss) == 0.0 and not got[:, :V].any()
    lg = T(buf, BF16)
    amax = new((R,), I32)
    call("polus_vocab_xent", lg.ptr, R, V, ldl, None, None, None, amax.ptr, None, st())
    np.testing.assert_array_equal(amax.numpy(), np.argmax(x, 1))
    np.testing.assert_array_equal(lg.numpy(), dev.bf16_round(buf))


@pytest.mark.parametrize("V", [50265, 250002])
def test_vocab_xent_full_batch_large_vocabulary(dev, V):
    """R = 10240 rows (69 waves of one row per SM) at the large vocabularies: the host reference runs in 256-row chunks;
    every row's NLL and argmax and the loss are checked, the gradient on every 8th chunk."""
    from polus_b200.tensor import BF16, F32, I32, Tensor
    R, CH = 10240, 256
    ldl = (V + 7) // 8 * 8
    rng = np.random.default_rng(V)
    y = rng.integers(0, V, R).astype(np.int32)
    w = rng.choice(np.array([0.0, 1.0, 0.5], np.float32), R)
    lg = new((R, ldl), BF16)
    nll_r, amax_r, kept = np.zeros(R), np.zeros(R, np.int64), {}
    for c0 in range(0, R, CH):
        x = np.zeros((CH, ldl), np.float32)
        x[:, :V] = dev.bf16_round(np.random.default_rng((V, c0)).standard_normal((CH, V), dtype=np.float32) * 3)
        x[:, V:] = -1.0
        chunk = T(x, BF16)
        call("polus_memcpy_d2d", lg.ptr + c0 * ldl * 2, chunk.ptr, CH * ldl * 2, st())
        _KEEP.remove(chunk)
        xv = x[:, :V]
        amax_r[c0:c0 + CH] = np.argmax(xv, 1)
        _, nll_r[c0:c0 + CH], _ = _xent_ref(xv, y[c0:c0 + CH], np.ones(CH, np.float32))
        if (c0 // CH) % 8 == 0:
            kept[c0] = xv
    nll, amax, loss = new((R,), F32), new((R,), I32), new((), F32)
    call("polus_vocab_xent", lg.ptr, R, V, ldl, T(y, I32).ptr, T(w, F32).ptr, nll.ptr, amax.ptr, loss.ptr, st())
    np.testing.assert_array_equal(amax.numpy(), amax_r)
    np.testing.assert_allclose(nll.numpy(), nll_r, rtol=1e-5, atol=1e-5)
    loss_r = float((w * nll_r).sum() / w.astype(np.float64).sum())
    assert abs(float(loss) - loss_r) <= 1e-5 * abs(loss_r), (float(loss), loss_r)
    for c0, xv in kept.items():
        got = Tensor((CH, ldl), BF16, ptr=lg.ptr + c0 * ldl * 2, block=lg.block).numpy()[:, :V]
        _, _, g_r = _xent_ref(xv, y[c0:c0 + CH], w[c0:c0 + CH])   # normalised by the chunk's sum of weights
        W, Wc = w.astype(np.float64).sum(), w[c0:c0 + CH].astype(np.float64).sum()
        g_r = g_r * (Wc / W) if Wc > 0 else g_r
        scale = (w[c0:c0 + CH] / W)[:, None]
        assert np.all(np.abs(got - g_r) <= BF16_EPS * np.abs(g_r) + 1e-6 * scale + 1e-30), c0


@pytest.mark.parametrize("H,B,S,P", [(768, 64, 128, 20), (16, 3, 5, 7), (1024, 8, 512, 80)])
def test_gather_scatter_positions_bit_exact(dev, H, B, S, P):
    from polus_b200.tensor import BF16, I32
    rng = np.random.default_rng(H + P)
    h = dev.bf16_round(rng.standard_normal((B, S, H)).astype(np.float32))
    pos = rng.integers(0, S, (B, P)).astype(np.int32)
    pos[0, :] = 0                                                     # padding slots all at position 0
    pos[1, 1:4] = pos[1, 0]                                           # a repeated position
    pos[-1, -1], pos[-1, 0] = S + 3, -2                               # clamped
    cl = np.clip(pos, 0, S - 1)
    out = new((B * P, H), BF16)
    pos_t = T(pos, I32)
    call("polus_gather_positions", T(h, BF16).ptr, pos_t.ptr, B, S, H, P, out.ptr, st())
    np.testing.assert_array_equal(out.numpy(), h[np.arange(B)[:, None], cl].reshape(B * P, H))
    g = dev.bf16_round(rng.standard_normal((B * P, H)).astype(np.float32)).reshape(B, P, H)
    dh = new((B, S, H), BF16)
    call("polus_scatter_positions_add", T(g.reshape(B * P, H), BF16).ptr, pos_t.ptr, B, S, H, P, dh.ptr, st())
    ref = np.zeros((B, S, H), np.float32)
    for b in range(B):
        for s in np.unique(cl[b]):
            acc = np.zeros(H, np.float32)
            for j in np.nonzero(cl[b] == s)[0]:
                acc = acc + g[b, j]
            ref[b, s] = acc
    np.testing.assert_array_equal(dh.numpy(), dev.bf16_round(ref))


@pytest.mark.parametrize("N", [30522, 50265, 250002, 997])
def test_gemm_vocabulary_width(dev, N):
    """Logits GEMM (K-major B, bf16 C with 16-byte rows, with and without bias) and the dgrad with K = V, against
    polus_gemm_small."""
    from polus_b200 import _lib
    from polus_b200.tensor import BF16, F32
    rng = np.random.default_rng(N)
    M, H = 320, 768
    ldc = (N + 7) // 8 * 8
    A = dev.bf16_round(rng.standard_normal((M, H)).astype(np.float32))
    W = dev.bf16_round((rng.standard_normal((N, H)) * 0.05).astype(np.float32))
    bias = rng.standard_normal(N).astype(np.float32)
    a_t, w_t, b_t = T(A, BF16), T(W, BF16), T(bias)
    for with_bias in (False, True):
        pad = np.full((M, ldc), 3.0, np.float32)
        c_t, r_t = T(pad, BF16), new((M, N), F32)
        g = _lib.Gemm()
        g.M, g.N, g.K, g.batch0, g.batch1 = M, N, H, 1, 1
        g.A = _lib.Operand(a_t.ptr, H, 0, 0, 0, _lib.BF16)
        g.B = _lib.Operand(w_t.ptr, H, 0, 0, 0, _lib.BF16)
        g.C, g.ldc, g.c_dtype, g.bias, g.alpha, g.act = c_t.ptr, ldc, _lib.BF16, b_t.ptr if with_bias else None, 1.0, 0
        g.accumulate, g.split_k = 0, 1
        assert call("polus_gemm_tc_supported", C.byref(g)) == 1
        call("polus_gemm_tc", C.byref(g), st())
        g.C, g.ldc, g.c_dtype = r_t.ptr, N, _lib.F32
        call("polus_gemm_small", C.byref(g), st())
        got, ref = c_t.numpy(), r_t.numpy()
        np.testing.assert_allclose(got[:, :N], ref, atol=2 * BF16_EPS * (np.abs(ref).max() + 1), rtol=0)
    # dgrad: dx[M,H] = G[M,N] . W[N,H], K = N; G rows of stride ldc whose padding columns hold garbage
    G = np.full((M, ldc), 1e4, np.float32)
    G[:, :N] = dev.bf16_round((rng.standard_normal((M, N)) * 0.01).astype(np.float32))
    g_t, dx_t, dr_t = T(G, BF16), new((M, H), BF16), new((M, H), F32)
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = M, H, N, 1, 1
    g.A = _lib.Operand(g_t.ptr, ldc, 0, 0, 0, _lib.BF16)
    g.B = _lib.Operand(w_t.ptr, H, 0, 0, 1, _lib.BF16)
    g.C, g.ldc, g.c_dtype, g.bias, g.alpha, g.act, g.accumulate, g.split_k = dx_t.ptr, H, _lib.BF16, None, 1.0, 0, 0, 1
    call("polus_gemm_tc", C.byref(g), st())
    host = G[:, :N].astype(np.float64) @ W.astype(np.float64)
    np.testing.assert_allclose(dx_t.numpy(), host, atol=2 * BF16_EPS * (np.abs(host).max() + 1), rtol=0)


def test_colsum_bf16_strided(dev):
    from polus_b200.tensor import BF16, F32
    rng = np.random.default_rng(3)
    R, N, ld = 10240, 30522, 30528
    x = dev.bf16_round(rng.standard_normal((R, ld)).astype(np.float32))
    out = T(np.full(N, 0.5, np.float32))
    call("polus_colsum_bf16", T(x, BF16).ptr, R, N, ld, out.ptr, st())
    ref = 0.5 + x[:, :N].astype(np.float64).sum(0)
    np.testing.assert_allclose(out.numpy(), ref, rtol=1e-4, atol=1e-3)


# ------------------------------------------------------------------------------------------------ model level
def _config(family, V, H, L, nh, I, S, **kw):
    from polus_b200.nn import BertConfig
    base = dict(vocab_size=V, hidden_size=H, num_hidden_layers=L, num_attention_heads=nh, intermediate_size=I,
                hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    if family == "roberta":
        base.update(model_type="roberta", pad_token_id=1, type_vocab_size=1, layer_norm_eps=1e-5, max_position_embeddings=S + 2)
    else:
        base.update(max_position_embeddings=max(S, 64))
    base.update(kw)
    return BertConfig(**base)


def _mlm_batch(rng, family, B, S, V, P):
    from polus_b200.mlm import mask_tokens
    pad = 1 if family == "roberta" else 0
    ids = rng.integers(4, V, (B, S)).astype(np.int32)
    lens = np.maximum(8, rng.integers(S // 2, S + 1, B))
    mask = (np.arange(S)[None, :] < lens[:, None]).astype(np.int32)
    ids[mask == 0] = pad
    ids, pos, lab, w = mask_tokens(ids, mask, vocab_size=V, mask_token_id=3, special_token_ids=(0, 1, 2, 3), max_predictions=P,
                                   rng=rng)
    x = {"input_ids": ids, "attention_mask": mask, "token_type_ids": np.zeros((B, S), np.int32), "masked_lm_positions": pos}
    return x, {"masked_lm_ids": lab, "masked_lm_weights": w}


def _build(family, V=997, H=128, L=2, nh=2, I=512, S=64, seed=5, **kw):
    from polus_b200 import ops, tensor
    from polus_b200.mlm import BertMaskedLMModel
    from polus_b200.utils import set_random_seed
    tensor.reset_arena()
    set_random_seed(seed)
    ops.set_step(0)
    return BertMaskedLMModel(_config(family, V, H, L, nh, I, S, **kw))


def _perturb(model, rng):
    from tests.parity import round_weights_to_bf16
    for w in model.weights:
        if w.name.endswith("gamma"):
            w.assign(1.0 + 0.1 * rng.standard_normal(w.shape))
        elif w.name.endswith(("beta", "bias")):
            w.assign(0.02 * rng.standard_normal(w.shape))
    round_weights_to_bf16(model)


def _hf_grads(model):
    """Our gradients in HF layout: assign them as values, export, restore."""
    from polus_b200.pretrained import export_hf_bert_weights
    vals = [w.numpy() for w in model.weights]
    for w in model.weights:
        w.assign(w.grad.numpy())
    out = export_hf_bert_weights(model)
    for w, v in zip(model.weights, vals):
        w.assign(v)
    return out


def _torch_mlm(family, model):
    import torch
    import transformers as tf
    from polus_b200.pretrained import export_hf_bert_weights
    c = model.config
    kw = dict(vocab_size=c.vocab_size, hidden_size=c.hidden_size, num_hidden_layers=c.num_hidden_layers,
              num_attention_heads=c.num_attention_heads, intermediate_size=c.intermediate_size, hidden_act="gelu",
              hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, max_position_embeddings=c.max_position_embeddings,
              type_vocab_size=c.type_vocab_size, layer_norm_eps=c.layer_norm_eps, pad_token_id=c.pad_token_id)
    if family == "roberta":
        net = tf.RobertaForMaskedLM(tf.RobertaConfig(**kw, attn_implementation="eager"))
        prefix = "roberta."
    else:
        net = tf.BertForMaskedLM(tf.BertConfig(**kw, attn_implementation="eager"))
        prefix = "bert."
    state = {(k if k.startswith(("cls.", "lm_head.")) else prefix + k): torch.from_numpy(np.ascontiguousarray(v))
             for k, v in export_hf_bert_weights(model).items()}
    missing, unexpected = net.load_state_dict(state, strict=False)
    assert not unexpected and all("decoder" in k or "position_ids" in k for k in missing), (missing, unexpected)
    net.train()
    return net, prefix


def _compare_with_torch(family, model, x, y, logit_tol=2e-2):
    import torch
    from polus_b200 import ops
    net, prefix = _torch_mlm(family, model)
    with ops.GradientTape() as tape:
        logits = model(**x, training=True)
        lg = logits.numpy()
        loss = model.loss(y, logits)
    tape.gradient(loss, model.trainable_weights)
    loss_dev = float(loss)
    g_dev = _hf_grads(model)
    B, S = x["input_ids"].shape
    labels = np.full((B, S), -100, np.int64)
    sel = y["masked_lm_weights"] > 0
    rows = np.nonzero(sel)[0]
    labels[rows, x["masked_lm_positions"][sel]] = y["masked_lm_ids"][sel]
    ti = torch.from_numpy(x["input_ids"].astype(np.int64))
    out = net(input_ids=ti, attention_mask=torch.from_numpy(x["attention_mask"].astype(np.int64)),
              token_type_ids=torch.from_numpy(x["token_type_ids"].astype(np.int64)), labels=torch.from_numpy(labels))
    out.loss.backward()
    ref_logits = out.logits.detach().numpy()[np.arange(B)[:, None], x["masked_lm_positions"]].reshape(lg.shape)
    scale = float(np.abs(ref_logits).max())
    np.testing.assert_allclose(lg, ref_logits, atol=logit_tol * scale, rtol=logit_tol)
    loss_ref = float(out.loss)
    assert abs(loss_dev - loss_ref) / abs(loss_ref) < 1e-2, (loss_dev, loss_ref)
    worst = (1.0, None)
    named = dict(net.named_parameters())
    for k, gd in g_dev.items():
        if k.endswith("attention.self.key.bias"):
            continue   # zero in exact arithmetic (softmax over keys ignores a per-query shift): both sides are noise
        p = named[k if k.startswith(("cls.", "lm_head.")) else prefix + k]
        if p.grad is None:
            continue
        gr = p.grad.numpy()
        denom = np.linalg.norm(gr) * np.linalg.norm(gd)
        cos = float((gr * gd).sum() / denom) if denom > 0 else 1.0
        if cos < worst[0]:
            worst = (cos, k)
    assert worst[0] >= 0.999, worst
    return net


@pytest.mark.parametrize("family", ["bert", "roberta"])
def test_small_mlm_matches_hf_torch(dev, family):
    rng = np.random.default_rng(1)
    model = _build(family)
    x, y = _mlm_batch(rng, family, 4, 64, 997, 12)
    _perturb(model, rng)
    net = _compare_with_torch(family, model, x, y)
    # inference against HF torch's argmax, on the rows whose top two logits are clearly apart
    import torch
    from polus_b200 import ops
    pred = model.inference(x).numpy()
    with torch.no_grad():
        ref = net(**{k: torch.from_numpy(x[k].astype(np.int64)) for k in ("input_ids", "attention_mask", "token_type_ids")}
                  ).logits.numpy()[np.arange(4)[:, None], x["masked_lm_positions"]]
    top2 = np.sort(ref, -1)[..., -2:]
    clear = top2[..., 1] - top2[..., 0] > 0.05 * np.abs(ref).max()
    assert clear.sum() >= 10
    np.testing.assert_array_equal(pred[clear], np.argmax(ref, -1)[clear])
    # the padded-row logits are refused by generic ops (V = 997: rows of 1000)
    logits = model(**x)
    with pytest.raises(ValueError):
        ops.argmax(logits)
    with pytest.raises(ValueError):
        ops.reshape(logits, (-1,))
    with pytest.raises(ValueError):
        model.inference(x["input_ids"])


@pytest.mark.parametrize("family,V,S,P", [("bert", 30522, 128, 20), ("roberta", 50265, 128, 20)])
def test_full_size_mlm_matches_hf_torch(dev, family, V, S, P):
    """BERT-base / RoBERTa-base dims against HF torch fp32 with the same weights: test_fullsize_gpu's bars, the tied word
    embeddings included; then three Adam steps against torch.optim.Adam (Keras epsilon placement differs: eps 1e-8 on
    both sides makes it immaterial), loss rel 1e-2."""
    import torch
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    rng = np.random.default_rng(2)
    model = _build(family, V=V, H=768, L=12, nh=12, I=3072, S=S, seed=3)
    x, y = _mlm_batch(rng, family, 4, S, V, P)
    _perturb(model, rng)
    net = _compare_with_torch(family, model, x, y)
    from polus_b200 import _lib, device
    for w in model.weights:
        _lib.call("polus_memset", w.grad.ptr, 0, w.grad.nbytes, device.stream())
    net.zero_grad()
    opt_t = torch.optim.Adam([p for p in net.parameters() if p.requires_grad], lr=1e-4, eps=1e-8)
    trainer = ClassifierTrainer(model, Adam(1e-4, epsilon=1e-8), model.loss)
    B, Sx = x["input_ids"].shape
    labels = np.full((B, Sx), -100, np.int64)
    sel = y["masked_lm_weights"] > 0
    labels[np.nonzero(sel)[0], x["masked_lm_positions"][sel]] = y["masked_lm_ids"][sel]
    targs = dict(input_ids=torch.from_numpy(x["input_ids"].astype(np.int64)),
                 attention_mask=torch.from_numpy(x["attention_mask"].astype(np.int64)),
                 token_type_ids=torch.from_numpy(x["token_type_ids"].astype(np.int64)), labels=torch.from_numpy(labels))
    for _ in range(3):
        ld = float(trainer.train_step(x, y))
        opt_t.zero_grad()
        out = net(**targs)
        out.loss.backward()
        opt_t.step()
        assert abs(ld - float(out.loss)) / abs(float(out.loss)) < 1e-2, (ld, float(out.loss))


def test_mlm_graph_replay_equals_eager_and_trains(dev, monkeypatch):
    """lr = 0 and dropout on: Adam's first moment after 4 steps agrees between op-by-op execution and graph replay;
    then with lr > 0 the loss falls on a fixed batch and inference equals the argmax of the head's logits."""
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer

    def run(eager):
        monkeypatch.setenv("POLUS_EAGER", "1" if eager else "0")
        model = _build("bert", hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, S=128, H=256, nh=4, I=1024)
        x, y = _mlm_batch(np.random.default_rng(0), "bert", 8, 128, 997, 20)
        opt = Adam(0.0)
        tr = ClassifierTrainer(model, opt, model.loss)
        losses = [float(tr.train_step(x, y)) for _ in range(4)]
        return losses, opt.variables()[0].numpy()
    le, me = run(True)
    lg, mg = run(False)
    np.testing.assert_allclose(lg, le, rtol=1e-5)
    scale = np.abs(me).max()
    assert scale > 0
    assert np.abs(mg - me).max() <= 2e-4 * scale, (np.abs(mg - me).max(), scale)

    monkeypatch.setenv("POLUS_EAGER", "0")
    model = _build("roberta")
    x, y = _mlm_batch(np.random.default_rng(4), "roberta", 8, 64, 997, 12)
    tr = ClassifierTrainer(model, Adam(1e-3), model.loss)
    losses = [float(tr.train_step(x, y)) for _ in range(8)]
    assert np.isfinite(losses).all() and losses[-1] < losses[0] - 0.5, losses
    pred = model.inference(x).numpy()
    logits = model(**x, training=False).numpy()
    np.testing.assert_array_equal(pred, np.argmax(logits, 1).reshape(pred.shape))
    acc = model.last_predictions.numpy()
    assert acc.shape == (8 * 12,)


# ------------------------------------------------------------------------------------------------ checkpoints
@pytest.mark.parametrize("family", ["bert", "roberta"])
def test_checkpoint_import_export_and_hf_round_trip(dev, family, tmp_path):
    import torch
    import transformers as tf
    from polus_b200 import pretrained
    from polus_b200.models import BertModel, bert_model_from_checkpoint
    from polus_b200.ner.models import BertNERModel
    rng = np.random.default_rng(9)
    model = _build(family)
    _perturb(model, rng)
    snap = tmp_path / "snap"
    pretrained.save_hf_checkpoint(model, str(snap))
    cfg = json.loads((snap / "config.json").read_text())
    assert cfg["model_type"] == model.config.model_type and cfg["pad_token_id"] == model.config.pad_token_id
    hf_cls = tf.RobertaForMaskedLM if family == "roberta" else tf.BertForMaskedLM
    net = hf_cls.from_pretrained(str(snap))
    exported = pretrained.export_hf_bert_weights(model)
    prefix = "roberta." if family == "roberta" else "bert."
    hf_state = net.state_dict()
    for k, v in exported.items():
        key = k if k.startswith(("cls.", "lm_head.")) else prefix + k
        assert torch.equal(hf_state[key], torch.from_numpy(v)), key
    dec = "lm_head.decoder.weight" if family == "roberta" else "cls.predictions.decoder.weight"
    assert torch.equal(hf_state[dec], torch.from_numpy(exported["embeddings.word_embeddings.weight"]))

    # import: HF's own save (no decoder.* tensors) into a fresh model reproduces every tensor
    hf_dir = tmp_path / "hf"
    net.save_pretrained(str(hf_dir))
    from safetensors.numpy import load_file
    saved = load_file(str(hf_dir / "model.safetensors"))
    other = _build(family, seed=77)
    assert pretrained.load_hf_bert_weights(other, saved) == []
    for k, v in pretrained.export_hf_bert_weights(other).items():
        np.testing.assert_array_equal(v, exported[k])
    # a tied decoder.weight is accepted, an untied one raises
    word = saved[prefix + "embeddings.word_embeddings.weight"]
    pretrained.load_hf_bert_weights(other, dict(saved, **{dec: word}))
    with pytest.raises(ValueError, match="untied"):
        pretrained.load_hf_bert_weights(other, dict(saved, **{dec: word + 1.0}))
    # a checkpoint without a head: strict raises, strict=False keeps the MLM model's head as initialised
    no_head = {k: v for k, v in saved.items() if not k.startswith(("cls.", "lm_head."))}
    with pytest.raises(KeyError):
        pretrained.load_hf_bert_weights(other, no_head)
    bias_before = other.cls.bias.numpy()
    other.cls.bias.assign(bias_before + 1.0)
    assert pretrained.load_hf_bert_weights(other, no_head, strict=False) == []
    np.testing.assert_array_equal(other.cls.bias.numpy(), bias_before + 1.0)
    # an encoder-only model leaves the head unused, as before
    enc = BertModel(model.config, add_pooling_layer=False)
    unused = pretrained.load_hf_bert_weights(enc, saved)
    assert unused and all(k.startswith(("cls.", "lm_head.")) for k in unused)

    # the saved directory as the encoder of an NER model: same encoder outputs
    x, _ = _mlm_batch(rng, family, 3, 64, 997, 8)
    feed = {k: x[k] for k in ("input_ids", "attention_mask", "token_type_ids")}
    h_mlm = model.bert(**feed)["last_hidden_state"].numpy()
    loaded = bert_model_from_checkpoint(str(snap))
    assert np.array_equal(loaded(**feed)["last_hidden_state"].numpy(), h_mlm)
    ner = BertNERModel(loaded.config, output_classes=4)
    pretrained.load_hf_bert_weights(ner.bert, str(snap / "model.safetensors"))
    assert np.array_equal(ner.bert(**feed)["last_hidden_state"].numpy(), h_mlm)


def test_save_load_model_round_trip(dev, tmp_path):
    from polus_b200 import mlm
    from polus_b200.models import load_model
    from polus_b200.tensor import reset_arena
    reset_arena()
    model = mlm.bert_mlm(model=dict(vocab_size=997, hidden_size=64, num_hidden_layers=1, num_attention_heads=2,
                                    intermediate_size=128, max_position_embeddings=64))
    ws = model.get_weights()
    assert [w.shape for w in ws[-5:]] == [(64, 64), (64,), (64,), (64,), (997,)]
    model.save(str(tmp_path))
    back = load_model(str(tmp_path / "bert_mlm.cfg"), external_module=mlm)
    for a, b in zip(back.get_weights(), ws):
        np.testing.assert_array_equal(a, b)
