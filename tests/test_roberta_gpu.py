"""RoBERTa-family encoders on the device: position ids derived from padding (polus_position_ids), the embedding block
with per-token position ids (polus_embed_ln_fwd_pos / polus_embed_ln_bwd_pos), checkpoint import of `roberta.`-prefixed
HuggingFace weights, and training of a RoBERTa-config NER+CRF model on the existing step.  References: the fp64 numpy
references (tests/roberta_ref.py on top of oracle/numpy_ref.py, pinned to HF torch RoBERTa by tests/test_roberta_cpu.py)
and, at full size, HF torch RobertaEmbeddings + RobertaLayer in fp32 (tests/roberta_ref.build_torch_roberta)."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
BF16_EPS = 2.0 ** -8
PAD = 1


@pytest.fixture(scope="module")
def dev():
    from polus_b200 import device
    device.init(0)
    return device


_KEEP = []


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


def padded_ids(rng, B, S, vocab, pad=PAD):
    """Rows cycling through: right-padded, left-padded, pad ids scattered mid-sequence, all pad, no pad."""
    ids = rng.integers(0, vocab, (B, S))
    ids[ids == pad] = pad + 1
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
    return ids.astype(np.int32)


@pytest.mark.parametrize("B", [1, 3, 256])
@pytest.mark.parametrize("S", [1, 7, 256, 512])
def test_position_ids_bit_exact(dev, B, S):
    from tests.roberta_ref import roberta_position_ids
    from polus_b200.tensor import I32
    rng = np.random.default_rng(B * 1000 + S)
    for pad in (1, 0):
        ids = padded_ids(rng, B, S, 50265, pad)
        out = new((B, S), I32)
        call("polus_position_ids", T(ids, I32).ptr, B, S, pad, out.ptr, st())
        np.testing.assert_array_equal(out.numpy(), roberta_position_ids(ids, pad))


@pytest.mark.parametrize("H", [64, 768, 1024, 2048])
@pytest.mark.parametrize("p", [0.0, 0.1])
def test_embedding_with_position_ids_fwd_bwd(dev, H, p):
    """Forward and backward against the fp64 oracle, every table row compared (the padding rows collect the pad tokens'
    gradients); dropout decisions equal those of polus_embed_ln_fwd at the same (seed, site, step)."""
    from oracle import philox
    from tests import roberta_ref as RR
    from polus_b200.tensor import BF16, F32, I32
    rng = np.random.default_rng(H)
    B, S, V = 24, 32, 300
    n_pos = S + PAD + 1
    P = {"word": rng.normal(0, 0.5, (V, H)).astype(np.float32), "pos": rng.normal(0, 0.5, (n_pos, H)).astype(np.float32),
         "type": rng.normal(0, 0.5, (1, H)).astype(np.float32), "emb_ln_g": (1 + 0.1 * rng.standard_normal(H)).astype(np.float32),
         "emb_ln_b": (0.1 * rng.standard_normal(H)).astype(np.float32)}
    ids = padded_ids(rng, B, S, V)
    pos_ids = RR.roberta_position_ids(ids, PAD).astype(np.int32)
    pos_ids[4, 0], pos_ids[4, 1] = n_pos + 7, -3          # out of range: clamped to the table, as token ids are
    pos_ref = np.clip(pos_ids, 0, n_pos - 1)
    tt = np.zeros((B, S), np.int32)
    seed, site, step = 77, 3, 9
    from polus_b200 import ops
    ops.set_step(step)
    sp = ops.step_counter()
    M = B * S
    dp = {k: T(v) for k, v in P.items()}
    ids_t, tt_t, pos_t = T(ids, I32), T(tt, I32), T(pos_ids, I32)
    y, z, mean, rstd = new((B, S, H), BF16), new((M, H), F32), new((M,), F32), new((M,), F32)
    call("polus_embed_ln_fwd_pos", ids_t.ptr, tt_t.ptr, dp["word"].ptr, dp["pos"].ptr, dp["type"].ptr, dp["emb_ln_g"].ptr,
         dp["emb_ln_b"].ptr, B, S, H, V, 1, 1e-5, p, seed, site, sp, y.ptr, z.ptr, mean.ptr, rstd.ptr, pos_t.ptr, n_pos, st())
    mask = philox.dropout_scale_mask((B, S, H), p, seed, site, step) if p > 0 else None
    P64 = {k: v.astype(np.float64) for k, v in P.items()}
    y_ref, cache = RR.embeddings_fwd(ids, tt, P64, pos_ref, mask)
    yd = y.numpy()
    np.testing.assert_allclose(yd, y_ref, atol=3 * BF16_EPS * (1 + np.abs(y_ref).max()), rtol=0)
    if p > 0:  # the same Philox decisions as the existing entry point (its position rows differ, its drops do not)
        y0, z0, m0, r0 = new((B, S, H), BF16), new((M, H), F32), new((M,), F32), new((M,), F32)
        call("polus_embed_ln_fwd", ids_t.ptr, tt_t.ptr, dp["word"].ptr, dp["pos"].ptr, dp["type"].ptr, dp["emb_ln_g"].ptr,
             dp["emb_ln_b"].ptr, B, S, H, V, 1, 1e-5, p, seed, site, sp, y0.ptr, z0.ptr, m0.ptr, r0.ptr, st())
        assert np.array_equal(yd == 0, y0.numpy() == 0) and np.array_equal(yd == 0, mask == 0)
    dy = dev.bf16_round(rng.standard_normal((B, S, H)).astype(np.float32))
    g = {k: new(v.shape, F32) for k, v in P.items()}
    ws = new((int(call("polus_embed_ws_floats", B, S, H)),), F32)
    call("polus_embed_ln_bwd_pos", T(dy, BF16).ptr, z.ptr, mean.ptr, rstd.ptr, dp["emb_ln_g"].ptr, ids_t.ptr, tt_t.ptr, B, S,
         H, V, 1, p, seed, site, sp, g["word"].ptr, g["pos"].ptr, g["type"].ptr, g["emb_ln_g"].ptr, g["emb_ln_b"].ptr, ws.ptr,
         pos_t.ptr, n_pos, st())
    g_ref = RR.embeddings_bwd(dy.astype(np.float64), cache, P64)
    assert np.abs(g_ref["pos"][PAD]).max() > 0
    for k in P:
        ref = g_ref[k]
        np.testing.assert_allclose(g[k].numpy(), ref, rtol=1e-4, atol=1e-4 * (np.abs(ref).max() + 1e-6), err_msg=k)


def _roberta_config(**kw):
    from polus_b200.nn import BertConfig
    base = dict(model_type="roberta", pad_token_id=PAD, type_vocab_size=1, layer_norm_eps=1e-5)
    base.update(kw)
    return BertConfig(**base)


def test_position_ids_argument_and_length_check(dev):
    """BertModel honours an explicit position_ids; a RoBERTa config derives the same ids itself; a BERT config without
    them keeps position s; derived ids that would leave the table raise before any launch."""
    from tests.roberta_ref import roberta_position_ids
    from polus_b200 import _lib, tensor
    from polus_b200.nn import BertConfig, BertModel
    tensor.reset_arena()
    B, S, V = 5, 24, 200
    rng = np.random.default_rng(4)
    ids = padded_ids(rng, B, S, V)
    dims = dict(vocab_size=V, hidden_size=64, num_hidden_layers=1, num_attention_heads=4, intermediate_size=128,
                max_position_embeddings=S + 2)
    rob = BertModel(_roberta_config(**dims), add_pooling_layer=False)
    pos_ids = roberta_position_ids(ids, PAD).astype(np.int32)
    derived = rob.bert.embeddings(ids, training=False).numpy()
    explicit = rob.bert.embeddings(ids, training=False, position_ids=pos_ids).numpy()
    assert np.array_equal(derived, explicit)
    h_rob = rob(input_ids=ids, position_ids=pos_ids)["last_hidden_state"].numpy()
    assert np.array_equal(h_rob, rob(input_ids=ids)["last_hidden_state"].numpy())
    bert = BertModel(BertConfig(**dims), add_pooling_layer=False)
    bert.bert.embeddings.position.assign(rob.bert.embeddings.position.numpy())
    default = bert.bert.embeddings(ids, training=False).numpy()
    arange = np.ascontiguousarray(np.broadcast_to(np.arange(S, dtype=np.int32), (B, S)))
    assert np.array_equal(default, bert.bert.embeddings(ids, training=False, position_ids=arange).numpy())
    assert not np.array_equal(default, bert.bert.embeddings(ids, training=False, position_ids=pos_ids).numpy())
    from polus_b200.nn import as_tensor
    from polus_b200.tensor import I32
    long_ids = as_tensor(np.full((1, S + 1), 5, np.int32), I32)   # S + 1 + pad + 1 > S + 2 learned positions
    n0 = _lib.call("polus_launch_count")
    with pytest.raises(ValueError):
        rob.bert.embeddings(long_ids, training=False)
    assert _lib.call("polus_launch_count") == n0


def _golden_state():
    z = np.load(os.path.join(HERE, "golden", "roberta_hf_torch.npz"))
    H = 16
    state = {"roberta.embeddings.word_embeddings.weight": z["w/emb/word"],
             "roberta.embeddings.position_embeddings.weight": z["w/emb/pos"],
             "roberta.embeddings.token_type_embeddings.weight": z["w/emb/type"],
             "roberta.embeddings.LayerNorm.weight": z["w/emb/emb_ln_g"], "roberta.embeddings.LayerNorm.bias": z["w/emb/emb_ln_b"],
             "lm_head.bias": np.zeros(24), "lm_head.dense.weight": np.eye(H), "lm_head.dense.bias": np.zeros(H),
             "lm_head.layer_norm.weight": np.ones(H), "lm_head.layer_norm.bias": np.zeros(H)}
    for i in range(2):
        p, w = f"roberta.encoder.layer.{i}.", lambda n: z[f"w/layers/{i}/{n}"]
        for j, n in enumerate(("query", "key", "value")):
            state[p + f"attention.self.{n}.weight"] = w("Wqkv")[:, j * H:(j + 1) * H].T
            state[p + f"attention.self.{n}.bias"] = w("bqkv")[j * H:(j + 1) * H]
        state.update({p + "attention.output.dense.weight": w("Wo").T, p + "attention.output.dense.bias": w("bo"),
                      p + "attention.output.LayerNorm.weight": w("ln1_g"), p + "attention.output.LayerNorm.bias": w("ln1_b"),
                      p + "intermediate.dense.weight": w("W1").T, p + "intermediate.dense.bias": w("b1"),
                      p + "output.dense.weight": w("W2").T, p + "output.dense.bias": w("b2"),
                      p + "output.LayerNorm.weight": w("ln2_g"), p + "output.LayerNorm.bias": w("ln2_b")})
    return z, {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in state.items()}


def _hidden_states(model, z):
    from polus_b200.nn import as_tensor
    from polus_b200.tensor import I32
    h = model.bert.embeddings(z["ids"].astype(np.int32), z["tt"].astype(np.int32), training=False)
    hs = [h.numpy()]
    m = as_tensor(z["mask"].astype(np.int32), I32)
    for layer in model.bert.encoder.layer:
        h = layer(h, attention_mask=m, training=False)[0]
        hs.append(h.numpy())
    return hs


def test_roberta_checkpoint_import_matches_hf_torch_golden(dev, tmp_path):
    """The golden RoBERTa blocks written as a `roberta.`-prefixed safetensors with `lm_head.*` extras: imported, every
    layer's hidden states within the BERT import test's bar, export(import(x)) == x, and a snapshot directory
    (config.json + model.safetensors) loads through bert_model_from_checkpoint."""
    from safetensors.numpy import save_file
    from polus_b200 import tensor
    from polus_b200.models import BertModel, bert_model_from_checkpoint
    from polus_b200.pretrained import export_hf_bert_weights, load_hf_bert_weights
    z, state = _golden_state()
    snap = tmp_path / "snapshot"
    snap.mkdir()
    save_file(state, str(snap / "model.safetensors"))
    config = {"model_type": "roberta", "architectures": ["RobertaForMaskedLM"], "vocab_size": 24, "hidden_size": 16,
              "num_hidden_layers": 2, "num_attention_heads": 1, "intermediate_size": 32, "max_position_embeddings": 16,
              "type_vocab_size": 1, "layer_norm_eps": 1e-5, "pad_token_id": PAD, "bos_token_id": 0, "eos_token_id": 2,
              "hidden_dropout_prob": 0.0, "attention_probs_dropout_prob": 0.0, "hidden_act": "gelu"}
    (snap / "config.json").write_text(json.dumps(config))
    tensor.reset_arena()
    model = BertModel(_roberta_config(vocab_size=24, hidden_size=16, num_hidden_layers=2, num_attention_heads=1,
                                      intermediate_size=32, max_position_embeddings=16, hidden_dropout_prob=0.0,
                                      attention_probs_dropout_prob=0.0), add_pooling_layer=False)
    unused = load_hf_bert_weights(model, str(snap / "model.safetensors"))
    assert unused == sorted(k for k in state if k.startswith("lm_head."))
    valid = z["mask"].astype(bool)
    hs = _hidden_states(model, z)
    for got, key in zip(hs, ("h0", "h1", "h2")):
        ref = z[key]
        np.testing.assert_allclose(got[valid], ref[valid], atol=4e-2 * (1 + np.abs(ref).max()) / 4, rtol=0)
    back = export_hf_bert_weights(model)
    for k, v in back.items():
        np.testing.assert_array_equal(v, state["roberta." + k])
    loaded = bert_model_from_checkpoint(str(snap))
    c = loaded.config
    assert (c.model_type, c.pad_token_id, c.layer_norm_eps, c.type_vocab_size) == ("roberta", PAD, 1e-5, 1)
    for a, b in zip(_hidden_states(loaded, z), hs):
        assert np.array_equal(a, b)


def _roberta_batch(rng, B, S, vocab, K):
    from tests.parity import make_batch
    ids, mask, tt, tags = make_batch(rng, B, S, vocab, K)
    ids[ids == PAD] = PAD + 1
    ids[mask == 0] = PAD                                   # right padding with the pad id
    ids[0, 3] = PAD                                        # and one pad id among real tokens
    return ids, mask, tt, tags


def test_roberta_ner_crf_matches_oracle_and_trains(dev):
    from oracle import ner_model as O
    from tests.roberta_ref import ner_loss_and_grads
    from polus_b200 import _lib, device, ops, tensor
    from polus_b200.ner.models import BertNERModel
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    from polus_b200.utils import set_random_seed
    from tests.parity import device_grads, device_params_to_oracle, round_weights_to_bf16
    B, S, H, nh, I, vocab, K, seed = 4, 64, 128, 2, 512, 1000, 4, 13
    tensor.reset_arena()
    set_random_seed(seed)
    ops.set_step(0)
    cfg = _roberta_config(vocab_size=vocab, hidden_size=H, num_hidden_layers=2, num_attention_heads=nh, intermediate_size=I,
                          max_position_embeddings=S + 2, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    model = BertNERModel(cfg, output_classes=K, hidden_space=128, droupout_p=0.0)
    rng = np.random.default_rng(seed)
    ids, mask, tt, tags = _roberta_batch(rng, B, S, vocab, K)
    x = {"input_ids": ids, "attention_mask": mask, "token_type_ids": tt}
    y = np.eye(K, dtype=np.float32)[tags]
    model(**x, training=False)
    for w in model.weights:
        if w.name.endswith("gamma"):
            w.assign(1.0 + 0.1 * rng.standard_normal(w.shape))
        elif w.name.endswith(("beta", "bias")):
            w.assign(0.05 * rng.standard_normal(w.shape))
    round_weights_to_bf16(model)
    params = device_params_to_oracle(model)
    with ops.GradientTape() as tape:
        e_dev = model.emissions(**x, training=True)
        loss_t = model.loss(y, model.crf(e_dev, training=True))
    tape.gradient(loss_t, model.trainable_weights)
    loss_dev, e_dev = float(loss_t), e_dev.numpy()
    g_dev = O.flatten(device_grads(model))
    for w in model.weights:
        _lib.call("polus_memset", w.grad.ptr, 0, w.grad.nbytes, device.stream())
    loss_ref, e_ref, g_ref = ner_loss_and_grads(params, ids, mask, tt, tags, nh, PAD)
    g_ref = O.flatten(g_ref)
    np.testing.assert_allclose(e_dev, e_ref, atol=2e-2, rtol=2e-2)
    assert abs(loss_dev - loss_ref) / abs(loss_ref) < 1e-2, (loss_dev, loss_ref)
    worst = min(((float((g_ref[k] * g_dev[k]).sum() / (np.linalg.norm(g_ref[k]) * np.linalg.norm(g_dev[k]) + 1e-300)), k)
                 for k in g_ref), key=lambda t: t[0])
    assert worst[0] >= 0.999, worst
    assert np.abs(g_dev["emb/pos"][PAD]).max() > 0                  # the pad tokens' row is trained, as under TF
    losses = [float(l) for l in (ClassifierTrainer(model, Adam(1e-3), model.loss).train_step(x, y) for _ in range(6))]
    assert np.isfinite(losses).all() and losses[-1] < losses[0], losses


def test_roberta_graph_replay_gradients_equal_eager(dev, monkeypatch):
    """lr = 0 and dropout on: Adam's first moment after 4 steps must agree between op-by-op execution and graph replay
    (the captured step also captures polus_position_ids)."""
    from polus_b200 import ops, tensor
    from polus_b200.ner.models import BertNERModel
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    from polus_b200.utils import set_random_seed

    def run(eager):
        monkeypatch.setenv("POLUS_EAGER", "1" if eager else "0")
        tensor.reset_arena()
        set_random_seed(5)
        ops.set_step(0)
        cfg = _roberta_config(vocab_size=1000, hidden_size=256, num_hidden_layers=2, num_attention_heads=4,
                              intermediate_size=1024, max_position_embeddings=130)
        model = BertNERModel(cfg, output_classes=4)
        ids, mask, tt, tags = _roberta_batch(np.random.default_rng(0), 8, 128, 1000, 4)
        x = {"input_ids": ids, "attention_mask": mask, "token_type_ids": tt}
        y = np.eye(4, dtype=np.float32)[tags]
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


def test_full_roberta_base_matches_fp32_torch_reference(dev):
    """RoBERTa-base dims (vocab 50265, 514 positions, one token type, eps 1e-5) at B = 2, S = 256 against HF torch
    RobertaEmbeddings + 12 RobertaLayers in fp32 with the same weights: test_fullsize_gpu's bars."""
    import torch
    from oracle import ner_model as O, torch_ref
    from tests.roberta_ref import build_torch_roberta
    from polus_b200 import ops, tensor
    from polus_b200.ner.models import BertNERModel
    from polus_b200.pretrained import export_hf_bert_weights
    from polus_b200.utils import set_random_seed
    from tests.parity import device_grads, round_weights_to_bf16
    B, S, vocab, seed = 2, 256, 50265, 21
    tensor.reset_arena()
    set_random_seed(seed)
    ops.set_step(0)
    cfg = _roberta_config(vocab_size=vocab, max_position_embeddings=514, hidden_dropout_prob=0.0,
                          attention_probs_dropout_prob=0.0)
    model = BertNERModel(cfg, output_classes=4, hidden_space=128, droupout_p=0.0)
    rng = np.random.default_rng(seed)
    ids, mask, tt, tags = _roberta_batch(rng, B, S, vocab, 4)
    x = {"input_ids": ids, "attention_mask": mask, "token_type_ids": tt}
    y = np.eye(4, dtype=np.float32)[tags]
    model(**x, training=False)
    for w in model.weights:
        if w.name.endswith("gamma"):
            w.assign(1.0 + 0.1 * rng.standard_normal(w.shape))
        elif w.name.endswith(("beta", "bias")):
            w.assign(0.02 * rng.standard_normal(w.shape))
    round_weights_to_bf16(model)
    torch.manual_seed(0)
    net = build_torch_roberta(vocab, 514, PAD, K=4, head_hidden=128, dropout=0.0)
    head = {"Wa": model.hidden.kernel.numpy(), "ba": model.hidden.bias.numpy(), "Wb": model.out.kernel.numpy(),
            "bb": model.out.bias.numpy(), "trans": model.crf.transitions.numpy()}
    torch_ref.load_weights(net, export_hf_bert_weights(model.bert), head)
    net.train()
    with ops.GradientTape() as tape:
        e_dev = model.emissions(**x, training=True)
        loss_t = model.loss(y, model.crf(e_dev, training=True))
    tape.gradient(loss_t, model.trainable_weights)
    loss_dev, e_dev = float(loss_t), e_dev.numpy()
    g_dev = O.flatten(device_grads(model))
    ti, tm, tt_, tg = (torch.from_numpy(a.astype(np.int64)) for a in (ids, mask, tt, tags))
    e_ref = torch_ref.emissions(net, ti, tm, tt_).detach().numpy()
    loss_ref_t = net(ti, tm, tt_, tg)
    loss_ref_t.backward()
    loss_ref = float(loss_ref_t.detach())
    g_ref = torch_ref.named_grads(net, 768)
    scale = float(np.abs(e_ref).max())
    np.testing.assert_allclose(e_dev, e_ref, atol=2e-2 * scale, rtol=2e-2)
    assert abs(loss_dev - loss_ref) / abs(loss_ref) < 1e-2, (loss_dev, loss_ref)
    assert set(g_ref) == set(g_dev)
    worst = (1.0, None)
    for k, gr in g_ref.items():
        gd = g_dev[k]
        assert gd.shape == gr.shape, k
        denom = np.linalg.norm(gr) * np.linalg.norm(gd)
        cos = float((gr * gd).sum() / denom) if denom > 0 else 1.0
        if cos < worst[0]:
            worst = (cos, k)
    assert worst[0] >= 0.999, worst
