"""GPU tests of the remaining SURVEY §8(a) rows through the polus-shaped API: split BERT / build_bert_embeddings
(a8, a9; mirrors the reference's tests/test_models.py with a two-sided comparison), CRF.loss_sample_weights and the
transition mask (a10, a13), the IR bi-encoder trainer (a19), and the two larger BASELINE configs as parity cases
(cross-encoder S=512 pairwise loss; BERT-large dims S=512)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _tiny_cfg(**kw):
    from polus_b200.models import BertConfig
    base = dict(vocab_size=400, hidden_size=128, num_hidden_layers=4, num_attention_heads=4, intermediate_size=256,
                max_position_embeddings=64, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    base.update(kw)
    return BertConfig(**base)


def _inputs(rng, B, S, vocab):
    ids = rng.integers(0, vocab, (B, S)).astype(np.int32)
    lens = rng.integers(S // 2, S + 1, B)
    mask = (np.arange(S)[None] < lens[:, None]).astype(np.int32)
    tt = (np.arange(S)[None] >= (lens[:, None] // 2)).astype(np.int32) * mask
    return {"input_ids": ids, "attention_mask": mask, "token_type_ids": tt}


def test_split_bert_model_and_build_bert_embeddings():
    """pre_model output == hidden state entering the cut; post_model(pre) == full model (tests/test_models.py:6-67)."""
    from polus_b200 import tensor
    from polus_b200.data import build_bert_embeddings
    from polus_b200.models import BertModel, TFBertSplited, split_bert_model
    from polus_b200.utils import set_random_seed
    tensor.reset_arena()
    set_random_seed(1)
    rng = np.random.default_rng(0)
    x = _inputs(rng, 3, 32, 400)
    full = BertModel(_tiny_cfg())
    ref_out = full(**x)["last_hidden_state"].numpy()
    with pytest.raises(AssertionError):
        split_bert_model(full, 0)
    pre, post = split_bert_model(full, -2)
    assert isinstance(post, TFBertSplited) and len(post.layer) == 2 and pre.config.num_hidden_layers == 2
    assert len(post.trainable_weights) == 2 * 12
    emb = build_bert_embeddings(pre)  # frozen lower part, as used for train_map_f preprocessing
    hidden = emb(**x)["last_hidden_state"]
    out = post(hidden, x["attention_mask"], training=False)
    np.testing.assert_array_equal(out["last_hidden_state"].numpy(), ref_out)  # same kernels, same order: bit-identical
    np.testing.assert_array_equal(out["pooler_output"].numpy(), ref_out[:, 0, :])  # models.py:216: no pooler dense
    # Keras-order weights round-trip: 16 arrays per layer
    w = post.layer[0].get_weights()
    assert len(w) == 16 and w[0].shape == (128, 128) and w[10].shape == (128, 256)
    post.layer[1].set_weights(w)
    np.testing.assert_array_equal(post.layer[1].get_weights()[4], w[4])


def test_crf_layer_loss_variants_match_oracle():
    from oracle import numpy_ref as R
    from polus_b200 import ops, tensor
    from polus_b200.layers import CRF
    from polus_b200.tensor import Tensor
    tensor.reset_arena()
    rng = np.random.default_rng(3)
    B, T, K = 6, 24, 4
    mask = np.ones((K, K), np.float32)
    mask[1, 3] = 0  # O -> I-Chemical forbidden
    crf = CRF(K, mask_impossible_transitions=mask)
    emis = rng.standard_normal((B, T, K)).astype(np.float32)
    tags = rng.integers(0, 2, (B, T))
    tags[1, 3], tags[4, 7] = 2, 3
    y = np.eye(K, dtype=np.float32)[tags]
    e_t = Tensor.from_numpy(emis)
    e_t.requires_grad = True
    out = crf(e_t, training=True)
    assert out is e_t or np.array_equal(out.numpy(), emis)      # training phase returns the emissions (layers.py:84)
    trans = crf.transitions.numpy()
    teff = R.crf_masked_transitions(trans, mask).astype(np.float64)
    lens = np.full(B, T)
    # plain loss
    with ops.GradientTape() as tape:
        loss = crf.loss(y, crf(e_t, training=True))
    g_e, g_t = tape.gradient(loss, [e_t, crf.transitions])
    _, loss_r, ge_r, gt_r = R.crf_nll_with_grads(emis.astype(np.float64), tags, lens, teff)
    np.testing.assert_allclose(float(loss), loss_r, rtol=1e-5)
    np.testing.assert_allclose(g_e.numpy(), ge_r, rtol=2e-3, atol=1e-5)
    np.testing.assert_allclose(g_t.numpy(), gt_r * mask, rtol=2e-3, atol=1e-5)   # d/dT of T*mask + const
    # sample-weighted loss (layers.py:101-126)
    crf.transitions.grad.numpy()
    mp = np.array([0, 0, 1, 1], np.float32)
    w = R.crf_sample_weights(y, mp, 0.2)
    loss_w = crf.loss_sample_weights(mp, 0.2)(y, crf(e_t, training=True))
    _, lw_r, _, _ = R.crf_nll_with_grads(emis.astype(np.float64), tags, lens, teff, w)
    np.testing.assert_allclose(float(loss_w), lw_r, rtol=1e-5)
    # inference phase: one-hot Viterbi path; NERBertModel.inference = argmax of it
    onehot = crf(e_t, training=False).numpy()
    path, _ = R.crf_decode(emis, lens, teff.astype(np.float32))
    assert np.array_equal(onehot.argmax(-1), path)


def test_ir_bi_encoder_trainer_in_batch_negatives():
    """EfficientDenseRetrievalTrainer (polus/ir/training.py): frozen encoders, trainable projections, user score + loss."""
    from polus_b200 import tensor
    from polus_b200.ir.models import BertBiEncoder, in_batch_scores, softmax_ranking_loss
    from polus_b200.ir.training import EfficientDenseRetrievalTrainer
    from polus_b200.optimizers import Adam
    from polus_b200.utils import set_random_seed
    tensor.reset_arena()
    set_random_seed(5)
    rng = np.random.default_rng(5)
    model = BertBiEncoder(_tiny_cfg(num_hidden_layers=2), projection_dim=64)
    B, S = 8, 32
    q = {k: v for k, v in _inputs(rng, B, S, 400).items() if k != "token_type_ids"}
    d = {k: v for k, v in _inputs(rng, B, S, 400).items() if k != "token_type_ids"}
    q_rep = model.encode_query(q).numpy().astype(np.float64)
    d_rep = model.encode_document(d).numpy().astype(np.float64)
    model.query_projection(model.encode_query(q))       # build the lazily-created projections
    model.document_projection(model.encode_document(d))
    enc_before = model.query_encoder.bert.encoder.layer[0].Wo.numpy().copy()
    Wq, bq = model.query_projection.kernel.numpy().astype(np.float64), model.query_projection.bias.numpy().astype(np.float64)
    Wd, bd = model.document_projection.kernel.numpy().astype(np.float64), model.document_projection.bias.numpy().astype(np.float64)
    trainer = EfficientDenseRetrievalTrainer(model, in_batch_scores, optimizer=Adam(1e-2), loss=softmax_ranking_loss)
    assert [id(w) for w in trainer.trainable_weights] == [id(w) for w in model.trainable_weights] and len(trainer.trainable_weights) == 4
    losses = [float(trainer.train_step(q, d)) for _ in range(6)]
    # oracle for the first loss: projections -> q d^T -> CE against the diagonal
    from polus_b200 import device
    rb = device.bf16_round
    qp = rb((rb(q_rep.astype(np.float32)).astype(np.float64) @ rb(Wq.astype(np.float32)) + bq).astype(np.float32)).astype(np.float64)
    dp = rb((rb(d_rep.astype(np.float32)).astype(np.float64) @ rb(Wd.astype(np.float32)) + bd).astype(np.float32)).astype(np.float64)
    s = qp @ dp.T
    lse = np.log(np.exp(s - s.max(1, keepdims=True)).sum(1)) + s.max(1)
    np.testing.assert_allclose(losses[0], float((lse - np.diag(s)).mean()), rtol=2e-2)
    assert losses[-1] < losses[0] * 0.7, losses                     # the projections learn
    np.testing.assert_array_equal(model.query_encoder.bert.encoder.layer[0].Wo.numpy(), enc_before)  # encoders stay frozen


def test_cross_encoder_pairwise_seq512():
    """BASELINE config 4 as a parity case: BERT cross-encoder, S=512, pairwise softplus loss (our definition: the
    reference ships no pairwise loss, SURVEY §0.9)."""
    from oracle import ner_model as O, numpy_ref as R
    from polus_b200 import ops, tensor
    from polus_b200.ir.models import BertCrossEncoder, pairwise_softplus_loss
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    from polus_b200.utils import set_random_seed
    from tests.parity import round_weights_to_bf16
    tensor.reset_arena()
    set_random_seed(9)
    rng = np.random.default_rng(9)
    cfg = _tiny_cfg(num_hidden_layers=2, max_position_embeddings=512)
    model = BertCrossEncoder(cfg)
    B2, S = 4, 512
    x = _inputs(rng, B2, S, 400)
    model(**x)
    round_weights_to_bf16(model)
    emb = model.bert.bert.embeddings
    r = lambda p: p.numpy().astype(np.float64)
    params = {"emb": {"word": r(emb.word), "pos": r(emb.position), "type": r(emb.token_type), "emb_ln_g": r(emb.ln_gamma),
                      "emb_ln_b": r(emb.ln_beta)},
              "layers": [{k: r(getattr(l, k)) for k in ("Wqkv", "bqkv", "Wo", "bo", "ln1_g", "ln1_b", "W1", "b1", "W2", "b2",
                                                        "ln2_g", "ln2_b")} for l in model.bert.bert.encoder.layer]}
    h, _ = R.bert_embeddings_fwd(x["input_ids"], x["token_type_ids"], params["emb"])
    add = R.attention_mask_additive(x["attention_mask"]).astype(np.float64)
    for lp in params["layers"]:
        h, _ = R.bert_layer_fwd(h, add, lp, 4)
    s_ref = (h[:, 0, :] @ r(model.score.kernel) + r(model.score.bias))[:, 0]
    loss_ref = np.mean(np.log1p(np.exp(s_ref[2:] - s_ref[:2])))
    scores = model(**x).numpy()
    np.testing.assert_allclose(scores[:, 0], s_ref, atol=2e-2, rtol=2e-2)
    trainer = ClassifierTrainer(model, Adam(1e-3), pairwise_softplus_loss)
    losses = [float(trainer.train_step(x, np.zeros(B2, np.float32))) for _ in range(5)]
    np.testing.assert_allclose(losses[0], loss_ref, rtol=2e-2, atol=2e-3)
    assert losses[-1] < losses[0]


def test_bert_large_dims_seq512_parity():
    """BASELINE config 5 dims (H=1024, 16 heads, I=4096, S=512) on one layer: forward+backward+Adam vs the oracle."""
    from tests.parity import run_tiny_ner_parity
    r = run_tiny_ner_parity(steps=2, B=1, S=512, H=1024, nh=16, I=4096, L=1, vocab=1200)
    assert r["ok"], r


def test_ner_sequential_metrics_on_device():
    """§8f rank 1 (validation path): token-level MacroF1 / Accuracy over [B, S] label tensors -- confusion matrix built by
    polus_confusion_matrix on the device, bit-exact against numpy; formulas of polus/ner/metrics.py:39-72."""
    from polus_b200 import device
    from polus_b200.ner.metrics import Accuracy, MacroF1Score
    device.init(0)
    rng = np.random.default_rng(5)
    K = 4
    f1, acc = MacroF1Score(num_classes=K), Accuracy(num_classes=K)
    cm = np.zeros((K, K), np.int64)
    for _ in range(3):
        y = rng.integers(0, K, (16, 256)).astype(np.int32)
        p = np.where(rng.random((16, 256)) < 0.7, y, rng.integers(0, K, (16, 256))).astype(np.int32)
        f1.samples_from_batch((y, p))
        acc.samples_from_batch((y, p))
        np.add.at(cm, (y.reshape(-1), p.reshape(-1)), 1)
    assert np.array_equal(f1.confusion_matrix, cm)
    tp = np.diag(cm).astype(np.float64)
    prec, rec = tp / cm.sum(-1), tp / cm.sum(-2)
    assert f1.evaluate() == pytest.approx(float(np.mean(2 / (1 / rec + 1 / prec))), rel=1e-12)
    assert acc.evaluate() == pytest.approx(float(tp.sum() / cm.sum()), rel=1e-12)


def test_hf_checkpoint_import_matches_hf_torch_golden(tmp_path):
    """§8f rank 3 + a direct device-vs-HuggingFace check: the golden fixture (HF torch BertEmbeddings + 2 BertLayers, fp64,
    tests/golden/make_golden.py) is written as a HuggingFace-named .safetensors checkpoint, imported with
    polus_b200.pretrained.load_hf_bert_weights, and the device forward must reproduce HF's hidden states of every layer
    within bf16 tolerance; export(import(x)) == x."""
    import os
    from polus_b200 import device, ops, tensor
    from polus_b200.models import BertConfig, BertModel
    from polus_b200.pretrained import export_hf_bert_weights, load_hf_bert_weights
    device.init(0)
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bert_hf_torch.npz"))
    H = 64
    state = {"bert.embeddings.word_embeddings.weight": z["w/emb/word"], "bert.embeddings.position_embeddings.weight": z["w/emb/pos"],
             "bert.embeddings.token_type_embeddings.weight": z["w/emb/type"], "bert.embeddings.LayerNorm.weight": z["w/emb/emb_ln_g"],
             "bert.embeddings.LayerNorm.bias": z["w/emb/emb_ln_b"], "cls.predictions.bias": np.zeros(100)}
    for i in range(2):
        p, w = f"bert.encoder.layer.{i}.", lambda n: z[f"w/layers/{i}/{n}"]
        for j, n in enumerate(("query", "key", "value")):
            state[p + f"attention.self.{n}.weight"] = w("Wqkv")[:, j * H:(j + 1) * H].T
            state[p + f"attention.self.{n}.bias"] = w("bqkv")[j * H:(j + 1) * H]
        state.update({p + "attention.output.dense.weight": w("Wo").T, p + "attention.output.dense.bias": w("bo"),
                      p + "attention.output.LayerNorm.weight": w("ln1_g"), p + "attention.output.LayerNorm.bias": w("ln1_b"),
                      p + "intermediate.dense.weight": w("W1").T, p + "intermediate.dense.bias": w("b1"),
                      p + "output.dense.weight": w("W2").T, p + "output.dense.bias": w("b2"),
                      p + "output.LayerNorm.weight": w("ln2_g"), p + "output.LayerNorm.bias": w("ln2_b")})
    state = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in state.items()}
    from safetensors.numpy import save_file
    path = str(tmp_path / "model.safetensors")
    save_file(state, path)
    tensor.reset_arena()
    cfg = BertConfig(vocab_size=100, hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=128,
                     max_position_embeddings=32, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    model = BertModel(cfg, add_pooling_layer=False)
    unused = load_hf_bert_weights(model, path)
    assert unused == ["cls.predictions.bias"]
    ids, tt, mask = z["ids"].astype(np.int32), z["tt"].astype(np.int32), z["mask"].astype(np.int32)
    h = model.bert.embeddings(ids, tt, training=False)
    hs = [h.numpy()]
    from polus_b200.nn import as_tensor
    from polus_b200.tensor import I32
    m = as_tensor(mask, I32)
    for layer in model.bert.encoder.layer:
        h = layer(h, attention_mask=m, training=False)[0]
        hs.append(h.numpy())
    valid = mask.astype(bool)  # HF's padded query rows attend to nothing meaningful: compare real tokens
    for got, key in zip(hs, ("h0", "h1", "h2")):
        ref = z[key]
        np.testing.assert_allclose(got[valid], ref[valid], atol=4e-2 * (1 + np.abs(ref).max()) / 4, rtol=0)
    back = export_hf_bert_weights(model)
    for k, v in back.items():
        np.testing.assert_array_equal(v, state["bert." + k])
    with pytest.raises(ValueError):
        load_hf_bert_weights(BertModel(BertConfig(vocab_size=99, hidden_size=64, num_hidden_layers=2, num_attention_heads=4,
                                                  intermediate_size=128, max_position_embeddings=32), add_pooling_layer=False), state)


def test_bench_dump_outputs_agree_between_two_runs(tmp_path):
    """`bench.py --dump-outputs`: with the same arguments the inputs and the weights each timed region starts from are the
    same, so two runs must write the same losses up to the last-bit differences of the float-atomic reductions.  Measured
    on a B200 with these arguments over three runs: 0 (resident) and 7.7e-8 (host-fed) relative spread; the same runs
    without the restore (the loss_last of the bench line) spread by 2.4e-5, so the 1e-6 bar tells the two apart."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    losses = []
    for run in ("a", "b"):
        out = tmp_path / run
        cmd = [sys.executable, os.path.join(root, "bench.py"), "--batch", "32", "--steps", "5", "--warmup", "3",
               "--preheat-steps", "10", "--sweep-batch", "0", "--no-strong", "--no-extra-configs", "--no-cpu-baseline",
               "--dump-outputs", str(out)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
        assert r.returncode == 0, r.stderr[-3000:]
        assert sorted(os.listdir(out)) == ["loss_e2e.npy", "loss_resident.npy"]
        losses.append({n: float(np.load(out / n)[0]) for n in os.listdir(out)})
    print("dumped losses:", losses)
    for name, a in losses[0].items():
        b = losses[1][name]
        assert np.isfinite(a) and abs(a - b) <= 1e-6 * abs(a), (name, a, b)
