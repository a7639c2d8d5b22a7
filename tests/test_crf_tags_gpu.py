"""CRF loss and Viterbi decode for wide tag sets (33 <= K <= 128) and for K <= 32 at lengths whose [T][K] tables do not fit
the tag-per-lane kernels (K = 31, 32 at T = 512), through the C ABI and through a BERT-NER model, against the fp64 numpy
oracle (itself pinned to brute-force enumeration in test_oracle_cpu.py).  Tolerances are test_kernels_gpu.py's."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from polus_b200 import device
    device.init(0)
    return device


_KEEP = []  # tensors created by T()/new() stay alive for the whole test: `T(x).ptr` must not dangle


@pytest.fixture(autouse=True)
def _keepalive():
    yield
    _KEEP.clear()


def T(arr, dtype=None):
    from polus_b200.tensor import Tensor
    t = Tensor.from_numpy(arr, dtype)
    _KEEP.append(t)
    return t


def new(shape, dtype, zero=True):
    from polus_b200.tensor import Tensor
    t = Tensor(shape, dtype, zero=zero)
    _KEEP.append(t)
    return t


def call(name, *a):
    from polus_b200 import _lib
    return _lib.call(name, *a)


def st():
    from polus_b200 import device
    return device.stream()


# -------------------------------------------------------------------------------------------------- loss and gradients
@pytest.mark.parametrize("B,Tn,K,lens,weighted", [
    (2, 512, 32, None, False), (2, 512, 31, None, False),  # K <= 32 beyond crf_nll_kernel's shared memory
    (3, 64, 33, "ragged", True), (4, 256, 64, "ragged", False), (2, 100, 128, "ragged", True), (2, 512, 128, None, False),
    (3, 1, 100, None, False),
    (4, 40, 48, [0, 1, 40, 17], True),
])
def test_crf_nll_and_grads_wide(dev, B, Tn, K, lens, weighted):
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32, I32
    rng = np.random.default_rng(B * Tn + K)
    emis = rng.standard_normal((B, Tn, K)).astype(np.float32) * 2
    tags = rng.integers(0, K, (B, Tn)).astype(np.int32)
    trans = rng.standard_normal((K, K)).astype(np.float32)
    if lens is None:
        ln = np.full(B, Tn, np.int32)
    elif lens == "ragged":
        ln = rng.integers(0, Tn + 1, B).astype(np.int32)
    else:
        ln = np.array(lens, np.int32)
    w = rng.uniform(0.2, 2.0, B).astype(np.float32) if weighted else None
    nll, loss, gtr = new((B,), F32), new((), F32), T(np.zeros((K, K), np.float32))
    gem = T(np.full((B, Tn, K), 7.0, np.float32))  # the kernel writes every row, zeros beyond len included
    call("polus_crf_nll", T(emis).ptr, T(tags, I32).ptr, T(ln, I32).ptr if lens is not None else None, T(trans).ptr,
         T(w).ptr if weighted else None, B, Tn, K, nll.ptr, loss.ptr, gem.ptr, gtr.ptr, st())
    nll_r, loss_r, gem_r, gtr_r = R.crf_nll_with_grads(emis.astype(np.float64), tags, ln, trans.astype(np.float64), w)
    np.testing.assert_allclose(nll.numpy(), nll_r, rtol=2e-5, atol=2e-4)
    np.testing.assert_allclose(float(loss), loss_r, rtol=2e-5, atol=1e-5)
    np.testing.assert_allclose(gem.numpy(), gem_r, rtol=2e-3, atol=1e-3 * np.abs(gem_r).max() + 1e-6)
    np.testing.assert_allclose(gtr.numpy(), gtr_r, rtol=2e-3, atol=1e-3 * np.abs(gtr_r).max() + 1e-5)
    np.testing.assert_allclose(-nll.numpy(), R.crf_log_likelihood(emis.astype(np.float64), tags, ln, trans.astype(np.float64)),
                               rtol=2e-5, atol=2e-4)


def test_crf_nll_wide_accumulates_into_transition_gradient(dev):
    """d_gtrans is accumulated into, as by the other CRF kernels (the layer adds a gradient it did not zero)."""
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32, I32
    rng = np.random.default_rng(5)
    B, Tn, K = 3, 50, 70
    emis = rng.standard_normal((B, Tn, K)).astype(np.float32)
    tags = rng.integers(0, K, (B, Tn)).astype(np.int32)
    trans = rng.standard_normal((K, K)).astype(np.float32)
    g0 = rng.standard_normal((K, K)).astype(np.float32)
    gtr = T(g0)
    call("polus_crf_nll", T(emis).ptr, T(tags, I32).ptr, None, T(trans).ptr, None, B, Tn, K, None, None,
         new((B, Tn, K), F32).ptr, gtr.ptr, st())
    _, _, _, gtr_r = R.crf_nll_with_grads(emis.astype(np.float64), tags, np.full(B, Tn), trans.astype(np.float64))
    np.testing.assert_allclose(gtr.numpy(), g0 + gtr_r, rtol=2e-3, atol=1e-3 * np.abs(gtr_r).max() + 1e-5)


# -------------------------------------------------------------------------------------------------- Viterbi
@pytest.mark.parametrize("B,Tn,K,ragged", [(B, Tn, K, rg) for K in (33, 64, 128) for Tn in (40, 512) for rg, B in ((False, 3), (True, 5))]
                         + [(2, 7000, 32, True)])  # K = 32 beyond crf_decode_kernel's shared memory
def test_viterbi_wide_bit_exact(dev, B, Tn, K, ragged):
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32, I32
    rng = np.random.default_rng(Tn + K + B)
    # quantised emissions/transitions => many exact ties, and fp32 sums that are exact in both implementations
    emis = (rng.integers(-4, 5, (B, Tn, K)) * 0.5).astype(np.float32)
    trans = (rng.integers(-2, 3, (K, K)) * 0.5).astype(np.float32)
    lens = rng.integers(0, Tn + 1, B).astype(np.int32) if ragged else np.full(B, Tn, np.int32)
    if ragged:
        lens[:2] = (0, 1)
    tags, score = new((B, Tn), I32), new((B,), F32)
    call("polus_crf_decode", T(emis).ptr, T(lens, I32).ptr if ragged else None, T(trans).ptr, B, Tn, K, tags.ptr, score.ptr, st())
    tags_r, score_r = R.crf_decode(emis, lens, trans)
    assert np.array_equal(tags.numpy(), tags_r)
    assert np.array_equal(score.numpy(), score_r.astype(np.float32))
    emis = rng.standard_normal((B, Tn, K)).astype(np.float32)
    trans = rng.standard_normal((K, K)).astype(np.float32)
    call("polus_crf_decode", T(emis).ptr, T(lens, I32).ptr if ragged else None, T(trans).ptr, B, Tn, K, tags.ptr, score.ptr, st())
    tags_r, _ = R.crf_decode(emis, lens, trans)
    assert np.array_equal(tags.numpy(), tags_r)


# -------------------------------------------------------------------------------------------------- mask and sample weights
def test_crf_mask_and_sample_weights_k64(dev):
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32
    rng = np.random.default_rng(64)
    K = 64
    trans = rng.standard_normal((K, K)).astype(np.float32)
    mask = (rng.uniform(size=(K, K)) > 0.3).astype(np.float32)
    out = new((K, K), F32)
    call("polus_crf_mask_transitions", T(trans).ptr, T(mask).ptr, K, out.ptr, st())
    assert np.array_equal(out.numpy(), R.crf_masked_transitions(trans, mask))
    B, Tn = 7, 30
    tags = rng.integers(0, 2, (B, Tn))
    tags[2, 5], tags[4, 7], tags[5, 0] = 40, 63, 33
    y = np.eye(K, dtype=np.float32)[tags]
    mp = (np.arange(K) >= 33).astype(np.float32)
    w = new((B,), F32)
    call("polus_crf_sample_weights", T(y).ptr, T(mp).ptr, 0.25, B, Tn, K, w.ptr, st())
    assert np.array_equal(w.numpy(), R.crf_sample_weights(y, mp, 0.25))


# -------------------------------------------------------------------------------------------------- model level
def _ner_model(K, seed):
    from polus_b200 import ops, tensor
    from polus_b200.models import BertConfig
    from polus_b200.ner.models import BertNERModel
    from polus_b200.utils import set_random_seed
    tensor.reset_arena()
    set_random_seed(seed)
    ops.set_step(0)
    cfg = BertConfig(vocab_size=1000, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256,
                     max_position_embeddings=128, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    return BertNERModel(cfg, output_classes=K, droupout_p=0.0)


def _ner_batch(K, B=4, S=128):
    from tests.parity import make_batch
    ids, mask, tt, tags = make_batch(np.random.default_rng(K), B, S, 1000, K)
    return {"input_ids": ids, "attention_mask": mask, "token_type_ids": tt}, np.eye(K, dtype=np.float32)[tags]


@pytest.mark.parametrize("K", [45, 64])  # tag projection on gemm_small (K % 8 != 0) and on the tcgen05 GEMM
def test_bert_ner_wide_tags_graph_replay_equals_eager(dev, monkeypatch, K):
    """Eager first step, capture, replays vs op-by-op execution, with lr = 0 so that every step computes the same
    gradients (tolerances of test_model_gpu.py::test_graph_replay_gradients_equal_eager)."""
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    x, y = _ner_batch(K)

    def run(eager):
        monkeypatch.setenv("POLUS_EAGER", "1" if eager else "0")
        model = _ner_model(K, 5)
        opt = Adam(0.0)
        tr = ClassifierTrainer(model, opt, model.loss)
        losses = [float(tr.train_step(x, y)) for _ in range(4)]
        return losses, opt.variables()[0].numpy()
    le, me = run(True)
    lg, mg = run(False)
    assert np.all(np.isfinite(le)) and le[0] > 0
    np.testing.assert_allclose(lg, le, rtol=1e-5)
    scale = np.abs(me).max()
    assert scale > 0
    assert np.abs(mg - me).max() <= 2e-4 * scale, (np.abs(mg - me).max(), scale)


@pytest.mark.parametrize("K", [45, 64])
def test_bert_ner_wide_tags_trains_and_decodes(dev, monkeypatch, K):
    from oracle import numpy_ref as R
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    monkeypatch.setenv("POLUS_EAGER", "0")
    x, y = _ner_batch(K)
    model = _ner_model(K, 7)
    tr = ClassifierTrainer(model, Adam(1e-3), model.loss)
    losses = [float(tr.train_step(x, y)) for _ in range(8)]
    assert np.all(np.isfinite(losses))
    assert losses[-1] < 0.9 * losses[0], losses
    # inference = Viterbi over the full length on the emissions and transitions the model holds
    pred = model.inference(x).numpy()
    emis = model.emissions(**x, training=False).numpy().astype(np.float32)
    B, S = pred.shape
    tags_r, _ = R.crf_decode(emis, np.full(B, S), model.crf.transitions.numpy())
    assert np.array_equal(pred, tags_r)
