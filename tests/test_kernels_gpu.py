"""GPU parity tests, kernel by kernel, through the C ABI (ctypes) against the CPU oracle.

Bar (BASELINE.md §3): bit-exact for integer / index work (Viterbi paths, dropout masks, argmax, confusion
matrix); fp32 kernels rtol 1e-5-ish (stated per test); bf16-storage kernels within bf16 rounding (2^-8 rel).
"""
import ctypes as C

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


def step_ptr(value=0):
    from polus_b200 import ops
    ops.set_step(value)
    return ops.step_counter()


BF16_EPS = 2.0 ** -8


# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,H,p", [(64, 768, 0.0), (37, 128, 0.0), (50, 1024, 0.1), (8, 2048, 0.0), (0, 768, 0.0),
                                   (21, 384, 0.1), (33, 640, 0.0), (29, 1000, 0.1),
                                   # several rows per warp: the backward's 296 CTAs x 8 warps take a second row past
                                   # M = 2368 (7109 = three row strides + 5), the forward's 2368 x 4 warps past 9472
                                   (7109, 256, 0.1), (20000, 256, 0.0), (7109, 512, 0.0), (20000, 512, 0.1),
                                   (7109, 768, 0.1), (20000, 768, 0.0), (7109, 1024, 0.0), (20000, 1024, 0.1),
                                   (5000, 4096, 0.1)])
def test_ln_residual_fwd_bwd(dev, M, H, p):
    from oracle import numpy_ref as R, philox
    from polus_b200.tensor import BF16, F32
    rng = np.random.default_rng(M + H)
    x = dev.bf16_round(rng.standard_normal((M, H)).astype(np.float32))
    res = dev.bf16_round(rng.standard_normal((M, H)).astype(np.float32))
    gamma = (1 + 0.1 * rng.standard_normal(H)).astype(np.float32)
    beta = (0.1 * rng.standard_normal(H)).astype(np.float32)
    dy = dev.bf16_round(rng.standard_normal((M, H)).astype(np.float32))
    seed, site, step = 1234, 5, 3
    sp = step_ptr(step)
    dx_t, dres_t = new((M, H), BF16), new((M, H), BF16)
    x_t, res_t, g_t, b_t, y_t = T(x, BF16), T(res, BF16), T(gamma), T(beta), new((M, H), BF16)
    mean_t, rstd_t = new((M,), F32), new((M,), F32)
    from polus_b200.tensor import U8
    keep_t = new((max(M * (H // 8), 1),), U8)
    call("polus_ln_res_fwd", x_t.ptr, res_t.ptr, g_t.ptr, b_t.ptr, M, H, 1e-12, p, seed, site, sp, y_t.ptr, mean_t.ptr, rstd_t.ptr,
         keep_t.ptr if p > 0 else None, st())
    if M == 0:
        return
    mask = philox.dropout_scale_mask((M, H), p, seed, site, step) if p > 0 else np.ones((M, H), np.float32)
    z = x * mask + res
    y_ref, cache = R.layer_norm(z.astype(np.float64), gamma, beta)
    np.testing.assert_allclose(y_t.numpy(), y_ref, atol=3 * BF16_EPS * (1 + np.abs(y_ref).max()), rtol=0)
    z_dev = x_t.numpy()  # x was overwritten with z
    np.testing.assert_allclose(z_dev, z, atol=BF16_EPS * (1 + np.abs(z).max()), rtol=0)
    # backward uses the device's (bf16-rounded) z
    ggam, gbet, gbx = new((H,), F32), new((H,), F32), new((H,), F32)
    dy_t = T(dy, BF16)
    # d(y) arrives as two contributions (residual stream): dy = dy_a + dy_b, summed inside the kernel
    dy_a = dev.bf16_round((0.5 * dy).astype(np.float32))
    dy_b = dev.bf16_round((dy - dy_a).astype(np.float32))
    dy = dy_a + dy_b
    call("polus_ln_res_bwd", T(dy_a, BF16).ptr, T(dy_b, BF16).ptr, x_t.ptr, mean_t.ptr, rstd_t.ptr, g_t.ptr, M, H, p, seed,
         site, sp, dx_t.ptr, dres_t.ptr, ggam.ptr, gbet.ptr, gbx.ptr, keep_t.ptr if p > 0 else None, st())
    if p > 0:  # keep bits are exactly the oracle's Philox decisions; regenerating them in-kernel gives the same dx
        bits = np.unpackbits(keep_t.numpy()[:M * (H // 8)].reshape(M, H // 8, 1), axis=2, bitorder="little").reshape(M, H)
        assert np.array_equal(bits.astype(bool), mask > 0)
        dx2_t = new((M, H), BF16)
        call("polus_ln_res_bwd", T(dy_a, BF16).ptr, T(dy_b, BF16).ptr, x_t.ptr, mean_t.ptr, rstd_t.ptr, g_t.ptr, M, H, p, seed,
             site, sp, dx2_t.ptr, dres_t.ptr, new((H,), F32).ptr, new((H,), F32).ptr, None, None, st())
        assert np.array_equal(dx2_t.numpy(), dx_t.numpy())
    _, cache_dev = R.layer_norm(z_dev.astype(np.float64), gamma, beta)
    dz_ref, gg_ref, gb_ref = R.layer_norm_bwd(dy.astype(np.float64), cache_dev, gamma)
    tol = 3 * BF16_EPS * (1 + np.abs(dz_ref).max())
    np.testing.assert_allclose(dres_t.numpy(), dz_ref, atol=tol, rtol=0)
    np.testing.assert_allclose(dx_t.numpy(), dz_ref * mask, atol=tol * 1.2, rtol=0)
    np.testing.assert_allclose(ggam.numpy(), gg_ref, rtol=2e-3, atol=2e-3 * np.abs(gg_ref).max())
    np.testing.assert_allclose(gbet.numpy(), gb_ref, rtol=2e-3, atol=2e-3 * np.abs(gb_ref).max())
    gx_ref = dx_t.numpy().astype(np.float64).sum(0)  # bias gradient of the producing Dense = column sums of dx
    np.testing.assert_allclose(gbx.numpy(), gx_ref, rtol=1e-2, atol=1e-2 * (np.abs(gx_ref).max() + 1))


def test_dropout_mask_bit_exact(dev):
    """Index work: the Philox keep-mask regenerated by the oracle must equal the device's exactly."""
    from oracle import philox
    from polus_b200.tensor import BF16
    n = 8 * 4099
    x = np.ones(n, np.float32)
    for p, seed, site, step in [(0.1, 42, 1, 0), (0.5, 2 ** 40 + 17, 9, 123456)]:
        sp = step_ptr(step)
        y = new((n,), BF16)
        call("polus_dropout", T(x, BF16).ptr, y.ptr, n, p, seed, site, sp, st())
        keep_dev = y.numpy() != 0
        keep_ref = philox.dropout_keep_mask(n, p, seed, site, step)
        assert np.array_equal(keep_dev, keep_ref)
        assert abs(keep_dev.mean() - (1 - p)) < 0.01


@pytest.mark.parametrize("B,S,H,V,p", [(3, 16, 128, 50, 0.0), (2, 64, 768, 300, 0.1)])
def test_embedding_ln_fwd_bwd(dev, B, S, H, V, p):
    from oracle import numpy_ref as R, philox
    from polus_b200.tensor import BF16, F32, I32
    rng = np.random.default_rng(5)
    P = {"word": rng.normal(0, 0.5, (V, H)).astype(np.float32), "pos": rng.normal(0, 0.5, (S + 3, H)).astype(np.float32),
         "type": rng.normal(0, 0.5, (2, H)).astype(np.float32), "emb_ln_g": (1 + 0.1 * rng.standard_normal(H)).astype(np.float32),
         "emb_ln_b": (0.1 * rng.standard_normal(H)).astype(np.float32)}
    ids = rng.integers(0, V, (B, S)).astype(np.int32)
    ids[0, :4] = 7  # repeated ids: scatter-add collisions
    tt = rng.integers(0, 2, (B, S)).astype(np.int32)
    seed, site, step = 99, 2, 11
    sp = step_ptr(step)
    M = B * S
    y, z, mean, rstd = new((B, S, H), BF16), new((M, H), F32), new((M,), F32), new((M,), F32)
    dp = {k: T(v) for k, v in P.items()}
    ids_t, tt_t = T(ids, I32), T(tt, I32)
    call("polus_embed_ln_fwd", ids_t.ptr, tt_t.ptr, dp["word"].ptr, dp["pos"].ptr, dp["type"].ptr, dp["emb_ln_g"].ptr,
         dp["emb_ln_b"].ptr, B, S, H, V, 2, 1e-12, p, seed, site, sp, y.ptr, z.ptr, mean.ptr, rstd.ptr, st())
    mask = philox.dropout_scale_mask((B, S, H), p, seed, site, step) if p > 0 else None
    P64 = {k: v.astype(np.float64) for k, v in P.items()}
    y_ref, cache = R.bert_embeddings_fwd(ids, tt, P64, mask)
    np.testing.assert_allclose(y.numpy(), y_ref, atol=3 * BF16_EPS * (1 + np.abs(y_ref).max()), rtol=0)
    dy = dev.bf16_round(rng.standard_normal((B, S, H)).astype(np.float32))
    g = {k: new(v.shape, F32) for k, v in P.items()}
    ws = new((int(call("polus_embed_ws_floats", B, S, H)),), F32)
    call("polus_embed_ln_bwd", T(dy, BF16).ptr, z.ptr, mean.ptr, rstd.ptr, dp["emb_ln_g"].ptr, ids_t.ptr, tt_t.ptr, B, S, H,
         V, 2, p, seed, site, sp, g["word"].ptr, g["pos"].ptr, g["type"].ptr, g["emb_ln_g"].ptr, g["emb_ln_b"].ptr, ws.ptr, st())
    g_ref = R.bert_embeddings_bwd(dy.astype(np.float64), cache, P64)
    for k in P:
        ref = g_ref[k]
        np.testing.assert_allclose(g[k].numpy(), ref, rtol=1e-4, atol=1e-4 * (np.abs(ref).max() + 1e-6), err_msg=k)


@pytest.mark.parametrize("B,nh,S,p,use_mask", [(2, 2, 64, 0.0, True), (1, 3, 256, 0.1, True), (2, 1, 512, 0.0, False), (1, 2, 40, 0.1, True)])
def test_softmax_fwd_bwd(dev, B, nh, S, p, use_mask):
    from oracle import numpy_ref as R, philox
    from polus_b200.tensor import BF16, I32
    rng = np.random.default_rng(S)
    scores = dev.bf16_round(rng.standard_normal((B, nh, S, S)).astype(np.float32) * 4)
    lens = rng.integers(S // 2, S + 1, B)
    mask = (np.arange(S)[None] < lens[:, None]).astype(np.int32)
    scale = 0.125
    seed, site, step = 7, 3, 2
    sp = step_ptr(step)
    s_t = T(scores, BF16)
    P_t = s_t
    Pd_t = new(scores.shape, BF16) if p > 0 else P_t
    call("polus_softmax_fwd", s_t.ptr, T(mask, I32).ptr if use_mask else None, B, nh, S, S, scale, p, seed, site, sp,
         P_t.ptr, Pd_t.ptr, st())
    add = R.attention_mask_additive(mask) if use_mask else 0.0
    P_ref = R.softmax(scores.astype(np.float64) * scale + add)
    P_dev = P_t.numpy()
    np.testing.assert_allclose(P_dev, P_ref, atol=2 * BF16_EPS, rtol=0)
    dm = philox.dropout_scale_mask(scores.shape, p, seed, site, step) if p > 0 else np.ones_like(scores)
    np.testing.assert_allclose(Pd_t.numpy(), dev.bf16_round((P_dev * dm).astype(np.float32)), atol=2 * BF16_EPS, rtol=0)
    dPd = dev.bf16_round(rng.standard_normal(scores.shape).astype(np.float32))
    dP_t = T(dPd, BF16)
    call("polus_softmax_bwd", P_t.ptr, dP_t.ptr, B, nh, S, S, scale, p, seed, site, sp, st())
    dP = dPd.astype(np.float64) * dm
    dS_ref = scale * P_dev * (dP - (P_dev * dP).sum(-1, keepdims=True))
    np.testing.assert_allclose(dP_t.numpy(), dS_ref, atol=3 * BF16_EPS * np.abs(dS_ref).max() + 1e-6, rtol=2 * BF16_EPS)
    if p > 0:  # P buffer now holds the dropped probabilities
        np.testing.assert_allclose(P_t.numpy(), dev.bf16_round((P_dev * dm).astype(np.float32)), atol=2 * BF16_EPS, rtol=0)


@pytest.mark.parametrize("act", ["gelu", "swish", "relu", "tanh", "mish", None])
def test_act_bwd_colsum(dev, act):
    from oracle import numpy_ref as R
    from polus_b200 import _lib
    from polus_b200.tensor import BF16, F32
    rng = np.random.default_rng(3)
    M, N = 333, 520
    dy = dev.bf16_round(rng.standard_normal((M, N)).astype(np.float32))
    z = dev.bf16_round(rng.standard_normal((M, N)).astype(np.float32) * 2)
    dz_t, gb = new((M, N), BF16), T(np.full(N, 0.5, np.float32))
    code = _lib.ACT[act]
    call("polus_act_bwd_colsum", T(dy, BF16).ptr, T(z, BF16).ptr, M, N, code, dz_t.ptr if code else None, gb.ptr, None, st())
    ref = dy.astype(np.float64) * R.ACT[act][1](z.astype(np.float64))
    if code:
        np.testing.assert_allclose(dz_t.numpy(), ref, atol=2 * BF16_EPS * (np.abs(ref).max() + 1), rtol=0)
    np.testing.assert_allclose(gb.numpy(), 0.5 + ref.sum(0), rtol=2e-3, atol=2e-2)
    if code:  # the derivative supplied directly (what the forward GEMM stores with c2_kind = 1)
        d = dev.bf16_round(R.ACT[act][1](z.astype(np.float64)).astype(np.float32))
        gb2 = T(np.zeros(N, np.float32))
        call("polus_act_bwd_colsum", T(dy, BF16).ptr, T(d, BF16).ptr, M, N, _lib.ACT_DERIV, dz_t.ptr, gb2.ptr, None, st())
        ref2 = dy.astype(np.float64) * d
        np.testing.assert_allclose(dz_t.numpy(), ref2, atol=2 * BF16_EPS * (np.abs(ref2).max() + 1), rtol=0)
        np.testing.assert_allclose(gb2.numpy(), ref2.sum(0), rtol=2e-3, atol=2e-2)


# -------------------------------------------------------------------------------------------------- CRF
@pytest.mark.parametrize("B,Tn,K,ragged,weighted", [(4, 256, 4, False, False), (5, 33, 4, True, True), (3, 1, 4, False, False),
                                                    (2, 50, 9, True, False), (2, 12, 32, True, True),
                                                    # K = 4 with T > 851: four sequences overflow shared memory, one tag per lane
                                                    (2, 1000, 4, True, False)])
def test_crf_nll_and_grads(dev, B, Tn, K, ragged, weighted):
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32, I32
    rng = np.random.default_rng(B * Tn + K)
    emis = rng.standard_normal((B, Tn, K)).astype(np.float32) * 2
    tags = rng.integers(0, K, (B, Tn)).astype(np.int32)
    trans = rng.standard_normal((K, K)).astype(np.float32)
    lens = rng.integers(0 if ragged else Tn, Tn + 1, B).astype(np.int32) if ragged else np.full(B, Tn, np.int32)
    w = rng.uniform(0.2, 2.0, B).astype(np.float32) if weighted else None
    nll, loss, gem, gtr = new((B,), F32), new((), F32), new((B, Tn, K), F32), T(np.zeros((K, K), np.float32))
    call("polus_crf_nll", T(emis).ptr, T(tags, I32).ptr, T(lens, I32).ptr if ragged else None, T(trans).ptr,
         T(w).ptr if weighted else None, B, Tn, K, nll.ptr, loss.ptr, gem.ptr, gtr.ptr, st())
    nll_r, loss_r, gem_r, gtr_r = R.crf_nll_with_grads(emis.astype(np.float64), tags, lens, trans.astype(np.float64), w)
    np.testing.assert_allclose(nll.numpy(), nll_r, rtol=2e-5, atol=2e-4)
    np.testing.assert_allclose(float(loss), loss_r, rtol=2e-5, atol=1e-5)
    # fp32 forward-backward over T steps vs the fp64 oracle: error ~ T * eps_fp32 * |log-space magnitude|
    np.testing.assert_allclose(gem.numpy(), gem_r, rtol=2e-3, atol=1e-3 * np.abs(gem_r).max() + 1e-6)
    np.testing.assert_allclose(gtr.numpy(), gtr_r, rtol=2e-3, atol=1e-3 * np.abs(gtr_r).max() + 1e-5)
    # the log-likelihood itself equals tfa.text.crf_log_likelihood's definition
    np.testing.assert_allclose(-nll.numpy(), R.crf_log_likelihood(emis.astype(np.float64), tags, lens, trans.astype(np.float64)),
                               rtol=2e-5, atol=2e-4)


@pytest.mark.parametrize("B,Tn,K,ragged", [(8, 256, 4, False), (6, 77, 4, True), (3, 1, 4, False), (4, 40, 32, True), (2, 512, 4, False)])
def test_viterbi_bit_exact(dev, B, Tn, K, ragged):
    """Index work: decoded paths must equal the oracle's exactly (ties -> lowest index), given identical emissions."""
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32, I32
    rng = np.random.default_rng(Tn + K)
    # quantised emissions/transitions => many exact ties, and fp32 sums that are exact in both implementations
    emis = (rng.integers(-4, 5, (B, Tn, K)) * 0.5).astype(np.float32)
    trans = (rng.integers(-2, 3, (K, K)) * 0.5).astype(np.float32)
    lens = rng.integers(0, Tn + 1, B).astype(np.int32) if ragged else np.full(B, Tn, np.int32)
    tags, score = new((B, Tn), I32), new((B,), F32)
    call("polus_crf_decode", T(emis).ptr, T(lens, I32).ptr if ragged else None, T(trans).ptr, B, Tn, K, tags.ptr, score.ptr, st())
    tags_r, score_r = R.crf_decode(emis, lens, trans)
    assert np.array_equal(tags.numpy(), tags_r)
    assert np.array_equal(score.numpy(), score_r.astype(np.float32))
    # random real-valued case too
    emis = rng.standard_normal((B, Tn, K)).astype(np.float32)
    trans = rng.standard_normal((K, K)).astype(np.float32)
    call("polus_crf_decode", T(emis).ptr, T(lens, I32).ptr if ragged else None, T(trans).ptr, B, Tn, K, tags.ptr, score.ptr, st())
    tags_r, _ = R.crf_decode(emis, lens, trans)
    assert np.array_equal(tags.numpy(), tags_r)


def test_crf_mask_and_sample_weights(dev):
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32
    rng = np.random.default_rng(1)
    K = 4
    trans = rng.standard_normal((K, K)).astype(np.float32)
    mask = np.ones((K, K), np.float32)
    mask[1, 3] = 0  # O -> I-Chemical forbidden: the only concrete mask in the reference (tests/test_utils.py:77)
    out = new((K, K), F32)
    call("polus_crf_mask_transitions", T(trans).ptr, T(mask).ptr, K, out.ptr, st())
    assert np.array_equal(out.numpy(), R.crf_masked_transitions(trans, mask))
    B, Tn = 6, 20
    tags = rng.integers(0, 2, (B, Tn))
    tags[0] = 1
    tags[2, 5] = 2
    tags[4, 7] = 3
    y = np.eye(K, dtype=np.float32)[tags]
    mp = np.array([0, 0, 1, 1], np.float32)
    w = new((B,), F32)
    call("polus_crf_sample_weights", T(y).ptr, T(mp).ptr, 0.25, B, Tn, K, w.ptr, st())
    assert np.array_equal(w.numpy(), R.crf_sample_weights(y, mp, 0.25))


# -------------------------------------------------------------------------------------------------- losses
@pytest.mark.parametrize("rows,Cn", [(128, 10), (1000, 4), (7, 33), (0, 5)])
def test_cross_entropy_family(dev, rows, Cn):
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32, I32
    rng = np.random.default_rng(rows + Cn)
    logits = (rng.standard_normal((rows, Cn)) * 3).astype(np.float32)
    labels = rng.integers(0, Cn, rows).astype(np.int32)
    cw = rng.uniform(0.5, 2, Cn).astype(np.float32)
    loss, g = new((), F32), new((rows, Cn), F32)
    call("polus_xent", 0, T(logits).ptr, T(labels, I32).ptr, None, 0.0, rows, Cn, loss.ptr, g.ptr, st())
    if rows == 0:
        assert float(loss) == 0.0
        return
    lr, gr = R.sparse_softmax_xent(logits.astype(np.float64), labels)
    np.testing.assert_allclose(float(loss), lr, rtol=1e-5)
    np.testing.assert_allclose(g.numpy(), gr, rtol=1e-4, atol=1e-7)
    y = np.eye(Cn, dtype=np.float32)[labels]
    call("polus_xent", 1, T(logits).ptr, T(y).ptr, T(cw).ptr, 0.0, rows, Cn, loss.ptr, g.ptr, st())
    lr, gr = R.weighted_softmax_xent(logits.astype(np.float64), y.astype(np.float64), cw)
    np.testing.assert_allclose(float(loss), lr, rtol=1e-5)
    np.testing.assert_allclose(g.numpy(), gr, rtol=1e-4, atol=1e-7)
    ym = (rng.uniform(size=(rows, Cn)) < 0.2).astype(np.float32)
    ym[0] = 0
    call("polus_xent", 2, T(logits).ptr, T(ym).ptr, T(cw).ptr, 0.3, rows, Cn, loss.ptr, g.ptr, st())
    lr, gr = R.weighted_sigmoid_xent(logits.astype(np.float64), ym.astype(np.float64), cw, 0.3)
    np.testing.assert_allclose(float(loss), lr, rtol=1e-5)
    np.testing.assert_allclose(g.numpy(), gr, rtol=1e-4, atol=1e-7)


# -------------------------------------------------------------------------------------------------- optimizer
@pytest.mark.parametrize("n,schedule,wd", [(1000003, 0, 0.0), (4096, 1, 0.0), (777, 0, 0.01)])
def test_adam_matches_keras_formula(dev, n, schedule, wd):
    from oracle import numpy_ref as R
    from polus_b200 import _lib
    from polus_b200.tensor import BF16, F32, U8
    rng = np.random.default_rng(n)
    p0 = rng.standard_normal(n).astype(np.float32)
    p, m, v = T(p0), new((n,), F32), new((n,), F32)
    pb = new((n,), BF16)
    decay = (rng.uniform(size=n) < 0.5).astype(np.uint8)
    g_t = new((n,), F32)
    cfg = _lib.AdamCfg(lr=1e-2, schedule=schedule, warmup_steps=2, decay_steps=8, end_lr=1e-7, beta1=0.9, beta2=0.999,
                       eps=1e-7, weight_decay=wd, grad_scale=0.5)
    sp = step_ptr(0)
    pr, mr, vr = p0.astype(np.float64), np.zeros(n), np.zeros(n)
    for t in range(1, 5):
        g = rng.standard_normal(n).astype(np.float32)
        dev.upload(g_t.ptr, g)
        call("polus_adam", p.ptr, g_t.ptr, m.ptr, v.ptr, pb.ptr, T(decay, U8).ptr if wd > 0 else None, n, C.byref(cfg), None, sp, 1, st())
        lr = R.warmup_schedule_lr(t - 1, 10, 1e-2, 0.2) if schedule else 1e-2
        if wd > 0:
            pr = np.where(decay == 1, pr - lr * wd * pr, pr)
        pr, mr, vr = R.adam_step(pr, g.astype(np.float64) * 0.5, mr, vr, t, lr)
        np.testing.assert_allclose(p.numpy(), pr, rtol=2e-5, atol=2e-6)
        assert not g_t.numpy().any(), "adam must zero the consumed gradients"
        np.testing.assert_array_equal(pb.numpy(), dev.bf16_round(p.numpy()))
    assert int(dev.download(sp, (1,), np.uint32)[0]) == 4


# -------------------------------------------------------------------------------------------------- small utilities
def test_argmax_onehot_confusion_bit_exact(dev):
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32, I32
    rng = np.random.default_rng(0)
    x = rng.integers(-3, 4, (1000, 7)).astype(np.float32)  # plenty of ties
    out = new((1000,), I32)
    call("polus_argmax_f32", T(x).ptr, 1000, 7, out.ptr, st())
    assert np.array_equal(out.numpy(), x.argmax(-1).astype(np.int32))
    oh = new((1000, 7), F32)
    call("polus_one_hot_f32", out.ptr, 1000, 7, oh.ptr, st())
    assert np.array_equal(oh.numpy(), np.eye(7, dtype=np.float32)[x.argmax(-1)])
    yt, yp = rng.integers(0, 10, 50000).astype(np.int32), rng.integers(0, 10, 50000).astype(np.int32)
    cm = new((10, 10), I32)
    call("polus_confusion_matrix", T(yt, I32).ptr, T(yp, I32).ptr, 50000, 10, cm.ptr, st())
    assert np.array_equal(cm.numpy(), R.confusion_matrix(yt, yp, 10))


def test_gemm_tc_vs_checker_and_host(dev):
    """tcgen05 GEMM vs the CUDA-core checker on device and numpy on host, all major combinations."""
    from polus_b200 import _lib
    from polus_b200.tensor import BF16, F32
    rng = np.random.default_rng(11)
    for (M, N, K, a_mn, b_mn, split) in [(128, 128, 64, 0, 0, 1), (200, 136, 200, 0, 1, 1), (328, 72, 520, 1, 1, 1),
                                         (256, 256, 1024, 1, 1, 4), (96, 64, 64, 1, 0, 1), (512, 768, 256, 0, 1, 1)]:
        A = dev.bf16_round(rng.standard_normal((K, M) if a_mn else (M, K)).astype(np.float32))
        B = dev.bf16_round(rng.standard_normal((K, N) if b_mn else (N, K)).astype(np.float32) * 0.1)
        bias = rng.standard_normal(N).astype(np.float32)
        a_t, b_t, bias_t = T(A, BF16), T(B, BF16), T(bias)
        c_t, r_t = new((M, N), F32), new((M, N), F32)
        g = _lib.Gemm()
        g.M, g.N, g.K, g.batch0, g.batch1 = M, N, K, 1, 1
        g.A = _lib.Operand(a_t.ptr, M if a_mn else K, 0, 0, a_mn, _lib.BF16)
        g.B = _lib.Operand(b_t.ptr, N if b_mn else K, 0, 0, b_mn, _lib.BF16)
        g.C, g.ldc, g.c_dtype, g.bias, g.alpha, g.act = c_t.ptr, N, _lib.F32, bias_t.ptr, 1.0, 0
        g.accumulate, g.split_k = (1 if split > 1 else 0), split
        call("polus_gemm_tc", C.byref(g), st())
        g.C, g.accumulate, g.split_k = r_t.ptr, 0, 1
        call("polus_gemm_small", C.byref(g), st())
        host = (A.T if a_mn else A).astype(np.float64) @ (B if b_mn else B.T).astype(np.float64) + bias
        np.testing.assert_allclose(c_t.numpy(), host, rtol=1e-4, atol=1e-4 * np.abs(host).max())
        np.testing.assert_allclose(r_t.numpy(), host, rtol=1e-4, atol=1e-4 * np.abs(host).max())


@pytest.mark.parametrize("M,N,K,a_mn,b_mn,f32", [(32768, 768, 192, 0, 0, 0), (32768, 768, 136, 0, 1, 0), (32700, 576, 200, 0, 0, 1),
                                                  (32768, 768, 64, 1, 1, 0), (32768, 576, 128, 1, 0, 0), (32768, 768, 3072, 0, 1, 0)])
def test_gemm_tc_pair_tiles_ragged_shapes(dev, M, N, K, a_mn, b_mn, f32):
    """Pair tiles on N = 768 / 576 outputs at about 32768 rows: both operand majors, bias, bf16 and fp32 outputs, ragged
    M, K and N (576 is not a multiple of 256), column sums -- against numpy fp64."""
    from polus_b200 import _lib
    from polus_b200.tensor import BF16, F32, Tensor
    rng = np.random.default_rng(M + N + K + a_mn)
    A = dev.bf16_round(rng.standard_normal((K, M) if a_mn else (M, K)).astype(np.float32))
    B = dev.bf16_round(rng.standard_normal((K, N) if b_mn else (N, K)).astype(np.float32) * 0.1)
    bias = rng.standard_normal(N).astype(np.float32)
    a_t, b_t, bias_t = Tensor.from_numpy(A, BF16), Tensor.from_numpy(B, BF16), Tensor.from_numpy(bias, F32)
    c_t = Tensor((M, N), F32 if f32 else BF16)
    cs_t = Tensor.from_numpy(np.zeros(N, np.float32), F32)
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = M, N, K, 1, 1
    g.A = _lib.Operand(a_t.ptr, M if a_mn else K, 0, 0, a_mn, _lib.BF16)
    g.B = _lib.Operand(b_t.ptr, N if b_mn else K, 0, 0, b_mn, _lib.BF16)
    g.C, g.ldc, g.c_dtype, g.bias, g.alpha, g.act = c_t.ptr, N, (_lib.F32 if f32 else _lib.BF16), bias_t.ptr, 1.0, 0
    g.accumulate, g.split_k = 0, 1
    if not f32:
        g.colsum = cs_t.ptr
    _lib.call("polus_gemm_tc", C.byref(g), st())
    host = (A.T if a_mn else A).astype(np.float64) @ (B if b_mn else B.T).astype(np.float64) + bias
    out = c_t.numpy().astype(np.float64)
    scale = np.abs(host).max()
    if f32:
        np.testing.assert_allclose(out, host, rtol=1e-4, atol=1e-4 * scale)
    else:
        np.testing.assert_allclose(out, host, rtol=1e-2, atol=1e-2 * scale)
        np.testing.assert_allclose(cs_t.numpy(), out.sum(0), rtol=1e-4, atol=1e-4 * np.abs(out).sum(0).max())


@pytest.mark.parametrize("M,N,K,cg", [(512, 768, 256, 2), (300, 200, 136, 2), (8192, 3072, 768, 2), (128, 320, 64, 1), (77, 72, 520, 1)])
def test_gemm_tc_fused_activation_backward(dev, M, N, K, cg):
    """The two epilogue modes that replace GeluGrad + BiasAddGrad (polus_gemm_t.c2_kind / Emul / colsum):
    forward  C = gelu(A.B^T + bias), C2 = gelu'(A.B^T + bias);
    backward C = (A.B^T) * Emul, colsum += column sums of C  -- against numpy (fp64) and the CUDA-core checker."""
    from oracle import numpy_ref as R
    from polus_b200 import _lib
    from polus_b200.tensor import BF16, F32
    rng = np.random.default_rng(M + N + K)
    A = dev.bf16_round(rng.standard_normal((M, K)).astype(np.float32))
    B = dev.bf16_round(rng.standard_normal((N, K)).astype(np.float32) * (1.5 / np.sqrt(K)))
    bias = (0.1 * rng.standard_normal(N)).astype(np.float32)
    a_t, b_t, bias_t = T(A, BF16), T(B, BF16), T(bias)
    y_t, d_t = new((M, N), BF16), new((M, N), BF16)
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = M, N, K, 1, 1
    g.A = _lib.Operand(a_t.ptr, K, 0, 0, 0, _lib.BF16)
    g.B = _lib.Operand(b_t.ptr, K, 0, 0, 0, _lib.BF16)
    g.C, g.ldc, g.c_dtype, g.bias, g.alpha, g.act = y_t.ptr, N, _lib.BF16, bias_t.ptr, 1.0, _lib.ACT["gelu"]
    g.C2, g.c2_kind, g.split_k = d_t.ptr, 1, 1
    call("polus_gemm_tc", C.byref(g), st())
    z = A.astype(np.float64) @ B.T.astype(np.float64) + bias
    np.testing.assert_allclose(y_t.numpy(), R.ACT["gelu"][0](z), atol=2 * BF16_EPS * (np.abs(z).max() + 1), rtol=0)
    np.testing.assert_allclose(d_t.numpy(), R.ACT["gelu"][1](z), atol=2 * BF16_EPS * 1.2, rtol=0)
    # backward form: multiplier tile + column sums
    E = dev.bf16_round(rng.standard_normal((M, N)).astype(np.float32))
    e_t = T(E, BF16)
    c_t, r_t = new((M, N), BF16), new((M, N), BF16)
    cs_t, cs_r = T(np.full(N, 0.25, np.float32)), T(np.full(N, 0.25, np.float32))
    g.C, g.C2, g.c2_kind, g.bias, g.act = c_t.ptr, None, 0, None, 0
    g.Emul, g.colsum = e_t.ptr, cs_t.ptr
    call("polus_gemm_tc", C.byref(g), st())
    g.C, g.colsum = r_t.ptr, cs_r.ptr
    call("polus_gemm_small", C.byref(g), st())
    ref = (A.astype(np.float64) @ B.T.astype(np.float64)) * E
    tol = 2 * BF16_EPS * (np.abs(ref).max() + 1)
    np.testing.assert_allclose(c_t.numpy(), ref, atol=tol, rtol=0)
    np.testing.assert_allclose(r_t.numpy(), ref, atol=tol, rtol=0)
    cs_ref = 0.25 + c_t.numpy().astype(np.float64).sum(0)  # the column sums are those of the stored (bf16) values
    np.testing.assert_allclose(cs_t.numpy(), cs_ref, rtol=1e-4, atol=1e-4 * (np.abs(cs_ref).max() + 1))
    np.testing.assert_allclose(cs_r.numpy(), 0.25 + r_t.numpy().astype(np.float64).sum(0), rtol=1e-4, atol=1e-4 * (np.abs(cs_ref).max() + 1))


@pytest.mark.parametrize("M,N,K", [(8192, 3072, 768), (5000, 1536, 256)])
def test_gemm_tc_gelu_derivative_as_8bit_fixed_point(dev, M, N, K):
    """polus_gemm_t.c2_kind = 2: the FFN-up GEMM stores gelu' as one byte per element, q = 28 + round(200 gelu'), and the
    dgrad GEMM of the next layer (or polus_act_bwd_colsum, when that GEMM cannot fuse it) multiplies by (q - 28) * 0.005.
    Bars: decoded derivative within half a step (0.0025) + fp32 noise of numpy's gelu'; products against the DECODED
    derivative within the bf16 output tolerance; problems the 16-warp kernel does not take are reported as unsupported."""
    from oracle import numpy_ref as R
    from polus_b200 import _lib
    from polus_b200.tensor import BF16, F32, U8
    rng = np.random.default_rng(M + N + K)
    A = dev.bf16_round(rng.standard_normal((M, K)).astype(np.float32))
    B = dev.bf16_round(rng.standard_normal((N, K)).astype(np.float32) * (1.5 / np.sqrt(K)))
    bias = (0.1 * rng.standard_normal(N)).astype(np.float32)
    a_t, b_t, bias_t = T(A, BF16), T(B, BF16), T(bias)
    y_t, d_t = new((M, N), BF16), new((M, N), U8)
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = M, N, K, 1, 1
    g.A = _lib.Operand(a_t.ptr, K, 0, 0, 0, _lib.BF16)
    g.B = _lib.Operand(b_t.ptr, K, 0, 0, 0, _lib.BF16)
    g.C, g.ldc, g.c_dtype, g.bias, g.alpha, g.act = y_t.ptr, N, _lib.BF16, bias_t.ptr, 1.0, _lib.ACT["gelu"]
    g.C2, g.c2_kind, g.split_k = d_t.ptr, 2, 1
    assert call("polus_gemm_tc_supported", C.byref(g)) == 1
    call("polus_gemm_tc", C.byref(g), st())
    z = A.astype(np.float64) @ B.T.astype(np.float64) + bias
    np.testing.assert_allclose(y_t.numpy(), R.ACT["gelu"][0](z), atol=2 * BF16_EPS * (np.abs(z).max() + 1), rtol=0)
    q = d_t.numpy().astype(np.float64)
    assert q.min() >= 2 and q.max() <= 254
    dec = (q - 28.0) * 0.005
    np.testing.assert_allclose(dec, R.ACT["gelu"][1](z), atol=0.0025 + 2e-4, rtol=0)
    # backward: C = (dY . W^T) * decoded derivative, column sums of the stored values
    c_t = new((M, N), BF16)
    cs_t = T(np.full(N, 0.25, np.float32))
    g.C, g.C2, g.bias, g.act = c_t.ptr, None, None, 0
    g.Emul, g.colsum = d_t.ptr, cs_t.ptr
    assert call("polus_gemm_tc_supported", C.byref(g)) == 1
    call("polus_gemm_tc", C.byref(g), st())
    prod = A.astype(np.float64) @ B.T.astype(np.float64)
    ref = prod * dec
    np.testing.assert_allclose(c_t.numpy(), ref, atol=2 * BF16_EPS * (np.abs(ref).max() + 1), rtol=0)
    cs_ref = 0.25 + c_t.numpy().astype(np.float64).sum(0)
    np.testing.assert_allclose(cs_t.numpy(), cs_ref, rtol=1e-4, atol=1e-4 * (np.abs(cs_ref).max() + 1))
    # the unfused route: dz = dy * decoded derivative + bias-gradient column sums
    dy = dev.bf16_round(rng.standard_normal((M, N)).astype(np.float32))
    dz_t, gb_t = new((M, N), BF16), T(np.zeros(N, np.float32))
    call("polus_act_bwd_colsum", T(dy, BF16).ptr, d_t.ptr, M, N, _lib.ACT_DERIV_U8, dz_t.ptr, gb_t.ptr, None, st())
    np.testing.assert_allclose(dz_t.numpy(), dy * dec, atol=2 * BF16_EPS * 6, rtol=0)
    np.testing.assert_allclose(gb_t.numpy(), (dy * dec).sum(0), rtol=1e-2, atol=1e-2 * np.sqrt(M))
    # a shape the 16-warp pair kernel does not take (one 128-row tile) must say so instead of misreading the bytes
    g.M = 128
    assert call("polus_gemm_tc_supported", C.byref(g)) == 0


@pytest.mark.parametrize("M,K,N,act,xdt", [(8192, 128, 4, None, "bf16"), (128, 128, 10, None, "bf16"), (333, 768, 3, "swish", "f32"),
                                           (50, 40, 32, "relu", "f32"), (0, 128, 4, None, "bf16")])
def test_skinny_linear_fwd_bwd(dev, M, K, N, act, xdt):
    """Narrow dense layer (tag projection, polus/ner/models.py:37) vs numpy."""
    from oracle import numpy_ref as R
    from polus_b200 import _lib
    from polus_b200.tensor import BF16, F32
    rng = np.random.default_rng(M + K + N)
    x = dev.bf16_round(rng.standard_normal((M, K)).astype(np.float32))
    W = (rng.standard_normal((K, N)) * 0.2).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    dt = BF16 if xdt == "bf16" else F32
    assert call("polus_skinny_supported", K, N) == 1
    x_t, W_t, b_t = T(x, dt), T(W), T(b)
    y, z = new((M, N), F32), new((M, N), F32)
    code = _lib.ACT[act]
    call("polus_skinny_fwd", x_t.ptr, dt, W_t.ptr, b_t.ptr, M, K, N, code, y.ptr, z.ptr, st())
    if M == 0:
        return
    zr = x.astype(np.float64) @ W + b
    np.testing.assert_allclose(z.numpy(), zr, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(y.numpy(), R.ACT[act][0](zr), rtol=1e-4, atol=1e-4)
    dz = rng.standard_normal((M, N)).astype(np.float32)
    gW, gb = T(np.full((K, N), 0.25, np.float32)), T(np.full(N, -1.0, np.float32))
    dx = new((M, K), dt)
    call("polus_skinny_bwd", x_t.ptr, dt, W_t.ptr, T(dz).ptr, M, K, N, dx.ptr, dt, gW.ptr, gb.ptr, st())
    np.testing.assert_allclose(gW.numpy(), 0.25 + x.astype(np.float64).T @ dz, rtol=1e-3, atol=1e-3 * max(1, M ** 0.5))
    np.testing.assert_allclose(gb.numpy(), -1.0 + dz.sum(0), rtol=1e-3, atol=1e-3 * max(1, M ** 0.5))
    dxr = dz.astype(np.float64) @ W.T
    np.testing.assert_allclose(dx.numpy(), dxr, rtol=1e-2 if dt == BF16 else 1e-4, atol=2e-2 if dt == BF16 else 1e-4)


@pytest.mark.parametrize("B,nh,S,p,use_mask", [(2, 2, 64, 0.0, True), (1, 3, 256, 0.1, True), (2, 2, 128, 0.0, False),
                                               (1, 2, 192, 0.1, True), (3, 1, 32, 0.0, True), (2, 2, 96, 0.1, False),
                                               (2, 2, 224, 0.1, True), (1, 2, 160, 0.0, False), (1, 1, 256, 0.1, False),
                                               # S > 256: four key segments forward; two query halves per head backward
                                               # (K / V stages refilled, dK / dV partial sums reduce-added by the TMA unit)
                                               (2, 2, 512, 0.1, True), (1, 3, 512, 0.0, False), (2, 1, 384, 0.1, True),
                                               (1, 2, 288, 0.0, True), (1, 2, 448, 0.1, False), (3, 2, 320, 0.1, True)])
def test_fused_attention_fwd_bwd(dev, B, nh, S, p, use_mask):
    """Fused attention (scores/probabilities in TMEM/smem) vs the oracle with the device's own dropout masks, and vs
    the unfused GEMM+softmax path (same Philox counters => same masks)."""
    from tests.attention_ref import check_attention_case
    check_attention_case(dev, B, nh, S, p, use_mask)


def test_attention_fwd_keepbits_bit_exact(dev):
    """The fused forward writes into `keepbits` exactly the dropout decisions the oracle's Philox4x32-10 gives for
    (seed, site, step), at an even and an odd step: the backward kernel reads them from there."""
    from oracle import philox
    from polus_b200.tensor import BF16, F32, I32
    B, S, nh, p, seed, site = 2, 128, 3, 0.1, 991, 4
    H = nh * 64
    words = int(call("polus_attention_keepbits_words", B, S, nh))
    assert words == B * nh * S * S // 32
    rng = np.random.default_rng(0)
    qkv = T(dev.bf16_round(rng.standard_normal((B, S, 3 * H)).astype(np.float32)), BF16)
    for step in (6, 7):
        keep = philox.dropout_keep_mask(B * nh * S * S, p, seed, site, step).reshape(-1, 32)
        want = (keep.astype(np.uint32) << np.arange(32, dtype=np.uint32)).sum(1, dtype=np.uint64).astype(np.uint32)
        ctx, lse, kb = new((B, S, H), BF16), new((B, nh, S), F32), new((words,), I32)
        call("polus_attention_fwd", qkv.ptr, None, B, S, nh, 64, p, seed, site, step_ptr(step), ctx.ptr, lse.ptr, kb.ptr, st())
        assert np.array_equal(kb.numpy().view(np.uint32), want)
