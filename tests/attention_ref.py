"""Self-attention forward and backward through ops.attention / ops._attention_unfused against the fp64 oracle, with the
device's own dropout masks (Philox site 1 of the step): shared by the fused-kernel tests and the shapes only the GEMM +
softmax path serves."""
import numpy as np


def attention_oracle(qkv, dctx, mask, nh, dh, p, seed, site, step):
    """ctx and d(qkv) of softmax(Q K^T / sqrt(dh) + (1 - mask) * -10000) V in float64 (mask None: no mask)."""
    from oracle import numpy_ref as R, philox
    B, S, _ = qkv.shape
    H = nh * dh
    q, k, v = [qkv[..., i * H:(i + 1) * H].reshape(B, S, nh, dh).transpose(0, 2, 1, 3).astype(np.float64) for i in range(3)]
    scale = 1.0 / np.sqrt(dh)
    sc = q @ k.transpose(0, 1, 3, 2) * scale + (R.attention_mask_additive(mask) if mask is not None else 0.0)
    P = R.softmax(sc)
    dm = philox.dropout_scale_mask((B, nh, S, S), p, seed, site, step).astype(np.float64) if p > 0 else 1.0
    Pd = P * dm
    ctx = (Pd @ v).transpose(0, 2, 1, 3).reshape(B, S, H)
    do = dctx.reshape(B, S, nh, dh).transpose(0, 2, 1, 3).astype(np.float64)
    dPd = do @ v.transpose(0, 1, 3, 2)
    dv = Pd.transpose(0, 1, 3, 2) @ do
    dP = dPd * dm
    dS = P * (dP - (P * dP).sum(-1, keepdims=True)) * scale
    dq, dk = dS @ k, dS.transpose(0, 1, 3, 2) @ q
    dqkv = np.concatenate([t.transpose(0, 2, 1, 3).reshape(B, S, H) for t in (dq, dk, dv)], -1)
    return ctx, dqkv


def assert_no_gain(out, ref, what):
    """dQ and dK are linear in the softmax scale, and bf16 rounding is unbiased: their least-squares gain against the
    oracle is 1 within about 6e-4 on these shapes (B200, without dropout).  A scale off by 2^-10 moves it by 1e-3 to
    2e-3 while hiding under the elementwise bars."""
    ref = ref.astype(np.float64).ravel()
    gain = float(np.dot(out.astype(np.float64).ravel(), ref) / np.dot(ref, ref))
    assert abs(gain - 1.0) <= 2.0 ** -10, f"{what}: gain {gain:.6f} against the oracle"


def check_attention_case(dev, B, nh, S, p, use_mask, dh=64, lens=None, fused=True, seed=None):
    """fused: ops.attention on the fused kernels (QKV bias gradient included) and ops._attention_unfused, both against the
    oracle.  Otherwise ops.attention on a shape the fused kernels do not take, against the oracle, plus the gain check."""
    from polus_b200 import ops
    from polus_b200.tensor import BF16, I32, Param, Tensor
    rng = np.random.default_rng(S + nh if seed is None else seed)
    H = nh * dh
    qkv = dev.bf16_round(rng.standard_normal((B, S, 3 * H)).astype(np.float32))
    dctx = dev.bf16_round(rng.standard_normal((B, S, H)).astype(np.float32))
    if lens is None:
        lens = rng.integers(max(S // 2, 1), S + 1, B)
    mask = (np.arange(S)[None] < np.asarray(lens)[:, None]).astype(np.int32)
    ops.set_seed(77)
    ops.set_step(3)
    bias = Param(np.zeros(3 * H, np.float32), name="qkv_bias")  # only its .grad is touched

    def run(which):
        ops.reset_dropout_sites()
        x = Tensor.from_numpy(qkv, BF16)
        x.requires_grad = True
        m = Tensor.from_numpy(mask, I32) if use_mask else None
        with ops.GradientTape() as tape:
            if which == "unfused":
                ctx = ops._attention_unfused(x, m, nh, p)
            else:
                ctx = ops.attention(x, m, nh, p, qkv_bias=bias if fused else None)
        # seed the backward with dctx: d(sum(ctx*dctx))
        tape.nodes[-1].output = ctx
        g = tape.nodes[-1].backward(Tensor.from_numpy(dctx, BF16))[0]
        return ctx.numpy(), g.numpy()

    ctx_r, dqkv_r = attention_oracle(qkv, dctx, mask if use_mask else None, nh, dh, p, 77, 1, 3)
    tol_c, tol_g = 2e-2 * np.abs(ctx_r).max(), 2e-2 * np.abs(dqkv_r).max()
    ctx_a, dq_a = run("attention")
    np.testing.assert_allclose(ctx_a, ctx_r, atol=tol_c, rtol=0)
    np.testing.assert_allclose(dq_a, dqkv_r, atol=tol_g, rtol=0)
    if not fused:
        if p == 0:
            for i, name in enumerate(("dq", "dk")):
                assert_no_gain(dq_a[..., i * H:(i + 1) * H], dqkv_r[..., i * H:(i + 1) * H], name)
        return
    # the fused backward also accumulates the QKV bias gradient = column sums of the dqkv it stored
    gb_ref = dq_a.astype(np.float64).reshape(-1, 3 * H).sum(0)
    if S <= 256:
        np.testing.assert_allclose(bias.grad.numpy(), gb_ref, rtol=1e-4, atol=1e-4 * (np.abs(gb_ref).max() + 1))
    else:
        # two CTAs per head: the bias sums add each half's bf16 partial dK / dV, the stored tensor holds the bf16 sum of
        # the two partials -- they differ by that final rounding (<= 2^-9 |x| per element, worst case over the column)
        bound = 2.0 ** -9 * np.abs(dq_a.astype(np.float64)).reshape(-1, 3 * H).sum(0) + 1e-4 * (np.abs(gb_ref).max() + 1)
        assert np.all(np.abs(bias.grad.numpy() - gb_ref) <= bound)
    ctx_u, dq_u = run("unfused")
    np.testing.assert_allclose(ctx_u, ctx_r, atol=tol_c, rtol=0)
    np.testing.assert_allclose(dq_u, dqkv_r, atol=tol_g, rtol=0)
