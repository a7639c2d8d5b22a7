"""The GEMM, unfused-attention and LayerNorm kernels at the shapes and layouts a training step launches, against numpy
fp64 on the same bf16 inputs.

GEMM cases use the operand majors and pointers `ops.linear` and `ops._attention_unfused` pass, at BERT-base and
BERT-large sizes and at two row counts (8192 selects 256-wide tiles for the H-wide outputs, 4072 = 4000 + 72 selects
128-wide tiles and leaves a ragged last row tile).  Every output lives inside a larger allocation prefilled with a canary
bit pattern (a NaN in bf16 and fp32), at least 256 rows of C on each side; after the call every byte outside the view
must be unchanged.  `polus_gemm_tc_plan` names the kernel each case runs, and the last test checks that the cases
together reach every instantiation polus_gemm_tc can launch.

Bars (BASELINE.md section 3 states the looser model-level ones):
  fp32 C  |C - ref| <= 1e-4 max|ref| elementwise and ||C - ref||_F <= 1e-5 ||ref||_F
  bf16 C  |C - ref| <= 2^-8 |ref| + 2^-12 max|ref| elementwise
  8-bit gelu'  decoded value within half a step (0.0025) of gelu'(ref)
With unit-variance products these fail when a single 64-deep k-block is dropped (an error of about sqrt(64 / K) of the
output scale) or when the bias (half the output scale) is added twice.
"""
import ctypes as C
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BF16_EPS = 2.0 ** -8
CANARY = 0x7FA17FA1  # NaN as bf16 and as fp32: a kernel that reads it by mistake poisons its output


@pytest.fixture(scope="module")
def dev():
    from polus_b200 import device
    device.init(0)
    return device


_KEEP = []  # device tensors of the running test: raw pointers taken from them must not dangle


@pytest.fixture(autouse=True)
def _keepalive():
    yield
    _KEEP.clear()


def call(name, *a):
    from polus_b200 import _lib
    return _lib.call(name, *a)


def st():
    from polus_b200 import device
    return device.stream()


def upload_bytes(host_u8):
    from polus_b200.tensor import Tensor, U8
    t = Tensor.from_numpy(host_u8, U8)
    _KEEP.append(t)
    return t


# -------------------------------------------------------------------------------------------------- guarded buffers
_BITS = {1: np.uint8, 2: np.uint16, 4: np.uint32}


class Guarded:
    """A strided view [b1][b0][rows][cols] (element strides s1, s0, ld, 1) of `esize`-byte elements inside an allocation
    whose other bytes, including the gaps between rows and batches, hold CANARY."""

    def __init__(self, shape, strides, esize, init_bits=None):
        b1, b0, rows, cols = shape
        s1, s0, ld = strides
        self.esize, self.shape = esize, shape
        span = 1 + (b1 - 1) * s1 + (b0 - 1) * s0 + (rows - 1) * ld + (cols - 1)
        margin = 256 * max(ld, cols) + 4096
        margin = -(-margin * esize // 1024) * 1024 // esize  # keeps the view 1024-byte aligned
        nbytes = -(-(2 * margin + span) * esize // 4) * 4
        self.before = np.full(nbytes // 4, CANARY, np.uint32).view(_BITS[esize])
        self.idx = (margin + np.arange(b1)[:, None, None, None] * s1 + np.arange(b0)[None, :, None, None] * s0
                    + np.arange(rows)[None, None, :, None] * ld + np.arange(cols)[None, None, None, :])
        if init_bits is not None:
            self.before[self.idx] = init_bits
        self.t = upload_bytes(self.before.view(np.uint8))
        self.ptr = self.t.ptr + margin * esize

    def result_bits(self):
        from polus_b200 import device
        after = device.download(self.t.ptr, (self.before.size * self.esize,), np.uint8).view(_BITS[self.esize])
        outside = np.ones(after.size, bool)
        outside[self.idx.ravel()] = False
        bad = np.flatnonzero(outside & (after != self.before))
        assert bad.size == 0, f"{bad.size} elements outside the view changed, first at element offset {bad[0]}"
        return after[self.idx]


def bf16_bits(x):
    from polus_b200 import device
    return device.f32_to_bf16_bits(np.asarray(x, np.float32))


def from_bf16_bits(b):
    from polus_b200 import device
    return device.bf16_bits_to_f32(b).reshape(b.shape).astype(np.float64)


def assert_f32(out, ref, what):
    scale = np.abs(ref).max()
    err = np.abs(out - ref)
    assert err.max() <= 1e-4 * scale, f"{what}: max error {err.max():.3g} > 1e-4 * {scale:.3g}"
    rel = np.linalg.norm(out - ref) / np.linalg.norm(ref)
    assert rel <= 1e-5, f"{what}: relative Frobenius error {rel:.3g} > 1e-5"


def assert_bf16(out, ref, what):
    bound = BF16_EPS * np.abs(ref) + 2.0 ** -12 * np.abs(ref).max()
    excess = np.abs(out - ref) - bound
    assert excess.max() <= 0, f"{what}: {(excess > 0).sum()} elements outside 2^-8|ref| + 2^-12 max|ref|, worst at {np.unravel_index(excess.argmax(), excess.shape)}"


# -------------------------------------------------------------------------------------------------- GEMM cases
def spec(M, N, K, a_mn, b_mn, *, lda=None, ldb=None, ldc=None, b0=1, b1=1, abs0=0, abs1=0, bbs0=0, bbs1=0, cbs0=0,
         cbs1=0, c_f32=False, bias=False, alpha=1.0, act=None, acc=0, split_k=1, c2=False, c2_kind=0, emul=False,
         colsum=False):
    """One polus_gemm_tc problem; leading dims default to dense row-major tensors."""
    return dict(M=M, N=N, K=K, a_mn=a_mn, b_mn=b_mn, lda=lda or (M if a_mn else K), ldb=ldb or (N if b_mn else K),
                ldc=ldc or N, b0=b0, b1=b1, abs0=abs0, abs1=abs1, bbs0=bbs0, bbs1=bbs1, cbs0=cbs0, cbs1=cbs1,
                c_f32=c_f32, bias=bias, alpha=alpha, act=act, acc=acc, split_k=split_k, c2=c2, c2_kind=c2_kind,
                emul=emul, colsum=colsum)


def gemm_struct(s, a_ptr, b_ptr, c_ptr, c2_ptr=None, bias_ptr=None, emul_ptr=None, colsum_ptr=None):
    from polus_b200 import _lib
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = s["M"], s["N"], s["K"], s["b0"], s["b1"]
    g.A = _lib.Operand(a_ptr, s["lda"], s["abs0"], s["abs1"], s["a_mn"], _lib.BF16)
    g.B = _lib.Operand(b_ptr, s["ldb"], s["bbs0"], s["bbs1"], s["b_mn"], _lib.BF16)
    g.C, g.ldc, g.cbs0, g.cbs1 = c_ptr, s["ldc"], s["cbs0"], s["cbs1"]
    g.c_dtype = _lib.F32 if s["c_f32"] else _lib.BF16
    g.C2, g.bias, g.alpha, g.act = c2_ptr, bias_ptr, s["alpha"], _lib.ACT[s["act"]]
    g.accumulate, g.split_k, g.c2_kind, g.Emul, g.colsum = s["acc"], s["split_k"], s["c2_kind"], emul_ptr, colsum_ptr
    return g


def instantiation(s, plan):
    """The kernel template polus_gemm_tc launches: (epilogue warps, CTAs per tile, BN, A MN-major, B MN-major)."""
    cg, bn, _, epi16 = plan
    return (16 if epi16 else 8, cg, bn, s["a_mn"], s["b_mn"])


def plan_of(s):
    """polus_gemm_tc_plan for a spec, with stand-in addresses (the query reads no memory)."""
    fake = 1 << 24
    g = gemm_struct(s, fake, fake, fake, fake if s["c2"] else None, fake if s["bias"] else None,
                    fake if s["emul"] else None, fake if s["colsum"] else None)
    out = (C.c_int * 4)()
    call("polus_gemm_tc_plan", C.byref(g), out)
    return tuple(out)


def operand(rng, b1, b0, mn, k, ld, bs0, bs1, mn_major, scale):
    """Random bf16 operand in its strided layout -> (device tensor, logical [b1][b0][mn][k] fp64)."""
    from polus_b200.tensor import BF16, Tensor
    span = 1 + (b1 - 1) * bs1 + (b0 - 1) * bs0 + ((k - 1) * ld + mn - 1 if mn_major else (mn - 1) * ld + k - 1)
    flat = rng.standard_normal(span).astype(np.float32) * np.float32(scale)
    t = Tensor.from_numpy(flat, BF16)
    _KEEP.append(t)
    flat = from_bf16_bits(bf16_bits(flat))
    i1 = np.arange(b1)[:, None, None, None] * bs1 + np.arange(b0)[None, :, None, None] * bs0
    r, c = np.arange(mn)[None, None, :, None], np.arange(k)[None, None, None, :]
    return t, flat[i1 + (c * ld + r if mn_major else r * ld + c)]


def run_case(dev, s, seed):
    """Launch one spec with canary-guarded outputs and check every output against numpy fp64.  -> kernel instantiation"""
    from oracle import numpy_ref as R
    from polus_b200.tensor import F32, Tensor
    rng = np.random.default_rng(seed)
    M, N, K, b0, b1 = s["M"], s["N"], s["K"], s["b0"], s["b1"]
    plan = plan_of(s)
    a_t, A = operand(rng, b1, b0, M, K, s["lda"], s["abs0"], s["abs1"], s["a_mn"], 1.0)
    b_t, B = operand(rng, b1, b0, N, K, s["ldb"], s["bbs0"], s["bbs1"], s["b_mn"], 1.0 / math.sqrt(K))
    z = s["alpha"] * np.matmul(A, B.swapaxes(-1, -2))  # [b1][b0][M][N]
    cshape, cstr = (b1, b0, M, N), (s["cbs1"], s["cbs0"], s["ldc"])
    bias_t = None
    if s["bias"]:
        bias = (0.5 * rng.standard_normal(N)).astype(np.float32)
        bias_t = Tensor.from_numpy(bias, F32)
        _KEEP.append(bias_t)
        z = z + bias
    c_before = None
    if s["acc"]:  # C += result: start from an existing gradient, not from zeros
        c_before = rng.standard_normal(cshape).astype(np.float32)
        Cg = Guarded(cshape, cstr, 4, c_before.view(np.uint32))
    else:
        Cg = Guarded(cshape, cstr, 4 if s["c_f32"] else 2)
    C2g = Eg = csg = None
    if s["c2"]:
        C2g = Guarded(cshape, cstr, 1 if s["c2_kind"] == 2 else 2)
    mult = None
    if s["emul"]:
        if s["c2_kind"] == 2:
            q = rng.integers(2, 255, cshape).astype(np.uint8)
            Eg, mult = Guarded(cshape, cstr, 1, q), (q.astype(np.float64) - 28.0) * 0.005
        else:
            e = rng.standard_normal(cshape).astype(np.float32)
            Eg, mult = Guarded(cshape, cstr, 2, bf16_bits(e)), from_bf16_bits(bf16_bits(e))
    cs_before = None
    if s["colsum"]:  # the bias-gradient vector, between canaries, holding an earlier gradient
        cs_before = rng.standard_normal(N).astype(np.float32)
        csg = Guarded((1, 1, 1, N), (0, 0, N), 4, cs_before.view(np.uint32))
    g = gemm_struct(s, a_t.ptr, b_t.ptr, Cg.ptr, C2g.ptr if C2g else None, bias_t.ptr if bias_t is not None else None,
                    Eg.ptr if Eg else None, csg.ptr if csg else None)
    call("polus_gemm_tc", C.byref(g), st())
    what = f"{M}x{N}x{K} plan {plan}"
    if s["c_f32"]:
        out = Cg.result_bits().view(np.float32).astype(np.float64)
        ref = z if c_before is None else c_before.astype(np.float64) + z
        assert_f32(out, ref, what)
    else:
        out = from_bf16_bits(Cg.result_bits())
        if s["act"] is not None:
            ref = R.ACT[s["act"]][0](z)
        elif mult is not None:
            ref = z * mult
        else:
            ref = z
        assert_bf16(out, ref, what)
        if C2g is not None:
            if s["c2_kind"] == 2:  # 8-bit gelu': decoded within half a step (+ fp32 noise of numpy's gelu')
                q = C2g.result_bits().astype(np.float64)
                assert q.min() >= 2 and q.max() <= 254
                np.testing.assert_allclose((q - 28.0) * 0.005, R.ACT[s["act"]][1](z), atol=0.0025 + 2e-4, rtol=0, err_msg=what)
            elif s["c2_kind"] == 1:
                assert_bf16(from_bf16_bits(C2g.result_bits()), R.ACT[s["act"]][1](z), what + " C2 = act'")
            else:
                assert_bf16(from_bf16_bits(C2g.result_bits()), z, what + " C2 = pre-activation")
        if Eg is not None:
            assert np.array_equal(Eg.result_bits(), Eg.before[Eg.idx])  # a read-only input: nothing in or around it written
        if csg is not None:  # column sums of the stored (bf16) values, added to what the vector held
            cs_ref = cs_before.astype(np.float64) + out.reshape(-1, N).sum(0)
            cs = csg.result_bits().view(np.float32).reshape(N)
            np.testing.assert_allclose(cs, cs_ref, rtol=1e-4, atol=1e-4 * (np.abs(cs_ref).max() + 1), err_msg=what + " colsum")
    return instantiation(s, plan)


# The training step's GEMMs, as ops.linear issues them for x [M, H] and weights W [in, out] (Keras layout):
#   forward  y = x . W           A = x K-major, B = W MN-major (ld = out), bf16 C, bias
#   dgrad    dx = dy . W^T       A = dy K-major, B = W K-major (ld = out), bf16 C (* act'(z) + bias-gradient colsum)
#   wgrad    dW += x^T . dy      A = x MN-major, B = dy MN-major, fp32 C, accumulate, split_k = 0 (planned split)
MODELS = {"base": (768, 3072), "large": (1024, 4096)}
ROWS = (8192, 4072)


def step_specs(H, I, M):
    fwd = lambda n, k, **kw: spec(M, n, k, 0, 1, bias=True, **kw)
    dgrad = lambda n, k, **kw: spec(M, n, k, 0, 0, ldb=k, **kw)
    wgrad = lambda k_in, n_out: spec(k_in, n_out, M, 1, 1, c_f32=True, acc=1, split_k=0)
    return {
        "fwd_qkv": fwd(3 * H, H),
        "fwd_attn_out": fwd(H, H),
        "fwd_ffn_up_gelu_d8": fwd(I, H, act="gelu", c2=True, c2_kind=2),
        "fwd_ffn_up_gelu_bf16": fwd(I, H, act="gelu", c2=True, c2_kind=1),
        "fwd_ffn_down": fwd(H, I),
        "dgrad_qkv": dgrad(H, 3 * H),
        "dgrad_attn_out": dgrad(H, H),
        "dgrad_ffn_up": dgrad(H, I),
        "dgrad_ffn_down_emul_d8": dgrad(I, H, emul=True, c2_kind=2, colsum=True),
        "dgrad_ffn_down_emul_bf16": dgrad(I, H, emul=True, c2_kind=1, colsum=True),
        "wgrad_qkv": wgrad(H, 3 * H),
        "wgrad_attn_out": wgrad(H, H),
        "wgrad_ffn_up": wgrad(H, I),
        "wgrad_ffn_down": wgrad(I, H),
    }


STEP_CASES = [(m, rows, name) for m in MODELS for rows in ROWS for name in step_specs(*MODELS[m], rows)]


@pytest.mark.parametrize("model,rows,name", STEP_CASES)
def test_gemm_step_shapes(dev, model, rows, name):
    s = step_specs(*MODELS[model], rows)[name]
    run_case(dev, s, seed=rows + len(name))


def attention_specs(Bsz, nh, S, dh):
    """The six batched GEMMs of ops._attention_unfused: batch0 = head, batch1 = sequence; q / k / v are column blocks of
    qkv [B, S, 3H], ctx is [B, S, H], and dQ / dK / dV are written into column blocks of one dqkv [B, S, 3H] (ldc = 3H)."""
    H = nh * dh
    qkv = dict(b0=nh, b1=Bsz)
    x3 = dict(ld=3 * H, bs0=dh, bs1=S * 3 * H)  # q, k or v per head: [S, dh] rows of qkv
    sq = dict(ld=S, bs0=S * S, bs1=S * S * nh)               # scores / probabilities [nb, S, S]
    o = dict(ld=H, bs0=dh, bs1=S * H)                        # ctx / dctx per head

    def mk(M, N, K, a, a_mn, b, b_mn, c):
        return spec(M, N, K, a_mn, b_mn, lda=a["ld"], abs0=a["bs0"], abs1=a["bs1"], ldb=b["ld"], bbs0=b["bs0"],
                    bbs1=b["bs1"], ldc=c["ld"], cbs0=c["bs0"], cbs1=c["bs1"], **qkv)
    return {
        "scores": mk(S, S, dh, x3, 0, x3, 0, sq),
        "ctx": mk(S, dh, S, sq, 0, x3, 1, o),
        "dP": mk(S, S, dh, o, 0, x3, 0, sq),
        "dV": mk(S, dh, S, sq, 1, o, 1, x3),
        "dQ": mk(S, dh, S, sq, 0, x3, 1, x3),
        "dK": mk(S, dh, S, sq, 1, x3, 1, x3),
    }


ATTN_SHAPES = [(2, 3, 200, 64), (1, 2, 520, 128), (2, 2, 40, 32)]


@pytest.mark.parametrize("Bsz,nh,S,dh", ATTN_SHAPES)
def test_gemm_unfused_attention_layouts(dev, Bsz, nh, S, dh):
    """Strided A, B and C through batch strides, and C written through ldc = 3H into one column block of dqkv: the
    other two blocks, the canaries between them, are left alone."""
    for i, (name, s) in enumerate(attention_specs(Bsz, nh, S, dh).items()):
        run_case(dev, s, seed=S * 10 + i)


SPLIT_CASE = spec(768, 768, 4072, 1, 1, c_f32=True, acc=1, split_k=4, bias=True, alpha=0.5)


def test_gemm_explicit_split_k_bias_alpha(dev):
    """split_k = 4 onto an existing fp32 gradient, with a bias and alpha = 0.5: C = C_before + alpha A.B^T + bias, the
    bias added by the first split only."""
    assert plan_of(SPLIT_CASE)[2] == 4
    run_case(dev, SPLIT_CASE, seed=4)


RAGGED_N_CASES = {
    # FFN-up forward at an intermediate size that is not a multiple of 256: partial last tile in the 16-warp kernel
    "fwd_gelu_n1000": spec(8192, 1000, 768, 0, 1, bias=True, act="gelu", c2=True, c2_kind=1),
    "dgrad_emul_n1288": spec(8192, 1288, 1024, 0, 0, emul=True, c2_kind=1, colsum=True),
}


@pytest.mark.parametrize("name", list(RAGGED_N_CASES))
def test_gemm_16warp_ragged_n(dev, name):
    """Regression: the 16-warp kernel stored the pre-activation instead of act'(z) in C2 (c2_kind = 1) for the partial last
    32-column block, so a GELU layer with N % 32 != 0 had a wrong derivative in its last N % 32 columns."""
    s = RAGGED_N_CASES[name]
    assert plan_of(s)[3] == 1, "expected the 16-epilogue-warp kernel"
    run_case(dev, s, seed=s["N"])


def sweep_specs():
    """One small problem per 8-epilogue-warp instantiation (CTAs per tile x BN x operand majors), bf16 and fp32 outputs,
    alpha != 1 on half of them."""
    out = {}
    for a_mn in (0, 1):
        for b_mn in (0, 1):
            k = f"a{a_mn}b{b_mn}"
            alt = (a_mn + b_mn) % 2
            out["cg1_bn64_" + k] = spec(296, 64, 200, a_mn, b_mn, bias=True, c_f32=bool(alt), alpha=0.75 if alt else 1.0)
            out["cg1_bn128_" + k] = spec(96, 120, 136, a_mn, b_mn, bias=True, c_f32=not alt, alpha=1.0 if alt else 1.5)
            out["cg1_bn256_" + k] = spec(120, 328, 1000, a_mn, b_mn, c_f32=True, acc=1, split_k=0)
            out["cg2_bn128_" + k] = spec(296, 200, 136, a_mn, b_mn, bias=True, c_f32=bool(alt), alpha=0.75 if alt else 1.0)
            out["cg2_bn256_" + k] = spec(384, 520, 1024, a_mn, b_mn, c_f32=True, acc=1, split_k=0)
    return out


@pytest.mark.parametrize("name", list(sweep_specs()))
def test_gemm_instantiation_sweep(dev, name):
    run_case(dev, sweep_specs()[name], seed=len(name))


def existing_kernel_test_specs():
    """The problems tests/test_kernels_gpu.py launches, for the coverage count."""
    out = []
    for (M, N, K, a, b, split) in [(128, 128, 64, 0, 0, 1), (200, 136, 200, 0, 1, 1), (328, 72, 520, 1, 1, 1),
                                   (256, 256, 1024, 1, 1, 4), (96, 64, 64, 1, 0, 1), (512, 768, 256, 0, 1, 1)]:
        out.append(spec(M, N, K, a, b, c_f32=True, bias=True, acc=int(split > 1), split_k=split))
    for (M, N, K, a, b, f32) in [(32768, 768, 192, 0, 0, 0), (32768, 768, 136, 0, 1, 0), (32700, 576, 200, 0, 0, 1),
                                 (32768, 768, 64, 1, 1, 0), (32768, 576, 128, 1, 0, 0), (32768, 768, 3072, 0, 1, 0)]:
        out.append(spec(M, N, K, a, b, c_f32=bool(f32), bias=True, colsum=not f32))
    for (M, N, K) in [(512, 768, 256), (300, 200, 136), (8192, 3072, 768), (128, 320, 64), (77, 72, 520), (5000, 1536, 256)]:
        out.append(spec(M, N, K, 0, 0, bias=True, act="gelu", c2=True, c2_kind=1))
        out.append(spec(M, N, K, 0, 0, emul=True, colsum=True))
    return out


def all_instantiations():
    """Every kernel polus_gemm_tc can launch: the 8-epilogue-warp kernel for one CTA (BN 64 / 128 / 256) or a CTA pair
    (BN 128 / 256) and each operand-major pair, and the 16-epilogue-warp pair kernel (BN 256, A K-major) for either B."""
    out = {(8, 1, bn, a, b) for bn in (64, 128, 256) for a in (0, 1) for b in (0, 1)}
    out |= {(8, 2, bn, a, b) for bn in (128, 256) for a in (0, 1) for b in (0, 1)}
    out |= {(16, 2, 256, 0, b) for b in (0, 1)}
    return out


def test_gemm_cases_reach_every_instantiation(dev):
    specs = {f"step:{m}:{r}:{n}": s for m in MODELS for r in ROWS for n, s in step_specs(*MODELS[m], r).items()}
    for shape in ATTN_SHAPES:
        specs.update({f"attention:{shape}:{n}": s for n, s in attention_specs(*shape).items()})
    specs["split"] = SPLIT_CASE
    specs.update({f"ragged:{n}": s for n, s in RAGGED_N_CASES.items()})
    specs.update({f"sweep:{n}": s for n, s in sweep_specs().items()})
    specs.update({f"existing:{i}": s for i, s in enumerate(existing_kernel_test_specs())})
    reached = {}
    for name, s in specs.items():
        reached.setdefault(instantiation(s, plan_of(s)), []).append(name)
    for key in sorted(reached):
        print("epilogue warps %d, CTAs %d, BN %3d, A_MN %d, B_MN %d:" % key, len(reached[key]), "cases, e.g.", reached[key][0])
    missing = all_instantiations() - set(reached)
    assert not missing, f"instantiations no case reaches: {sorted(missing)}"
    assert set(reached) <= all_instantiations()
    # the planned wgrad split reduce-adds partial sums at the step's shapes (it picks 1 where the tiles fill the SMs)
    assert any(plan_of(s)[2] > 1 for n, s in specs.items() if ":wgrad_" in n)


# -------------------------------------------------------------------------------------------------- unfused attention
@pytest.mark.parametrize("S", [40, 200, 520, 1000])
@pytest.mark.parametrize("dh", [32, 64, 128])
@pytest.mark.parametrize("p", [0.0, 0.1])
def test_unfused_attention_shapes(dev, S, dh, p):
    """ops.attention where no fused kernel takes the shape (S % 32 != 0, S > 512, dh != 64): three batched GEMMs and the
    row softmax, against the fp64 oracle with the device's dropout masks; one sequence of length 1."""
    from polus_b200 import _lib
    from tests.attention_ref import check_attention_case
    assert _lib.call("polus_attention_supported", S, dh) == 0
    Bsz, nh = (2, 2) if S <= 200 else (2, 1)
    lens = np.array([1, S - 3]) if Bsz == 2 else np.array([1])
    check_attention_case(dev, Bsz, nh, S, p, True, dh=dh, lens=lens, fused=False, seed=S + dh)


# -------------------------------------------------------------------------------------------------- LayerNorm backward variants
def _ln_problem(dev, M, H, p, seed):
    from oracle import numpy_ref as R, philox
    from polus_b200 import ops
    from polus_b200.tensor import BF16, F32, U8, Tensor
    rng = np.random.default_rng(seed)
    x = dev.bf16_round(rng.standard_normal((M, H)).astype(np.float32))
    res = dev.bf16_round(rng.standard_normal((M, H)).astype(np.float32))
    gamma = (1 + 0.1 * rng.standard_normal(H)).astype(np.float32)
    beta = (0.1 * rng.standard_normal(H)).astype(np.float32)
    seed_, site, step = 321, 7, 5
    ops.set_step(step)
    sp = ops.step_counter()
    x_t, res_t, g_t, b_t = (Tensor.from_numpy(a, d) for a, d in ((x, BF16), (res, BF16), (gamma, F32), (beta, F32)))
    y_t, mean_t, rstd_t = Tensor((M, H), BF16), Tensor((M,), F32), Tensor((M,), F32)
    keep_t = Tensor((M * (H // 8),), U8)
    _KEEP.extend([x_t, res_t, g_t, b_t, y_t, mean_t, rstd_t, keep_t])
    call("polus_ln_res_fwd", x_t.ptr, res_t.ptr, g_t.ptr, b_t.ptr, M, H, 1e-12, p, seed_, site, sp, y_t.ptr, mean_t.ptr,
         rstd_t.ptr, keep_t.ptr if p > 0 else None, st())
    mask = philox.dropout_scale_mask((M, H), p, seed_, site, step) if p > 0 else np.ones((M, H), np.float32)
    dy = dev.bf16_round(rng.standard_normal((M, H)).astype(np.float32))
    _, cache = R.layer_norm(x_t.numpy().astype(np.float64), gamma, beta)  # x now holds the device's z
    dz, gg, gb = R.layer_norm_bwd(dy.astype(np.float64), cache, gamma)
    return dict(M=M, H=H, p=p, seed=seed_, site=site, sp=sp, z=x_t, mean=mean_t, rstd=rstd_t, gamma=g_t, keep=keep_t,
                mask=mask, dy=dy, dz=dz, gg=gg, gb=gb)


def _ln_bwd(P, dy_ptr, dy2_ptr, dx, dres, keep):
    from polus_b200.tensor import F32, Tensor
    M, H = P["M"], P["H"]
    gg, gb, gx = Tensor((H,), F32, zero=True), Tensor((H,), F32, zero=True), Tensor((H,), F32, zero=True)
    _KEEP.extend([gg, gb, gx])
    call("polus_ln_res_bwd", dy_ptr, dy2_ptr, P["z"].ptr, P["mean"].ptr, P["rstd"].ptr, P["gamma"].ptr, M, H, P["p"],
         P["seed"], P["site"], P["sp"], dx.ptr, dres.ptr if dres is not None else None, gg.ptr, gb.ptr, gx.ptr, keep, st())
    return gg.numpy(), gb.numpy(), gx.numpy()


def _ln_check(P, dx, dres, grads):
    """The bars of test_ln_residual_fwd_bwd.  The parameter gradients are sums over M rows: their atol is relative to
    max|ref|, which grows as sqrt(M) for these random-sign rows, and so does the error of the fp32 sums."""
    tol = 3 * BF16_EPS * (1 + np.abs(P["dz"]).max())
    if dres is not None:
        np.testing.assert_allclose(dres, P["dz"], atol=tol, rtol=0)
    np.testing.assert_allclose(dx, P["dz"] * P["mask"], atol=tol * 1.2, rtol=0)
    gg, gb, gx = grads
    np.testing.assert_allclose(gg, P["gg"], rtol=2e-3, atol=2e-3 * np.abs(P["gg"]).max())
    np.testing.assert_allclose(gb, P["gb"], rtol=2e-3, atol=2e-3 * np.abs(P["gb"]).max())
    gx_ref = dx.astype(np.float64).sum(0)
    np.testing.assert_allclose(gx, gx_ref, rtol=1e-2, atol=1e-2 * (np.abs(gx_ref).max() + 1))


@pytest.mark.parametrize("H", [256, 512, 768, 1024])
def test_ln_residual_bwd_variants(dev, H):
    """At M = 7109 (three full row strides of the 296 x 8 warps plus 5: warps end on different slot parities), the
    variants of polus_ln_res_bwd the shape test does not run: one d(y) contribution (dy2 = NULL); the keep bits 8 bytes off
    16-byte alignment inside a larger buffer, which runs ln_res_bwd_kernel instead of the prefetching kernel (both must
    meet the bars, with the same dx); and dres == dx without dropout, as ops.layernorm_residual calls it.

    Regression: a dy 8 bytes off 16-byte alignment used to be sent to ln_res_bwd_kernel, whose 16-byte loads fault on it;
    the entry point now rejects row pointers that are not 16-byte aligned."""
    from polus_b200.tensor import BF16, U8, Tensor
    M = 7109
    P = _ln_problem(dev, M, H, 0.1, seed=H)
    dy_t = Tensor.from_numpy(P["dy"], BF16)
    kb = P["keep"].numpy()
    kb_off = Tensor((kb.size + 16,), U8)
    _KEEP.extend([dy_t, kb_off])
    dev.upload(kb_off.ptr + 8, kb)
    outs = {}
    for name, keep_ptr in (("prefetching", P["keep"].ptr), ("fallback", kb_off.ptr + 8)):
        dx, dres = Tensor((M, H), BF16), Tensor((M, H), BF16)
        _KEEP.extend([dx, dres])
        grads = _ln_bwd(P, dy_t.ptr, None, dx, dres, keep_ptr)
        _ln_check(P, dx.numpy(), dres.numpy(), grads)
        outs[name] = dx.numpy()
    assert np.array_equal(outs["prefetching"], outs["fallback"])  # same per-row arithmetic in both kernels
    with pytest.raises(ValueError, match="16-byte aligned"):
        _ln_bwd(P, dy_t.ptr + 8, None, Tensor((M, H), BF16), None, P["keep"].ptr)
    # no dropout: dres aliases dx, and d(y) arrives in two halves
    P = _ln_problem(dev, M, H, 0.0, seed=H + 1)
    dy_a = dev.bf16_round((0.5 * P["dy"]).astype(np.float32))
    dy_b = dev.bf16_round((P["dy"] - dy_a).astype(np.float32))
    assert np.array_equal(dy_a + dy_b, P["dy"])
    a_t, b_t, dx = Tensor.from_numpy(dy_a, BF16), Tensor.from_numpy(dy_b, BF16), Tensor((M, H), BF16)
    _KEEP.extend([a_t, b_t, dx])
    grads = _ln_bwd(P, a_t.ptr, b_t.ptr, dx, dx, None)
    _ln_check(P, dx.numpy(), None, grads)
