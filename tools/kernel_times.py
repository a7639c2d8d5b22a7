"""Isolated timings of the memory-bound kernels at the bench shapes (BERT-base, S=256), with a D2D memcpy of the same
byte count beside each as the practical floor.  Buffers rotate through NSETS copies so that every launch reads
HBM-cold data (NSETS x footprint > 126 MB L2), like inside the step.
    python tools/kernel_times.py [batch]"""
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from polus_b200 import _lib, device, ops  # noqa: E402
from polus_b200.tensor import BF16, F32, I32, U8, Tensor  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
# KT_H / KT_S: other hidden sizes and sequence lengths (H = 1024, S = 512: the BERT-large-sized configuration);
# KT_ONLY=ln: stop after the LayerNorm kernels
H = int(os.environ.get("KT_H", "768"))
S = int(os.environ.get("KT_S", "256"))
NH, I = H // 64, 4 * H
M = B * S
NSETS, REPS = 6, 5
device.init(0)
st = device.stream()
rng = np.random.default_rng(0)


def rnd(shape, dtype=BF16, scale=1.0):
    return Tensor.from_numpy((rng.standard_normal(shape) * scale).astype(np.float32), dtype)


def ev():
    e = C.c_void_p()
    _lib.call("polus_event_create", C.byref(e))
    return e


def timeit(fn):
    for k in range(NSETS):
        fn(k)
    e0, e1 = ev(), ev()
    device.device_sync()
    _lib.call("polus_event_record", e0, st)
    for r in range(REPS):
        for k in range(NSETS):
            fn(k)
    _lib.call("polus_event_record", e1, st)
    device.device_sync()
    ms = C.c_float()
    _lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
    return ms.value * 1e3 / (REPS * NSETS)


def report(name, us, nbytes):
    src = [Tensor((nbytes // 2,), U8) for _ in range(NSETS)]
    dst = [Tensor((nbytes // 2,), U8) for _ in range(NSETS)]
    floor = timeit(lambda k: _lib.call("polus_memcpy_d2d", dst[k].ptr, src[k].ptr, nbytes // 2, st))
    print(json.dumps({"kernel": name, "batch": B, "us": round(us, 2), "algorithmic_MB": round(nbytes / 1e6, 1),
                      "GBps": round(nbytes / us / 1e3, 0), "memcpy_same_bytes_us": round(floor, 2)}), flush=True)


step = ops.step_counter()
ops.set_step(1)
gamma, beta = rnd((H,), F32), rnd((H,), F32)
gg, gb, gx = Tensor((H,), F32, zero=True), Tensor((H,), F32, zero=True), Tensor((H,), F32, zero=True)
for p_drop in (0.1, 0.0):
    xs = [rnd((M, H)) for _ in range(NSETS)]
    rs = [rnd((M, H)) for _ in range(NSETS)]
    ys = [Tensor((M, H), BF16) for _ in range(NSETS)]
    mean, rstd = Tensor((M,), F32), Tensor((M,), F32)
    keep = [Tensor((M * H // 8,), U8) for _ in range(NSETS)]
    us = timeit(lambda k: _lib.call("polus_ln_res_fwd", xs[k].ptr, rs[k].ptr, gamma.ptr, beta.ptr, M, H, 1e-12, p_drop, 7, 3, step,
                                    ys[k].ptr, mean.ptr, rstd.ptr, keep[k].ptr if p_drop else None, st))
    report(f"ln_res_fwd p={p_drop}", us, M * H * 8)
    dxs = [Tensor((M, H), BF16) for _ in range(NSETS)]
    drs = [Tensor((M, H), BF16) for _ in range(NSETS)]
    us = timeit(lambda k: _lib.call("polus_ln_res_bwd", ys[k].ptr, rs[k].ptr, xs[k].ptr, mean.ptr, rstd.ptr, gamma.ptr, M, H, p_drop, 7, 3,
                                    step, dxs[k].ptr, drs[k].ptr if p_drop else dxs[k].ptr, gg.ptr, gb.ptr, gx.ptr,
                                    keep[k].ptr if p_drop else None, st))
    report(f"ln_res_bwd p={p_drop} (dy, dy2, z -> dx, dres)", us, M * H * (10 if p_drop else 8))
    del xs, rs, ys, dxs, drs, keep

if os.environ.get("KT_ONLY") == "ln":
    sys.exit(0)
# attention
for p_drop in (0.1, 0.0):
    qkv = [rnd((B, S, 3 * H)) for _ in range(NSETS)]
    ctx = [Tensor((B, S, H), BF16) for _ in range(NSETS)]
    dctx = [rnd((B, S, H)) for _ in range(NSETS)]
    dqkv = [Tensor((B, S, 3 * H), BF16) for _ in range(NSETS)]
    lse = Tensor((B, NH, S), F32)
    kb = Tensor((int(_lib.call("polus_attention_keepbits_words", B, S, NH)),), I32)
    mask = Tensor.from_numpy(np.ones((B, S), np.int32), I32)
    gbq = Tensor((3 * H,), F32, zero=True)
    us = timeit(lambda k: _lib.call("polus_attention_fwd", qkv[k].ptr, mask.ptr, B, S, NH, 64, p_drop, 7, 5, step, ctx[k].ptr, lse.ptr,
                                    kb.ptr if p_drop else None, st))
    report(f"attention_fwd p={p_drop}", us, M * H * 2 * 4)
    us = timeit(lambda k: _lib.call("polus_attention_bwd", qkv[k].ptr, mask.ptr, ctx[k].ptr, dctx[k].ptr, lse.ptr, B, S, NH, 64, p_drop, 7, 5,
                                    step, kb.ptr if p_drop else None, dqkv[k].ptr, gbq.ptr, st))
    report(f"attention_bwd p={p_drop}", us, M * H * 2 * 8)
    del qkv, ctx, dctx, dqkv

# activation backward (stored derivative) + bias colsum
dy = [rnd((M, I)) for _ in range(NSETS)]
dd = [rnd((M, I)) for _ in range(NSETS)]
dz = [Tensor((M, I), BF16) for _ in range(NSETS)]
gbias = Tensor((I,), F32, zero=True)
us = timeit(lambda k: _lib.call("polus_act_bwd_colsum", dy[k].ptr, dd[k].ptr, M, I, _lib.ACT_DERIV, dz[k].ptr, gbias.ptr, None, st))
report("act_bwd_colsum (dy * stored act')", us, M * I * 6)
us = timeit(lambda k: _lib.call("polus_act_bwd_colsum", dy[k].ptr, dd[k].ptr, M, I, _lib.ACT["gelu"], dz[k].ptr, gbias.ptr, None, st))
report("act_bwd_colsum (gelu' recomputed)", us, M * I * 6)

# CRF negative log-likelihood + gradients (latency-bound: T sequential steps per sequence, one CTA of two warps each)
K = 4
em = [Tensor.from_numpy(rng.standard_normal((B, S, K)).astype(np.float32), F32) for _ in range(NSETS)]
tg = Tensor.from_numpy(rng.integers(1, K, (B, S)).astype(np.int32), I32)
tr = Tensor.from_numpy(rng.standard_normal((K, K)).astype(np.float32), F32)
nll, loss, ge, gt = Tensor((B,), F32), Tensor((), F32, zero=True), Tensor((B, S, K), F32), Tensor((K, K), F32, zero=True)
us = timeit(lambda k: _lib.call("polus_crf_nll", em[k].ptr, tg.ptr, None, tr.ptr, None, B, S, K, nll.ptr, loss.ptr, ge.ptr, gt.ptr, st))
print(json.dumps({"kernel": "crf_nll (fwd+bwd recursions, K=4)", "batch": B, "us": round(us, 2), "steps": S,
                  "cycles_per_step_at_1.8GHz": round(us * 1800 / S)}), flush=True)
