"""Times polus_gemm_tc on every GEMM shape of one BERT-base training step (B=32, S=256): where do the GEMM
milliseconds go?  Usage: python tools/gemm_shapes.py [batch]"""
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from polus_b200 import _lib, device  # noqa: E402

Bsz = int(sys.argv[1]) if len(sys.argv) > 1 else 32
S, H, I, nh, dh = 256, 768, 3072, 12, 64
M = Bsz * S
device.init(0)
big = device.Buffer(1 << 30)
big2 = device.Buffer(1 << 30)
out = device.Buffer(1 << 30, zero=True)
bias = device.Buffer(1 << 16, zero=True)
device.synchronize()


def op(ptr, ld, mn, bs0=0, bs1=0):
    return _lib.Operand(ptr, ld, bs0, bs1, mn, _lib.BF16)


def case(name, M_, N_, K_, A, B, ldc, c_dtype, b0=1, b1=1, cbs0=0, cbs1=0, acc=0, split=1, act=0, c2=False, use_bias=True, count=1,
         c2_kind=0, emul=False, colsum=True):
    if os.environ.get("GEMM_ONLY") and os.environ["GEMM_ONLY"] not in name:
        return 0.0
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = M_, N_, K_, b0, b1
    g.A, g.B = A, B
    g.C, g.ldc, g.cbs0, g.cbs1, g.c_dtype = out.ptr, ldc, cbs0, cbs1, c_dtype
    g.C2 = (out.ptr + (1 << 29)) if c2 else None
    g.bias = bias.ptr if use_bias else None
    g.alpha, g.act, g.accumulate, g.split_k = 1.0, act, acc, split
    g.c2_kind = c2_kind
    if emul:  # fused activation backward: multiplier tile + bias-gradient column sums
        g.Emul, g.colsum = out.ptr + (1 << 29), (bias.ptr if colsum else None)
    assert _lib.call("polus_gemm_tc_supported", C.byref(g)) == 1, (name, _lib.last_error())
    e0, e1 = C.c_void_p(), C.c_void_p()
    _lib.call("polus_event_create", C.byref(e0)); _lib.call("polus_event_create", C.byref(e1))
    ncu = os.environ.get("GEMM_NCU") == "1"   # one launch per shape: `ncu --set full -k regex:gemm_tc -c 12` captures the step's 12 shapes
    if ncu and name.startswith("  ("):
        return 0.0
    for _ in range(0 if ncu else 3):
        _lib.call("polus_gemm_tc", C.byref(g), device.stream())
    reps = 1 if ncu else 20
    _lib.call("polus_event_record", e0, device.stream())
    for _ in range(reps):
        _lib.call("polus_gemm_tc", C.byref(g), device.stream())
    _lib.call("polus_event_record", e1, device.stream())
    device.synchronize()
    ms = C.c_float()
    _lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
    us = ms.value * 1000 / reps
    fl = 2.0 * M_ * N_ * K_ * b0 * b1
    r = {"case": name, "us": round(us, 1), "tflops": round(fl / us / 1e6, 1), "per_step_count": count, "ms_per_step": round(us * count / 1000, 3)}
    print(json.dumps(r), flush=True)
    return us * count / 1000


a, b = big.ptr, big2.ptr
tot = 0.0
L = 12
tot += case("fwd_qkv", M, 3 * H, H, op(a, H, 0), op(b, 3 * H, 1), 3 * H, _lib.BF16, count=L)
tot += case("fwd_attn_out", M, H, H, op(a, H, 0), op(b, H, 1), H, _lib.BF16, count=L)
tot += case("fwd_ffn1_gelu+gelu'(8-bit)", M, I, H, op(a, H, 0), op(b, I, 1), I, _lib.BF16, act=1, c2=True, c2_kind=2, count=L)
case("  (fwd_ffn1 gelu + bf16 gelu')", M, I, H, op(a, H, 0), op(b, I, 1), I, _lib.BF16, act=1, c2=True, c2_kind=1, count=L)
if os.environ.get("GEMM_EXTRA") == "1":   # what does the FFN-up epilogue pay for: the math, or the two staged stores?
    case("  x1 ffn1 gelu, one output (16-warp)", M, I, H, op(a, H, 0), op(b, I, 1), I, _lib.BF16, act=1, count=L)
    case("  x2 ffn1 no act, C + pre-activation copy (16-warp, no math)", M, I, H, op(a, H, 0), op(b, I, 1), I, _lib.BF16, act=0, c2=True, c2_kind=0, count=L)
    case("  x3 ffn1 relu + relu' (16-warp, cheap math, two outputs)", M, I, H, op(a, H, 0), op(b, I, 1), I, _lib.BF16, act=2, c2=True, c2_kind=1, count=L)
    case("  x4 ffn1 relu, one output (16-warp)", M, I, H, op(a, H, 0), op(b, I, 1), I, _lib.BF16, act=2, count=L)
    case("  x5 ffn1 plain (8-warp kernel)", M, I, H, op(a, H, 0), op(b, I, 1), I, _lib.BF16, act=0, count=L)
tot += case("fwd_ffn2", M, H, I, op(a, I, 0), op(b, H, 1), H, _lib.BF16, count=L)
tot += case("dgrad_qkv", M, H, 3 * H, op(a, 3 * H, 0), op(b, 3 * H, 0), H, _lib.BF16, use_bias=False, count=L)
tot += case("dgrad_attn_out", M, H, H, op(a, H, 0), op(b, H, 0), H, _lib.BF16, use_bias=False, count=L)
tot += case("dgrad_ffn1", M, H, I, op(a, I, 0), op(b, I, 0), H, _lib.BF16, use_bias=False, count=L)
tot += case("dgrad_ffn2*gelu'(8-bit)+colsum", M, I, H, op(a, H, 0), op(b, H, 0), I, _lib.BF16, use_bias=False, emul=True, c2_kind=2, count=L)
case("  (dgrad_ffn2 * bf16 gelu' + colsum)", M, I, H, op(a, H, 0), op(b, H, 0), I, _lib.BF16, use_bias=False, emul=True, count=L)
case("  (same without colsum)", M, I, H, op(a, H, 0), op(b, H, 0), I, _lib.BF16, use_bias=False, emul=True, colsum=False, count=L)
case("  (plain dgrad_ffn2, no Emul)", M, I, H, op(a, H, 0), op(b, H, 0), I, _lib.BF16, use_bias=False, count=L)
tot += case("wgrad_qkv", H, 3 * H, M, op(a, H, 1), op(b, 3 * H, 1), 3 * H, _lib.F32, acc=1, split=0, use_bias=False, count=L)
tot += case("wgrad_attn_out", H, H, M, op(a, H, 1), op(b, H, 1), H, _lib.F32, acc=1, split=0, use_bias=False, count=L)
tot += case("wgrad_ffn1", H, I, M, op(a, H, 1), op(b, I, 1), I, _lib.F32, acc=1, split=0, use_bias=False, count=L)
tot += case("wgrad_ffn2", I, H, M, op(a, I, 1), op(b, H, 1), H, _lib.F32, acc=1, split=0, use_bias=False, count=L)
print(json.dumps({"total_gemm_ms_per_step": round(tot, 3), "batch": Bsz}))
if len(sys.argv) <= 2:
    sys.exit(0)
# batched attention GEMMs of the UNFUSED path (S > 256 only; not part of the S=256 step)
H3 = 3 * H
qkv = lambda ptr, mn: op(ptr, H3, mn, dh, S * H3)
pm = lambda ptr, mn: op(ptr, S, mn, S * S, S * S * nh)
tot += case("attn_scores", S, S, dh, qkv(a, 0), qkv(a + H * 2, 0), S, _lib.BF16, nh, Bsz, S * S, S * S * nh, use_bias=False, count=L)
tot += case("attn_pv", S, dh, S, pm(b, 0), qkv(a + 2 * H * 2, 1), H, _lib.BF16, nh, Bsz, dh, S * H, use_bias=False, count=L)
tot += case("attn_dp", S, S, dh, op(a, H, 0, dh, S * H), qkv(a + 2 * H * 2, 0), S, _lib.BF16, nh, Bsz, S * S, S * S * nh, use_bias=False, count=L)
tot += case("attn_dv", S, dh, S, pm(b, 1), op(a, H, 1, dh, S * H), H3, _lib.BF16, nh, Bsz, dh, S * H3, use_bias=False, count=L)
tot += case("attn_dq", S, dh, S, pm(b, 0), qkv(a + H * 2, 1), H3, _lib.BF16, nh, Bsz, dh, S * H3, use_bias=False, count=L)
tot += case("attn_dk", S, dh, S, pm(b, 1), qkv(a, 1), H3, _lib.BF16, nh, Bsz, dh, S * H3, use_bias=False, count=L)
print(json.dumps({"total_gemm_ms_per_step": round(tot, 3), "batch": Bsz}))
