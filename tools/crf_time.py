"""Isolated timing of the CRF kernels (polus_crf_nll and polus_crf_decode):  python tools/crf_time.py [batch] [tags] [steps]
(defaults 128, 4, 256).  Four emission sets are cycled so that consecutive launches do not read the same buffer."""
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from polus_b200 import _lib, device  # noqa: E402
from polus_b200.tensor import F32, I32, Tensor  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 128
K = int(sys.argv[2]) if len(sys.argv) > 2 else 4
S = int(sys.argv[3]) if len(sys.argv) > 3 else 256
NSETS, REPS = 4, 10
device.init(0)
st = device.stream()
rng = np.random.default_rng(0)
em = [Tensor.from_numpy(rng.standard_normal((B, S, K)).astype(np.float32), F32) for _ in range(NSETS)]
tg = Tensor.from_numpy(rng.integers(1, K, (B, S)).astype(np.int32) if K > 1 else np.zeros((B, S), np.int32), I32)
tr = Tensor.from_numpy(rng.standard_normal((K, K)).astype(np.float32), F32)
nll, loss, ge, gt = Tensor((B,), F32), Tensor((), F32, zero=True), Tensor((B, S, K), F32), Tensor((K, K), F32, zero=True)
path, score = Tensor((B, S), I32), Tensor((B,), F32)


def run_nll(k):
    _lib.call("polus_crf_nll", em[k].ptr, tg.ptr, None, tr.ptr, None, B, S, K, nll.ptr, loss.ptr, ge.ptr, gt.ptr, st)


def run_decode(k):
    _lib.call("polus_crf_decode", em[k].ptr, None, tr.ptr, B, S, K, path.ptr, score.ptr, st)


e0, e1 = C.c_void_p(), C.c_void_p()
_lib.call("polus_event_create", C.byref(e0))
_lib.call("polus_event_create", C.byref(e1))


def time_us(fn):
    for k in range(NSETS):
        fn(k)
    device.device_sync()
    _lib.call("polus_event_record", e0, st)
    for _ in range(REPS):
        for k in range(NSETS):
            fn(k)
    _lib.call("polus_event_record", e1, st)
    device.device_sync()
    ms = C.c_float()
    _lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
    return ms.value * 1e3 / (REPS * NSETS)


us_nll = time_us(run_nll)
us_dec = time_us(run_decode)
print(json.dumps({"kernel": f"crf_nll K={K}", "batch": B, "steps": S, "tags": K, "us": round(us_nll, 2),
                  "decode_us": round(us_dec, 2), "loss": float(loss.numpy())}), flush=True)
