"""Isolated timing of the CRF loss kernel (polus_crf_nll, K=4, S=256):  python tools/crf_time.py [batch]"""
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from polus_b200 import _lib, device  # noqa: E402
from polus_b200.tensor import F32, I32, Tensor  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 128
S, K, NSETS, REPS = 256, 4, 4, 10
device.init(0)
st = device.stream()
rng = np.random.default_rng(0)
em = [Tensor.from_numpy(rng.standard_normal((B, S, K)).astype(np.float32), F32) for _ in range(NSETS)]
tg = Tensor.from_numpy(rng.integers(1, K, (B, S)).astype(np.int32), I32)
tr = Tensor.from_numpy(rng.standard_normal((K, K)).astype(np.float32), F32)
nll, loss, ge, gt = Tensor((B,), F32), Tensor((), F32, zero=True), Tensor((B, S, K), F32), Tensor((K, K), F32, zero=True)


def run(k):
    _lib.call("polus_crf_nll", em[k].ptr, tg.ptr, None, tr.ptr, None, B, S, K, nll.ptr, loss.ptr, ge.ptr, gt.ptr, st)


for k in range(NSETS):
    run(k)
e0, e1 = C.c_void_p(), C.c_void_p()
_lib.call("polus_event_create", C.byref(e0))
_lib.call("polus_event_create", C.byref(e1))
device.device_sync()
_lib.call("polus_event_record", e0, st)
for r in range(REPS):
    for k in range(NSETS):
        run(k)
_lib.call("polus_event_record", e1, st)
device.device_sync()
ms = C.c_float()
_lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
us = ms.value * 1e3 / (REPS * NSETS)
print(json.dumps({"kernel": "crf_nll K=4", "batch": B, "steps": S, "us": round(us, 2), "loss": float(loss.numpy())}), flush=True)
