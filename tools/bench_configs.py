"""Throughput of the two larger BASELINE.json configurations on one GPU (parity cases in tests/, timed here):
    cfg4  BERT-base cross-encoder ranking, S=512, pairwise softplus loss       (polus_b200.ir.models.BertCrossEncoder)
    cfg5  BERT-large-sized encoder (L24 H1024 nh16 I4096) NER + CRF, S=512     (polus_b200.ner.models.BertNERModel)
Same method as bench.py's `value`: batches resident in HBM, captured-graph replays, CUDA events, pre-heated.
    python tools/bench_configs.py [cfg4|cfg5|all] [batch] [steps]
Train GEMM FLOPs per sequence (SURVEY §8d): cfg4 289.91 GFLOP, cfg5 1005.0 GFLOP."""
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import polus_b200  # noqa: E402,F401
from polus_b200 import _lib, device, tensor  # noqa: E402
from polus_b200.models import BertConfig  # noqa: E402
from polus_b200.optimizers import Adam  # noqa: E402
from polus_b200.schedulers import warmup_scheduler  # noqa: E402
from polus_b200.training import ClassifierTrainer  # noqa: E402
from polus_b200.utils import set_random_seed  # noqa: E402

which = sys.argv[1] if len(sys.argv) > 1 else "all"
batch = int(sys.argv[2]) if len(sys.argv) > 2 else 16
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 20
S = 512
PEAK = 1366.3
try:
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")) as f:
        PEAK = json.load(f).get("bf16_tflops_sustained", PEAK)
except Exception:
    pass


def ev():
    e = C.c_void_p()
    _lib.call("polus_event_create", C.byref(e))
    return e


def inputs(rng, B, vocab, pair):
    ids = rng.integers(1000, vocab, size=(B, S)).astype(np.int32)
    ids[:, 0], ids[:, -1] = 101, 102
    tt = np.zeros((B, S), np.int32)
    if pair:  # [CLS] q [SEP] d [SEP]: token types split at U{16..64}
        for b, cut in enumerate(rng.integers(16, 65, size=B)):
            ids[b, cut] = 102
            tt[b, cut + 1:] = 1
    return {"input_ids": ids, "attention_mask": np.ones((B, S), np.int32), "token_type_ids": tt}


def run(name):
    tensor.reset_arena()
    set_random_seed(42)
    rng = np.random.default_rng(3)
    if name == "cfg4":
        from polus_b200.ir.models import BertCrossEncoder, pairwise_softplus_loss
        cfg = BertConfig()
        model = BertCrossEncoder(cfg)
        loss = pairwise_softplus_loss
        feeds = [(inputs(rng, batch, cfg.vocab_size, True), np.zeros(batch, np.float32)) for _ in range(2)]
        gflop, label = 289.91, "BERT-base cross-encoder, S=512, pairwise softplus loss"
    else:
        from polus_b200.ner.models import BertNERModel
        cfg = BertConfig(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096)
        model = BertNERModel(cfg, output_classes=4, hidden_space=128, droupout_p=0.1)
        loss = model.loss
        feeds = []
        for _ in range(2):
            y = np.eye(4, dtype=np.float32)[rng.integers(1, 4, size=(batch, S))]
            feeds.append((inputs(rng, batch, cfg.vocab_size, False), y))
        gflop, label = 1005.0, "BERT-large-sized encoder (L24 H1024 nh16 I4096) NER + CRF, S=512"
    trainer = ClassifierTrainer(model, Adam(warmup_scheduler(10000, 5e-5)), loss)
    dev = [({k: tensor.Tensor.from_numpy(v, tensor.I32) for k, v in x.items()}, tensor.Tensor.from_numpy(y, tensor.F32))
           for x, y in feeds]
    for i in range(4):
        last = trainer.train_step(*dev[i % 2])
    float(last)
    pre = max(20, int(1500 / 40))
    for i in range(pre):
        last = trainer.train_step(*dev[i % 2])
    float(last)
    e0, e1 = ev(), ev()
    device.device_sync()
    l0 = _lib.call("polus_launch_count")
    _lib.call("polus_event_record", e0, device.stream())
    for i in range(steps):
        last = trainer.train_step(*dev[i % 2])
    _lib.call("polus_event_record", e1, device.stream())
    lv = float(last)
    device.device_sync()
    ms = C.c_float()
    _lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
    per = ms.value / steps
    sps = batch / (per * 1e-3)
    fused = _lib.call("polus_attention_supported", S, 64) == 1
    print(json.dumps({"config": name, "workload": label, "batch": batch, "seq_len": S, "ms_per_step": round(per, 3),
                      "sequences_per_s": round(sps, 1), "step_mfu_vs_sustained_bf16": round(sps * gflop / 1e3 / PEAK, 4),
                      "fused_attention": fused, "launches_per_step": int((_lib.call("polus_launch_count") - l0) / steps),
                      "loss_last": lv}), flush=True)


device.init(0)
for n in (["cfg4", "cfg5"] if which == "all" else [which]):
    run(n)
