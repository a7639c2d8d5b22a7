"""Cost of RoBERTa position ids on one GPU, in one process:
  1. the embedding block (forward; backward = LayerNorm backward + scatter) with and without per-token position ids at
     B = 256, S = 256, H = 768, on a fully real batch and on a right-padded batch with about half pad tokens (row
     lengths uniform in 0..S).  Buffers rotate through NSETS copies of more than the 126 MB L2 each, so every launch
     reads HBM-cold data, as in tools/kernel_times.py;
  2. training throughput of RoBERTa-base NER+CRF against BERT-base NER+CRF (batch 256, S = 256, dropout 0.1, ragged
     batches), the two alternated over ROUNDS rounds;
  3. the GPU's name, power limit and SM clock, read by nvidia-smi before and after.
    python tools/roberta_time.py [rounds]"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from polus_b200 import _lib, device, ops, tensor  # noqa: E402
from polus_b200.tensor import BF16, F32, I32, Tensor  # noqa: E402

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 3
B, S, H, V, PAD = 256, 256, 768, 50265, 1
M = B * S
NSETS, REPS = 3, 10
STEPS, WARMUP = 20, 8


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


def ev():
    e = C.c_void_p()
    _lib.call("polus_event_create", C.byref(e))
    return e


def timeit(fn):
    """Microseconds per call, averaged over REPS passes through the NSETS buffer sets."""
    for k in range(NSETS):
        fn(k)
    e0, e1 = ev(), ev()
    device.device_sync()
    _lib.call("polus_event_record", e0, device.stream())
    for _ in range(REPS):
        for k in range(NSETS):
            fn(k)
    _lib.call("polus_event_record", e1, device.stream())
    device.device_sync()
    ms = C.c_float()
    _lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
    return ms.value * 1e3 / (REPS * NSETS)


def embedding_times():
    rng = np.random.default_rng(0)
    st = device.stream()
    f32 = lambda shape, scale=0.02: Tensor.from_numpy((rng.standard_normal(shape) * scale).astype(np.float32), F32)
    word, pos, typ = f32((V, H)), f32((514, H)), f32((1, H))
    gamma, beta = f32((H,), 1.0), f32((H,))
    gw, gp, gt, gg, gb = (Tensor(t.shape, F32, zero=True) for t in (word, pos, typ, gamma, beta))
    ys = [Tensor((M, H), BF16) for _ in range(NSETS)]
    zs = [Tensor((M, H), F32) for _ in range(NSETS)]
    means, rstds = [Tensor((M,), F32) for _ in range(NSETS)], [Tensor((M,), F32) for _ in range(NSETS)]
    dys = [Tensor.from_numpy(rng.standard_normal((M, H)).astype(np.float32), BF16) for _ in range(NSETS)]
    ws = Tensor((int(_lib.call("polus_embed_ws_floats", B, S, H)),), F32)
    ops.set_step(1)
    sp = ops.step_counter()
    out = []
    for batch in ("real", "half_padded"):
        ids = rng.integers(3, V, (B, S)).astype(np.int32)
        if batch == "half_padded":
            lens = rng.integers(0, S + 1, B)
            ids[np.arange(S)[None, :] >= lens[:, None]] = PAD
        ids_t = Tensor.from_numpy(ids, I32)
        tt_t = Tensor((B, S), I32, zero=True)
        pid_t = ops.position_ids_from_input_ids(ids_t, PAD)
        pid_us = timeit(lambda k: _lib.call("polus_position_ids", ids_t.ptr, B, S, PAD, pid_t.ptr, st))
        row = {"batch": batch, "pad_fraction": round(float((ids == PAD).mean()), 3), "position_ids_us": round(pid_us, 2)}
        for label, fwd, bwd, extra in (("bert", "polus_embed_ln_fwd", "polus_embed_ln_bwd", ()),
                                       ("pos_ids", "polus_embed_ln_fwd_pos", "polus_embed_ln_bwd_pos", (pid_t.ptr, 514))):
            row[f"fwd_{label}_us"] = round(timeit(lambda k: _lib.call(
                fwd, ids_t.ptr, tt_t.ptr, word.ptr, pos.ptr, typ.ptr, gamma.ptr, beta.ptr, B, S, H, V, 1, 1e-5, 0.1, 7, 3, sp,
                ys[k].ptr, zs[k].ptr, means[k].ptr, rstds[k].ptr, *extra, st)), 2)
            row[f"bwd_{label}_us"] = round(timeit(lambda k: _lib.call(
                bwd, dys[k].ptr, zs[k].ptr, means[k].ptr, rstds[k].ptr, gamma.ptr, ids_t.ptr, tt_t.ptr, B, S, H, V, 1, 0.1, 7,
                3, sp, gw.ptr, gp.ptr, gt.ptr, gg.ptr, gb.ptr, ws.ptr, *extra, st)), 2)
        row["bwd_ratio"] = round(row["bwd_pos_ids_us"] / row["bwd_bert_us"], 3)
        print(json.dumps({"embedding": row}), flush=True)
        out.append(row)
    return out


def training_seq_s(family, rng):
    from polus_b200.models import BertConfig
    from polus_b200.ner.models import BertNERModel
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    from polus_b200.utils import set_random_seed
    tensor.reset_arena()
    tensor._pool.release_cached()
    set_random_seed(42)
    if family == "roberta":
        cfg = BertConfig(model_type="roberta", pad_token_id=PAD, vocab_size=V, max_position_embeddings=514, type_vocab_size=1,
                         layer_norm_eps=1e-5)
        pad = PAD
    else:
        cfg = BertConfig()
        pad = 0
    model = BertNERModel(cfg, output_classes=4, hidden_space=128, droupout_p=0.1)
    trainer = ClassifierTrainer(model, Adam(5e-5), model.loss)
    feeds = []
    for _ in range(2):
        lens = rng.integers(S // 4, S + 1, B)
        mask = (np.arange(S)[None, :] < lens[:, None]).astype(np.int32)
        ids = np.where(mask > 0, rng.integers(3, cfg.vocab_size, (B, S)), pad).astype(np.int32)
        tags = rng.integers(1, 4, (B, S)) * mask
        x = {"input_ids": Tensor.from_numpy(ids, I32), "attention_mask": Tensor.from_numpy(mask, I32),
             "token_type_ids": Tensor((B, S), I32, zero=True)}
        feeds.append((x, Tensor.from_numpy(np.eye(4, dtype=np.float32)[tags], F32)))
    for i in range(WARMUP):
        last = trainer.train_step(*feeds[i % 2])
    float(last)
    e0, e1 = ev(), ev()
    device.device_sync()
    _lib.call("polus_event_record", e0, device.stream())
    for i in range(STEPS):
        last = trainer.train_step(*feeds[i % 2])
    _lib.call("polus_event_record", e1, device.stream())
    loss = float(last)
    device.device_sync()
    ms = C.c_float()
    _lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
    trainer.release_graphs()
    return B * STEPS / (ms.value * 1e-3), loss


def main():
    device.init(0)
    print(json.dumps({"gpu_before": gpu_info()}), flush=True)
    embedding_times()
    rng = np.random.default_rng(1)
    runs = {"bert": [], "roberta": []}
    for r in range(ROUNDS):
        for family in (("bert", "roberta") if r % 2 == 0 else ("roberta", "bert")):
            sps, loss = training_seq_s(family, rng)
            runs[family].append(round(sps, 1))
            print(json.dumps({"round": r, "model": f"{family}-base NER+CRF", "seq_s": round(sps, 1), "loss": round(loss, 3)}),
                  flush=True)
    med = {k: float(np.median(v)) for k, v in runs.items()}
    print(json.dumps({"training_seq_s": runs, "median": med, "roberta_over_bert": round(med["roberta"] / med["bert"], 4),
                      "batch": B, "seq": S, "gpu_after": gpu_info()}), flush=True)


if __name__ == "__main__":
    main()
