"""Cost of masked-LM training on one GPU, in one process:
  1. polus_vocab_xent at V in {30522, 250002}, R = 10240 (B = 256 x P = 40): time per call and achieved bytes/s over the
     algorithmic one read + one write of the bf16 logits (the gradient pass re-reads the row, meant to hit L2), and the
     argmax-only call (labels NULL: the first pass alone).  NSETS logit buffers rotate, each larger than the 126 MB L2
     at V = 250002, so every call starts HBM-cold there;
  2. the masked-LM head alone (gather, transform, tied decoder, cross-entropy, and their backward, op by op) against the
     captured MLM step: the head's share of the step;
  3. BERT-base MLM training throughput at S = 128, P = 20 (B = 256) and S = 512, P = 80 (B = 64), next to the NER+CRF
     step at the same shapes;
  4. the GPU's name, power limit and SM clock, read by nvidia-smi before and after.
    python tools/mlm_time.py"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from polus_b200 import _lib, device, ops, tensor  # noqa: E402
from polus_b200.tensor import BF16, F32, I32, Tensor  # noqa: E402

R_XENT, NSETS, REPS = 10240, 2, 10
STEPS, WARMUP = 20, 6


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


def ev():
    e = C.c_void_p()
    _lib.call("polus_event_create", C.byref(e))
    return e


def elapsed_ms(fn, reps):
    e0, e1 = ev(), ev()
    device.device_sync()
    _lib.call("polus_event_record", e0, device.stream())
    for i in range(reps):
        fn(i)
    _lib.call("polus_event_record", e1, device.stream())
    device.device_sync()
    ms = C.c_float()
    _lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
    return ms.value


def xent_times():
    rng = np.random.default_rng(0)
    st = device.stream()
    R = R_XENT
    for V in (30522, 250002):
        ldl = (V + 7) // 8 * 8
        bufs = []
        for _ in range(NSETS):
            t = Tensor((R, ldl), BF16)
            row = Tensor.from_numpy(rng.standard_normal((64, ldl)).astype(np.float32), BF16)
            for r0 in range(0, R, 64):
                _lib.call("polus_memcpy_d2d", t.ptr + r0 * ldl * 2, row.ptr, 64 * ldl * 2, st)
            bufs.append(t)
        labels = Tensor.from_numpy(rng.integers(0, V, R).astype(np.int32), I32)
        weights = Tensor.from_numpy(np.ones(R, np.float32), F32)
        nll, amax, loss = Tensor((R,), F32), Tensor((R,), I32), Tensor((), F32)
        # the gradient overwrites the logits: later calls see gradients as logits, which costs the same
        call = lambda i: _lib.call("polus_vocab_xent", bufs[i % NSETS].ptr, R, V, ldl, labels.ptr, weights.ptr, nll.ptr,
                                   amax.ptr, loss.ptr, st)
        elapsed_ms(call, NSETS)
        us = elapsed_ms(call, REPS * NSETS) * 1e3 / (REPS * NSETS)
        nbytes = 2 * R * V * 2
        # labels NULL: pass 1 alone (one read of the logits); the difference is what the gradient pass costs
        am = lambda i: _lib.call("polus_vocab_xent", bufs[i % NSETS].ptr, R, V, ldl, None, None, None, amax.ptr, None, st)
        am_us = elapsed_ms(am, REPS * NSETS) * 1e3 / (REPS * NSETS)
        print(json.dumps({"vocab_xent": {"V": V, "R": R, "us": round(us, 1), "algorithmic_bytes": nbytes,
                                         "TB_s": round(nbytes / (us * 1e-6) / 1e12, 3), "argmax_only_us": round(am_us, 1),
                                         "argmax_only_TB_s": round(nbytes / 2 / (am_us * 1e-6) / 1e12, 3)}}), flush=True)
        del bufs


def _bert_base():
    from polus_b200.models import BertConfig
    return BertConfig()


def _mlm_feed(rng, B, S, P, V):
    from polus_b200.mlm import mask_tokens
    lens = rng.integers(S // 2, S + 1, B)
    mask = (np.arange(S)[None, :] < lens[:, None]).astype(np.int32)
    ids = np.where(mask > 0, rng.integers(1000, V, (B, S)), 0).astype(np.int32)
    ids, pos, lab, w = mask_tokens(ids, mask, vocab_size=V, mask_token_id=103, special_token_ids=(0, 101, 102, 103),
                                   max_predictions=P, rng=rng)
    x = {"input_ids": Tensor.from_numpy(ids, I32), "attention_mask": Tensor.from_numpy(mask, I32),
         "token_type_ids": Tensor((B, S), I32, zero=True), "masked_lm_positions": Tensor.from_numpy(pos, I32)}
    return x, {"masked_lm_ids": Tensor.from_numpy(lab, I32), "masked_lm_weights": Tensor.from_numpy(w, F32)}


def _ner_feed(rng, B, S, V):
    lens = rng.integers(S // 2, S + 1, B)
    mask = (np.arange(S)[None, :] < lens[:, None]).astype(np.int32)
    ids = np.where(mask > 0, rng.integers(1000, V, (B, S)), 0).astype(np.int32)
    tags = rng.integers(1, 4, (B, S)) * mask
    x = {"input_ids": Tensor.from_numpy(ids, I32), "attention_mask": Tensor.from_numpy(mask, I32),
         "token_type_ids": Tensor((B, S), I32, zero=True)}
    return x, Tensor.from_numpy(np.eye(4, dtype=np.float32)[tags], F32)


def step_ms(kind, B, S, P, rng):
    from polus_b200.mlm import BertMaskedLMModel
    from polus_b200.ner.models import BertNERModel
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    from polus_b200.utils import set_random_seed
    tensor.reset_arena()
    tensor._pool.release_cached()
    set_random_seed(42)
    cfg = _bert_base()
    if kind == "mlm":
        model = BertMaskedLMModel(cfg)
        feeds = [_mlm_feed(rng, B, S, P, cfg.vocab_size) for _ in range(2)]
    else:
        model = BertNERModel(cfg, output_classes=4, hidden_space=128, droupout_p=0.1)
        feeds = [_ner_feed(rng, B, S, cfg.vocab_size) for _ in range(2)]
    trainer = ClassifierTrainer(model, Adam(5e-5), model.loss)
    for i in range(WARMUP):
        last = trainer.train_step(*feeds[i % 2])
    float(last)
    holder = {}

    def one(i):
        holder["loss"] = trainer.train_step(*feeds[i % 2])
    ms = elapsed_ms(one, STEPS) / STEPS
    loss = float(holder["loss"])
    head_ms = None
    if kind == "mlm":
        head_ms = head_alone_ms(model, feeds[0], B, S, P)
    trainer.release_graphs()
    return ms, loss, head_ms


def head_alone_ms(model, feed, B, S, P):
    """The head's forward and backward, op by op, on an encoder output of the step's shape (includes launch gaps the
    captured step does not have, so it bounds the head's share from above)."""
    x, y = feed
    h = Tensor((B, S, model.config.hidden_size), BF16, zero=True)
    h.requires_grad = True

    def one(i):
        with ops.GradientTape() as tape:
            logits = model.cls(ops.gather_positions(h, x["masked_lm_positions"]))
            loss = model.loss(y, logits)
        tape.gradient(loss, model.cls.trainable_weights)
    one(0)
    return elapsed_ms(one, 10) / 10


def main():
    device.init(0)
    print(json.dumps({"gpu_before": gpu_info()}), flush=True)
    xent_times()
    rng = np.random.default_rng(1)
    for B, S, P in ((256, 128, 20), (64, 512, 80)):
        mlm_ms, mlm_loss, head_ms = step_ms("mlm", B, S, P, rng)
        ner_ms, ner_loss, _ = step_ms("ner", B, S, P, rng)
        print(json.dumps({"shape": {"B": B, "S": S, "P": P},
                          "mlm": {"step_ms": round(mlm_ms, 2), "seq_s": round(B / mlm_ms * 1e3, 1), "loss": round(mlm_loss, 3),
                                  "head_alone_ms": round(head_ms, 2), "head_share": round(head_ms / mlm_ms, 3)},
                          "ner_crf": {"step_ms": round(ner_ms, 2), "seq_s": round(B / ner_ms * 1e3, 1),
                                      "loss": round(ner_loss, 3)}}), flush=True)
    print(json.dumps({"gpu_after": gpu_info()}), flush=True)


if __name__ == "__main__":
    main()
