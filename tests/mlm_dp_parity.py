"""N-rank data-parallel parity of masked-LM training: N ranks, each on its 1/N slice of a global batch with lr x N and
averaged gradients, must follow the same trajectory as one process on the whole batch with lr x N, and the replicas
must stay bit-identical.  This is the check on the tied word embeddings' two gradient producers: the embedding scatter
(main stream) and the decoder's weight-gradient GEMM (side stream during capture), which must both have landed in
word.grad before that bucket's allreduce and early optimizer update.

The masked-LM loss is normalised per replica (sum w nll / sum w over the rank's own rows, as TF BERT's pretraining
computes it per replica), so the N-rank average equals the whole-batch loss only when every slice carries the same
sum of weights: the batch below gives every row the same number of masked tokens.

Same structure as tests/dp_parity.py (the NER harness), with a BertMaskedLMModel; run as
    python -m torch.distributed.run --nproc-per-node 2 tests/mlm_dp_parity.py"""
import json
import os

import numpy as np


def _build(seed, family):
    from polus_b200 import ops, tensor
    from polus_b200.mlm import BertMaskedLMModel
    from polus_b200.models import BertConfig
    from polus_b200.utils import set_random_seed
    tensor.reset_arena()
    set_random_seed(seed)
    ops.set_step(0)
    kw = dict(vocab_size=997, hidden_size=128, num_hidden_layers=2, num_attention_heads=4, intermediate_size=256,
              hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    if family == "roberta":
        kw.update(model_type="roberta", pad_token_id=1, type_vocab_size=1, layer_norm_eps=1e-5, max_position_embeddings=66)
    else:
        kw.update(max_position_embeddings=64)
    return BertMaskedLMModel(BertConfig(**kw))


def make_batch(rng, B, S, V, P, family):
    """Full-length rows: every row masks the same n = min(P, round(0.15 (S - 2))) tokens, so equal slices carry equal
    sums of weights."""
    from polus_b200.mlm import mask_tokens
    ids = rng.integers(4, V, (B, S)).astype(np.int32)
    ids[:, 0], ids[:, -1] = 2, 3
    mask = np.ones((B, S), np.int32)
    ids, pos, lab, w = mask_tokens(ids, mask, vocab_size=V, mask_token_id=0 if family == "roberta" else 1,
                                   special_token_ids=(0, 1, 2, 3), max_predictions=P, rng=rng)
    assert np.all(w.sum(1) == w[0].sum())
    return ids, mask, pos, lab, w


def run_mlm_dp_parity(steps=3, per_rank=4, seq=64, P=12, base_lr=1e-3, seed=11, family="bert", log=None):
    """Returns {"world", "replicas_identical", "vs_single_rank_rel", "weights_max_abs_diff", "weights_mean_abs_diff",
    "word_mean_abs_diff", "lr", "steps", "losses_dp_mean", "losses_single"} on every rank."""
    from polus_b200 import comm, hvd, tensor
    from polus_b200.mock import horovod as mock_hvd
    from polus_b200.optimizers import Adam
    from polus_b200.training import ClassifierTrainer
    log = log or (lambda m: None)
    h = hvd()
    world, rank = h.size(), (h.rank() if hasattr(h, "rank") else 0)
    GB = per_rank * world
    ids, mask, pos, lab, w = make_batch(np.random.default_rng(5), GB, seq, 997, P, family)

    def feed(lo, hi):
        return ({"input_ids": ids[lo:hi], "attention_mask": mask[lo:hi], "token_type_ids": np.zeros_like(ids[lo:hi]),
                 "masked_lm_positions": pos[lo:hi]}, {"masked_lm_ids": lab[lo:hi], "masked_lm_weights": w[lo:hi]})

    # ---- arm 1: N ranks, each on its slice
    model = _build(seed, family)
    word = model.bert.bert.embeddings.word
    x, y = feed(rank * per_rank, (rank + 1) * per_rank)
    opt = Adam(base_lr)
    trainer = ClassifierTrainer(model, opt, model.loss)
    if trainer.use_horovod:
        trainer.broadcast_init_vars()
    losses = [float(trainer.train_step(x, y)) for _ in range(steps)]
    log(f"dp arm done, losses {losses}")
    w_dp = [p.numpy().copy() for p in model.weights]
    word_dp = word.numpy().copy()
    digest = float(sum(np.abs(a.astype(np.float64)).sum() for a in w_dp))
    probe = word_dp.reshape(-1)[:16].astype(np.float64).tolist()
    lr_used = float(opt.learning_rate.read_value())
    mine = json.dumps({"rank": rank, "losses": losses, "digest": digest, "probe": probe}).encode()
    everyone = [json.loads(b.decode()) for b in (comm._host_allgather(mine) if world > 1 else [mine])]
    everyone.sort(key=lambda d: d["rank"])
    identical = all(d["digest"] == everyone[0]["digest"] and d["probe"] == everyone[0]["probe"] for d in everyone)
    losses_dp_mean = np.mean([d["losses"] for d in everyone], axis=0)
    trainer.release_graphs()
    del trainer, model

    # ---- arm 2: one rank on the whole global batch with lr x N, no collective
    model = _build(seed, family)
    word = model.bert.bert.embeddings.word
    xg, yg = feed(0, GB)
    opt1 = Adam(base_lr * world)
    trainer1 = ClassifierTrainer(model, opt1, model.loss)
    if trainer1.use_horovod:   # undo what the constructor did for the N-rank world
        opt1.learning_rate.assign(base_lr * world)
        opt1.grad_scale = 1.0
        trainer1.use_horovod, trainer1.hvd = False, mock_hvd
    losses1 = [float(trainer1.train_step(xg, yg)) for _ in range(steps)]
    w_1 = [p.numpy().copy() for p in model.weights]
    word_1 = word.numpy().copy()
    log("single arm done")
    rel = float(np.max(np.abs(losses_dp_mean - np.asarray(losses1)) / np.maximum(np.abs(losses1), 1e-12)))
    wdiff = float(max(np.abs(a - b).max() for a, b in zip(w_dp, w_1)))
    wmean = float(sum(np.abs(a - b).sum() for a, b in zip(w_dp, w_1)) / sum(a.size for a in w_dp))
    trainer1.release_graphs()
    del trainer1, model
    tensor.reset_arena()
    return {"world": world, "replicas_identical": bool(identical), "vs_single_rank_rel": rel, "weights_max_abs_diff": wdiff,
            "weights_mean_abs_diff": wmean, "word_mean_abs_diff": float(np.abs(word_dp - word_1).mean()), "lr": lr_used,
            "steps": steps, "losses_dp_mean": [float(v) for v in losses_dp_mean], "losses_single": [float(v) for v in losses1]}


if __name__ == "__main__":   # python -m torch.distributed.run ... tests/mlm_dp_parity.py [family]
    import faulthandler
    import sys
    import time
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    faulthandler.dump_traceback_later(int(os.environ.get("DP_PARITY_WATCHDOG", "150")), exit=True)
    t0 = time.time()
    r = int(os.environ.get("RANK", "0"))

    def _log(m):
        sys.stderr.write(f"[mlm_dp_parity r{r} +{time.time() - t0:5.1f}s] {m}\n")
        sys.stderr.flush()
    import polus_b200
    from polus_b200 import device
    device.init(int(os.environ.get("LOCAL_RANK", r)))
    polus_b200.PolusContext()
    out = run_mlm_dp_parity(steps=4, family=sys.argv[1] if len(sys.argv) > 1 else "bert", log=_log)
    if r == 0:
        print("MLMDPPARITY " + json.dumps(out), flush=True)
    faulthandler.cancel_dump_traceback_later()
    sys.stdout.flush()
    os._exit(0)   # as tests/dp_parity.py: leave without tearing the communicator down
