"""Data-parallel masked-LM training: 2-rank NCCL data parallel == 1 rank on the global batch with bit-identical replicas
(needs >= 2 GPUs, skipped otherwise), the same harness in a world of one, and the order in which backward hands the
tied word embeddings' bucket to the allreduce / early optimizer update."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# the bars of tests/test_dist_gpu.py: the two arms differ only in the order of fp32 additions
LOSS_REL = 2e-3
WEIGHT_MEAN_ABS = 2e-5


@pytest.mark.parametrize("family", ["bert", "roberta"])
def test_two_rank_mlm_matches_single_rank_global_batch(family):
    from polus_b200 import _lib
    n = C.c_int(0)
    _lib.call("polus_device_count", C.byref(n))
    if n.value < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, POLUS_LOGGER_LEVEL="ERROR")
    run = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tests", "mlm_dp_parity.py"),
                          family], capture_output=True, text=True, timeout=600, env=env)
    assert run.returncode == 0, run.stderr[-3000:]
    lines = [l for l in run.stdout.splitlines() if l.startswith("MLMDPPARITY ")]
    assert len(lines) == 1, run.stdout[-2000:]
    r = json.loads(lines[0].split(" ", 1)[1])
    assert r["world"] == 2 and r["replicas_identical"], r
    assert r["vs_single_rank_rel"] < LOSS_REL, r
    assert r["weights_mean_abs_diff"] < WEIGHT_MEAN_ABS and r["word_mean_abs_diff"] < WEIGHT_MEAN_ABS, r
    assert r["weights_max_abs_diff"] <= 2.02 * r["lr"] * r["steps"], r


def test_mlm_dp_parity_harness_single_rank():
    """World of one: both arms are the same computation -- the harness itself must report exact agreement."""
    from polus_b200 import device
    from tests.mlm_dp_parity import run_mlm_dp_parity
    device.init(0)
    r = run_mlm_dp_parity(steps=3)
    assert r["world"] == 1 and r["replicas_identical"]
    assert r["vs_single_rank_rel"] < 1e-4 and r["weights_mean_abs_diff"] < 1e-6, r


def test_word_embedding_bucket_waits_for_both_gradient_producers():
    """The decoder node lists the word Param among its inputs, and the bucket holding the word table is launched only
    once backward has passed the embedding lookup (its first use), i.e. after both the decoder's weight gradient and the
    embedding scatter were issued.  Small buckets, so the word table is a bucket of its own."""
    from polus_b200 import comm, device, ops
    from tests.mlm_dp_parity import _build, make_batch
    device.init(0)
    model = _build(3, "bert")
    word = model.bert.bert.embeddings.word
    ids, mask, pos, lab, w = make_batch(np.random.default_rng(0), 4, 64, 997, 12, "bert")
    with ops.GradientTape() as tape:
        logits = model(input_ids=ids, attention_mask=mask, masked_lm_positions=pos, training=True)
        loss = model.loss({"masked_lm_ids": lab, "masked_lm_weights": w}, logits)
    nodes = list(tape.nodes)
    uses = [i for i, nd in enumerate(nodes) if any(t is word for t in nd.inputs)]
    assert len(uses) == 2, uses                                       # the embedding lookup and the decoder
    embed_idx, dec_idx = uses
    assert isinstance(nodes[dec_idx].output, ops.VocabLogits)
    weights = model.trainable_weights
    fired, cur = [], [None]
    small = 4 * word.size // 2                                          # the word table alone is >= bucket / 2

    def launch(b):
        fired.append((cur[0], [p for p in b[3]]))
    orig = comm.BUCKET_BYTES
    comm.BUCKET_BYTES = small
    try:
        before, flush = ops.bucket_schedule(nodes, weights, launch)
    finally:
        comm.BUCKET_BYTES = orig

    def hook(idx):
        cur[0] = idx
        before(idx)
    ops.run_backward(nodes, loss, hook)
    cur[0] = -1
    flush()
    word_fires = [at for at, ps in fired if any(p is word for p in ps)]
    assert word_fires and all(at is not None and at < embed_idx for at in word_fires), (word_fires, embed_idx, dec_idx)
    other = [at for at, ps in fired if not any(p is word for p in ps)]
    assert any(at is not None and at > embed_idx for at in other)     # the schedule does launch buckets early
    assert np.abs(word.grad.numpy()).sum() > 0
