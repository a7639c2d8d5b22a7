#!/usr/bin/env python
"""Hunt for non-finite values in the data-parallel step (run under torchrun on >= 2 GPUs):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/nan_hunt.py [batch] [steps]

Several trials in one process, each a fresh model: the bench's warm-up sequence (op-by-op step, capture, broadcast) and
`steps` replays with the loss read every 10 steps.  At the first non-finite loss the trial reports which variables,
gradient spans and optimizer slots hold non-finite values."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


_KEEP = []


def nonfinite_report(trainer):
    from polus_b200 import device
    from polus_b200.tensor import Param
    bad = []
    for w in trainer.trainable_weights:
        if not isinstance(w, Param):
            continue
        a = w.numpy()
        g = w.grad.numpy()
        nb, ng = int((~np.isfinite(a)).sum()), int((~np.isfinite(g)).sum())
        if nb or ng:
            bad.append((w.name, tuple(w.shape), nb, ng))
    slots = []
    for t in trainer.optimizer.variables():
        a = t.numpy()
        slots.append(int((~np.isfinite(a)).sum()))
    return bad, slots


def trial(name, batch, steps, check_every=10, workload="ner_base"):
    rank = int(os.environ.get("RANK", "0"))
    trainer, batches, _, _, _ = bench.build_workload(workload, batch)
    t0 = time.time()
    for i in range(5):
        loss = trainer.train_step(*batches[i % len(batches)])
    from polus_b200 import comm

    def any_rank_bad(v):   # every rank must leave the loop at the same step (the step holds a collective)
        flags = comm._host_allgather(b"1" if not np.isfinite(v) else b"0")
        return any(f == b"1" for f in flags)
    first_bad = None
    if any_rank_bad(float(loss)):
        first_bad = 4
    if trainer.use_horovod and os.environ.get("NANHUNT_NOBCAST") != "1":
        trainer.broadcast_init_vars()
    dev = bench.to_device(batches)
    i = 0
    while first_bad is None and i < steps:
        last = trainer.train_step(*dev[i % len(dev)])
        i += 1
        if i % check_every == 0 and any_rank_bad(float(last)):
            first_bad = 5 + i
    from polus_b200.tensor import Param
    ch = next(w for w in trainer.trainable_weights if isinstance(w, Param)).chunk
    out = {"trial": name, "rank": rank, "g_ptr": hex(ch.g.ptr), "p_ptr": hex(ch.p.ptr), "first_nonfinite_step": first_bad, "loss": float(last) if first_bad is None else None,
           "s": round(time.time() - t0, 1)}
    if first_bad is not None:
        bad, slots = nonfinite_report(trainer)
        out["bad_vars"] = len(bad)
        out["bad_first"] = bad[:6]
        out["bad_last"] = bad[-6:]
        out["slots_nonfinite"] = slots
    if os.environ.get("NANHUNT_KEEP") == "1":      # never free anything a previous model owned (arena, slots, graphs)
        from polus_b200 import tensor as _t
        _KEEP.append((trainer, dev, _t.arena()))
    else:
        trainer.release_graphs()
    del trainer, dev
    print("NANHUNT " + json.dumps(out), flush=True)
    return first_bad


def main():
    batch = int(sys.argv[1]) if len(sys.argv) > 1 else 128
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 150
    import polus_b200
    from polus_b200 import device
    rank = int(os.environ.get("RANK", "0"))
    device.init(int(os.environ.get("LOCAL_RANK", str(rank))))
    polus_b200.PolusContext()
    variants = os.environ.get("NANHUNT_VARIANTS", ",".join(["base"] * 7)).split(",")
    for k, v in enumerate(variants):
        v, _, wl = v.partition(":")            # "base:cfg4" = bench.py's cfg4 workload
        wl, _, wb = (wl or "ner_base").partition("@")   # "base:cfg5@32" = ... at batch 32
        trial(f"{v}:{wl}#{k}", int(wb) if wb else batch, steps,
              check_every=int(os.environ.get("NANHUNT_CHECK_EVERY", "10")), workload=wl)
    sys.stdout.flush()
    os._exit(0)


if __name__ == "__main__":
    main()
