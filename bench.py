#!/usr/bin/env python
"""Headline benchmark: training sequences/s of BERT-base NER (+CRF) at seq 256 on N B200s (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU port of the reference step (oracle/torch_ref.py)

One "step" = one full optimisation step (forward, CRF loss, backward, [allreduce], Adam) of
polus_b200.training.ClassifierTrainer.train_step on one synthetic batch per GPU.
`value`  : inputs already resident in HBM, K captured-graph replays, CUDA events, max over ranks.
`e2e`    : the same K steps fed from HOST numpy batches through the public trainer API: pinned-memory
           H2D copy of every input and the D2H read of the loss are inside the timed region.
`roofline`: tcgen05 GEMM launches (the dominant kernel family, ~all FLOPs).  One op-by-op step counts the launches and
           their 2mnk FLOPs; `frac` = those FLOPs / the CUDA-event time of a captured replay of the step in which
           every other kernel entry point is a no-op (same order, buffers, streams), vs the measured sustained bf16
           peak; `frac_marginal` = the same FLOPs / (step time - step time with the GEMMs removed).  `traffic` and
           `tensor_pipe_active_pct` are read from the newest profiles/rNN_gemm_roofline.json (an ncu capture).
`strong_gb256`: the same step at global batch 256 split over the N GPUs (BASELINE.json configs[2]).
`configs`  : device-resident throughput of BASELINE.json configs[3] (cross-encoder S=512) and configs[4] (BERT-large
           dims S=512), data parallel over the same N GPUs.
`dp_parity`: N > 1 only -- N ranks on slices of a global batch vs one rank on the whole batch (tests/dp_parity.py).

--dump-outputs DIR: each timed region starts from the model's initial weights (restore_state) and, after them, rank 0
writes the loss of each region's last step as DIR/<name>.npy (dump_outputs), so that two builds run with the same
arguments (identical seeded inputs and starting weights) can be compared output for output.  Two runs of one build
still differ in the last bits of every step's float-atomic reductions, and the steps of a region compound that: on a
B200 the losses agree to <1e-7 relative after 5 steps at batch 32, and to ~1e-6..1e-5 after 20 steps at batch 256.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEQ = 256
TRAIN_GFLOP_PER_SEQ = 137.71  # BASELINE.md §3 (GEMM FLOPs, fwd+bwd = 3x fwd), BERT-base S=256


def workload_name(batch):
    return (f"BERT-base (L12 H768 nh12 I3072) polus.ner token classification + CRF, seq {SEQ}, "
            f"batch {batch}/GPU, dropout 0.1, Adam+warmup")


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_batches(n, batch, seq, vocab, K, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        ids = rng.integers(1000, vocab, size=(batch, seq)).astype(np.int32)
        ids[:, 0], ids[:, -1] = 101, 102
        mask = np.ones((batch, seq), np.int32)  # throughput config: full-length sequences (SURVEY §8d)
        tt = np.zeros((batch, seq), np.int32)
        tags = rng.integers(1, K, size=(batch, seq))
        y = np.eye(K, dtype=np.float32)[tags]
        out.append(({"input_ids": ids, "attention_mask": mask, "token_type_ids": tt}, y))
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import torch_ref
    batch = args.ref_batch
    sps, dt, threads = torch_ref.time_train_steps(batch=batch, seq=SEQ, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": "train_sequences_per_second", "value": sps, "unit": "sequences/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.batch), "global_batch": args.batch * args.gpus, "seq_len": SEQ,
                       "parallelism": f"dp{args.gpus}", "per_step_sample": f"{batch} sequences of the same workload per timed step",
                       "note": "CPU port of the reference step (TensorFlow is not installable in this image; oracle/torch_ref.py)"},
            "cpu_baseline": {"value": sps, "unit": "sequences/s", "cores": threads, "kind": "port",
                             "sample": f"{args.steps} steps of {batch} sequences x {SEQ} tokens"},
            "e2e": {"value": sps, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


_T0 = time.time()


def dbg(msg):
    if os.environ.get("BENCH_DEBUG"):
        sys.stderr.write(f"[bench r{os.environ.get('RANK', '0')} +{time.time() - _T0:6.1f}s] {msg}\n")
        sys.stderr.flush()


def build_workload(name, batch, seq=None):
    """(trainer, host batches, train GFLOP per sequence, label, seq).  `ner_base` = BASELINE.json configs[1] (the
    headline), `cfg4` / `cfg5` = configs[3] / configs[4] (SURVEY §8d sizes)."""
    from polus_b200 import tensor
    from polus_b200.models import BertConfig
    from polus_b200.optimizers import Adam
    from polus_b200.schedulers import warmup_scheduler
    from polus_b200.training import ClassifierTrainer
    from polus_b200.utils import set_random_seed
    rank = int(os.environ.get("RANK", "0"))
    tensor.reset_arena()
    tensor._pool.release_cached()
    set_random_seed(42)
    K = 4
    if name == "ner_base":
        from polus_b200.ner.models import BertNERModel
        S = seq or SEQ
        cfg = BertConfig()  # BERT-base: L12 H768 nh12 I3072 vocab 30522, dropout 0.1
        model = BertNERModel(cfg, output_classes=K, hidden_space=128, droupout_p=0.1)
        loss, gflop, label = model.loss, TRAIN_GFLOP_PER_SEQ, workload_name(batch)
        feeds = synthetic_batches(4, batch, S, cfg.vocab_size, K, seed=1 + rank)
    elif name == "cfg4":
        from polus_b200.ir.models import BertCrossEncoder, pairwise_softplus_loss
        S = seq or 512
        cfg = BertConfig()
        model = BertCrossEncoder(cfg)
        loss, gflop = pairwise_softplus_loss, 289.91
        label = f"polus.ir BERT-base cross-encoder, seq {S}, pairwise softplus loss, batch {batch}/GPU"
        rng = np.random.default_rng(3 + rank)
        feeds = []
        for _ in range(2):
            x, _ = synthetic_batches(1, batch, S, cfg.vocab_size, K, seed=int(rng.integers(1 << 30)))[0]
            for b_, cut in enumerate(rng.integers(16, 65, size=batch)):  # [CLS] q [SEP] d [SEP]: token types split at U{16..64}
                x["input_ids"][b_, cut] = 102
                x["token_type_ids"][b_, cut + 1:] = 1
            feeds.append((x, np.zeros(batch, np.float32)))
    elif name == "cfg5":
        from polus_b200.ner.models import BertNERModel
        S = seq or 512
        cfg = BertConfig(hidden_size=1024, num_hidden_layers=24, num_attention_heads=16, intermediate_size=4096)
        model = BertNERModel(cfg, output_classes=K, hidden_space=128, droupout_p=0.1)
        loss, gflop = model.loss, 1005.0
        label = f"BERT-large-sized encoder (L24 H1024 nh16 I4096) polus.ner + CRF, seq {S}, batch {batch}/GPU"
        feeds = synthetic_batches(2, batch, S, cfg.vocab_size, K, seed=5 + rank)
    else:
        raise ValueError(name)
    trainer = ClassifierTrainer(model, Adam(warmup_scheduler(10000, 5e-5)), loss)
    return trainer, feeds, gflop, label, S


class Timer:
    """CUDA-event timing of K train_step calls, barrier + device sync on both sides, max over ranks by the caller."""

    def __init__(self, world):
        import ctypes as C
        from polus_b200 import _lib, comm, device
        self.C, self._lib, self.comm, self.device, self.world = C, _lib, comm, device, world

    def ev(self):
        e = self.C.c_void_p()
        self._lib.call("polus_event_create", self.C.byref(e))
        return e

    def barrier(self):
        self.device.device_sync()
        if self.world > 1:
            self.comm.barrier()

    def max_over_ranks(self, values):
        if self.world == 1:
            return list(values)
        allv = [json.loads(b.decode()) for b in self.comm._host_allgather(json.dumps(list(values)).encode())]
        return [max(a[i] for a in allv) for i in range(len(values))]

    def timed(self, trainer, feed, steps):
        _lib, device = self._lib, self.device
        e0, e1 = self.ev(), self.ev()
        self.barrier()
        l0 = _lib.call("polus_launch_count")
        _lib.call("polus_event_record", e0, device.stream())
        last = None
        for i in range(steps):
            last = trainer.train_step(*feed[i % len(feed)])
        _lib.call("polus_event_record", e1, device.stream())
        float(last)
        self.barrier()
        ms = self.C.c_float()
        _lib.call("polus_event_elapsed_ms", e0, e1, self.C.byref(ms))
        return ms.value, _lib.call("polus_launch_count") - l0, float(last)


def initial_state(trainer, x):
    """Host copy of every trainable weight before the first training step.  A forward pass without training builds the
    lazily created variables (NER head, CRF) first; it updates nothing."""
    trainer.model(**x, training=False)
    return [(w, w.numpy()) for w in trainer.model.trainable_weights]


def restore_state(trainer, start):
    """Back to the weights of initial_state() with zeroed Adam moments.  The gradient reductions add with float atomics,
    so each training step differs from run to run in the last bits and successive steps compound that; timed regions
    that start from this state start from the same weights on every run.  The step counter keeps its value: the
    learning-rate schedule and the dropout streams go on as they would without the restore."""
    from polus_b200 import _lib, device
    for w, value in start:
        w.assign(value)
    for slot in trainer.optimizer.variables():   # Adam's first and second moments
        _lib.call("polus_memset", slot.ptr, 0, slot.nbytes, device.stream())
    device.device_sync()


def dump_outputs(out_dir, losses):
    """What a caller of the timed train steps receives: the loss of the last step of each timed region, as
    DIR/loss_<region>.npy (float32, shape (1,))."""
    os.makedirs(out_dir, exist_ok=True)
    for region, value in losses.items():
        np.save(os.path.join(out_dir, f"loss_{region}.npy"), np.asarray([value], np.float32))


def to_device(batches):
    from polus_b200 import tensor
    out = []
    for x, y in batches:
        out.append(({k: tensor.Tensor.from_numpy(v, tensor.I32) for k, v in x.items()}, tensor.Tensor.from_numpy(y, tensor.F32)))
    return out


def quick_config(name, batch, steps, timer, world, preheat=15):
    """Device-resident throughput of one of the other BASELINE configs (same method as `value`)."""
    trainer, feeds, gflop, label, S = build_workload(name, batch)
    dev = to_device(feeds)
    for i in range(4):
        last = trainer.train_step(*dev[i % len(dev)])
    float(last)
    if trainer.use_horovod:
        trainer.broadcast_init_vars()
    for i in range(preheat):
        last = trainer.train_step(*dev[i % len(dev)])
    float(last)
    ms, launches, loss = timer.timed(trainer, dev, steps)
    (ms,) = timer.max_over_ranks([ms])
    trainer.release_graphs()
    peaks, _ = read_peaks()
    peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    sps = batch * world * steps / (ms * 1e-3)
    return {"workload": label, "seq_s": sps, "ms_per_step": ms / steps, "batch_per_gpu": batch, "seq_len": S, "steps": steps,
            "step_mfu": sps / world * gflop / 1e3 / peak, "launches_per_step": int(launches / steps), "loss_last": loss}


def load_roofline_capture():
    """Per-launch DRAM traffic and tensor-pipe activity of the GEMM kernel from the newest committed ncu capture
    (tools/ncu_summary.py --roofline-json): profiles/rNN_gemm_roofline.json, highest round first."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_gemm_roofline.json")), reverse=True):
        try:
            with open(path) as f:
                doc = json.load(f)
            doc["_path"] = os.path.relpath(path, ROOT)
            return doc
        except Exception:
            continue
    return None


def run_ours(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", str(rank)))
    import ctypes as C
    import polus_b200
    from polus_b200 import _lib, comm, device, ops

    device.init(local_rank)
    dbg("device ready")
    polus_b200.PolusContext()  # brings NCCL up when WORLD_SIZE > 1
    dbg("context ready")
    timer = Timer(world)
    barrier, timed = timer.barrier, timer.timed

    # ---- N-rank == single-rank-on-the-global-batch parity, before anything is timed (tests/dp_parity.py)
    dp_parity = None
    if world > 1 and not args.no_dp_parity:
        from tests.dp_parity import run_dp_parity
        dp_parity = run_dp_parity(steps=3, log=dbg)
        dbg(f"dp parity: {dp_parity}")

    trainer, batches, _, _, _ = build_workload("ner_base", args.batch)
    start = initial_state(trainer, batches[0][0]) if args.dump_outputs else None
    dbg("model built")
    for i in range(max(args.warmup, 3)):
        loss = trainer.train_step(*batches[i % len(batches)])
        if i < 3:
            device.device_sync()
            dbg(f"warmup step {i} done")
    float(loss)
    dbg("warmup done")
    if trainer.use_horovod:
        trainer.broadcast_init_vars()
    dev_batches = to_device(batches)

    # bring the GPU to its steady operating point (power-capped clocks) before either timed region: the first seconds
    # after start-up run at boost clocks, which made whichever region came first look 3-5 % faster than the other
    # (a FIXED number of steps: every rank must issue the same sequence of collectives)
    for i in range(args.preheat_steps):
        last = trainer.train_step(*dev_batches[i % len(dev_batches)])
        if i % 10 == 9:
            float(last)
    dbg("pre-heat done")
    if start is not None:
        restore_state(trainer, start)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_dev, launches, loss_dev = timed(trainer, dev_batches, args.steps)
    dbg("timed (resident) done")
    if start is not None:
        restore_state(trainer, start)
    ms_e2e, _, loss_e2e = timed(trainer, batches, args.steps)
    h2d = trainer.last_h2d_bytes  # bytes the public API copied host -> device for ONE step of the e2e region
    dbg("timed (e2e) done")
    clocks = sampler.stop() if sampler else None
    ms_dev, ms_e2e = timer.max_over_ranks([ms_dev, ms_e2e])
    if not (np.isfinite(loss_dev) and np.isfinite(loss_e2e)):
        # a step that diverged runs on NaNs (less switching, higher clocks): its timing is not a measurement
        raise RuntimeError(f"bench: non-finite training loss (resident {loss_dev}, e2e {loss_e2e}) on rank {rank}")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"resident": loss_dev, "e2e": loss_e2e})

    # ---- roofline of the dominant kernel family (tcgen05 GEMMs, ~all FLOPs of the step)
    # (1) one op-by-op step counts the launches and their algorithmic FLOPs (2mnk each);
    # (2) a second captured graph of the SAME step in which every kernel entry point except polus_gemm_tc is a
    #     no-op (polus_b200._lib.set_only) replays exactly the step's GEMM launches -- same order, shapes, buffers
    #     and streams -- and is timed with CUDA events like the step itself: duration of the GEMM launches of one
    #     step, free of host launch latency (bracketing single launches op-by-op charges ~5 us of host time each);
    # (3) the marginal figure (step minus the step with polus_gemm_tc ablated) is reported next to it.
    roof = None
    prof = []
    ops.GEMM_PROFILE = prof
    trainer.use_graph = False
    float(trainer.train_step(*batches[0]))  # every rank runs it (it contains the gradient allreduce)
    ops.GEMM_PROFILE = None
    trainer.use_graph = True
    tot_flop = sum(flop for kind, flop, _, _ in prof if kind == "tc")
    n_tc = sum(1 for kind, _, _, _ in prof if kind == "tc")
    barrier()

    def replay_ms(only=None, ablate=None, feed=None):
        feed = dev_batches if feed is None else feed
        saved = (trainer._compiled, trainer._warm, _lib._ONLY, _lib._ABLATE)
        trainer._compiled, trainer._warm = {}, set()
        if only is not None:
            _lib.set_only(only)
        if ablate is not None:
            _lib._ABLATE = frozenset(ablate)
        try:
            for i in range(3):
                float(trainer.train_step(*feed[i % len(feed)]))
            ms, _, _ = timed(trainer, feed, args.steps)
        finally:
            trainer.release_graphs()
            trainer._compiled, trainer._warm = saved[0], saved[1]
            _lib._ONLY, _lib._ABLATE = saved[2], saved[3]
        return ms / args.steps

    gemm_only_ms = replay_ms(only={"polus_gemm_tc"})
    no_gemm_ms = replay_ms(ablate={"polus_gemm_tc"})
    dbg("gemm-only replays done")
    no_comm_ms = None
    if world > 1:
        # the same step without its collective: step(N) - this = allreduce time the step fails to hide under backward
        no_comm_ms = replay_ms(ablate={"polus_comm_allreduce_f32", "polus_comm_allreduce_bf16"})
        gemm_only_ms, no_gemm_ms, no_comm_ms = timer.max_over_ranks([gemm_only_ms, no_gemm_ms, no_comm_ms])
    if rank == 0:
        peaks, how = read_peaks()
        peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
        achieved = tot_flop / (gemm_only_ms * 1e-3) / 1e12 if gemm_only_ms > 0 else 0.0
        step_ms = ms_dev / args.steps
        marginal_ms = step_ms - no_gemm_ms
        cap = load_roofline_capture()
        scale = args.batch / float(cap["batch"]) if cap else None
        roof = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "frac_marginal": (tot_flop / (marginal_ms * 1e-3) / 1e12 / peak) if marginal_ms > 0 else None,
                "traffic": cap["traffic_bytes_per_launch"] * scale if cap else None,
                "traffic_source": (f"{cap['_path']} ({cap['n_launches']} launches, ncu --set full, batch {cap['batch']}; "
                                   f"scaled linearly to batch {args.batch})") if cap else None,
                "tensor_pipe_active_pct": cap["tensor_pipe_active_pct_time_weighted"] if cap else None,
                # sum over the step's GEMMs of (A + B + C bytes) / launches at batch 128: 244.2 MB with a bf16 gelu' tensor,
                # 227.8 MB since the derivative travels as one byte per element (12 x 2 x 100.7 MB less over 147 launches)
                "algorithmic_bytes_per_launch": 227.8e6 * args.batch / 128.0,
                "kernel": "gemm_tc_kernel (all tcgen05 GEMM launches of one step)", "launches": n_tc,
                "gemm_ms_per_step": gemm_only_ms, "gemm_gflop_per_step": tot_flop / 1e9,
                "method": "frac: CUDA-event time of a captured replay of the step's GEMM launches alone (same order/buffers/"
                          "streams); frac_marginal: step time minus the same step with the GEMM launches removed",
                "gemm_marginal_ms_per_step": marginal_ms,
                "peak_source": f"{how} bf16_tflops_sustained (kernel timed inside a long step)",
                "step_mfu": (args.batch * TRAIN_GFLOP_PER_SEQ * 1e9 / (step_ms * 1e-3)) / 1e12 / peak}
    # ---- the exchange step alone: bucketed NCCL allreduce of the gradient arena, back to back (in the step it is
    # overlapped with backward); bus bandwidth = bytes * 2(N-1)/N / time  (NCCL's definition)
    allreduce = None
    if world > 1:
        buckets = comm.plan_buckets(trainer.trainable_weights)
        nelem = sum(n for _, _, n, _ in buckets)
        st = device.stream()

        def ar_all():
            for ch, off, n, _ in buckets:
                comm.allreduce_bucket(ch, off, n, st)
        for _ in range(3):
            ar_all()
        e0, e1 = timer.ev(), timer.ev()
        barrier()
        _lib.call("polus_event_record", e0, st)
        for _ in range(10):
            ar_all()
        _lib.call("polus_event_record", e1, st)
        barrier()
        ms = C.c_float()
        _lib.call("polus_event_elapsed_ms", e0, e1, C.byref(ms))
        (ar_ms,) = timer.max_over_ranks([ms.value / 10])
        # leave the gradient arena zeroed, as the optimizer kernel does
        for ch, off, n, _ in buckets:
            _lib.call("polus_memset", ch.g.ptr + off * 4, 0, n * 4, st)
        device.device_sync()
        wire = comm.wire_bytes_per_element()
        nbytes = nelem * wire
        allreduce = {"bytes": int(nbytes), "wire_dtype": comm.WIRE_DTYPE, "buckets": len(buckets), "ms": ar_ms,
                     "busbw_GBps": nbytes * 2 * (world - 1) / world / (ar_ms * 1e-3) / 1e9,
                     "nvlink_peak_GBps": 900.0, "nvlink_measured_allreduce_GBps": 725.0,
                     "in_step_exposed_ms": (ms_dev / args.steps - no_comm_ms) if no_comm_ms is not None else None,
                     "step_ms_without_allreduce": no_comm_ms,
                     "limiting_collective": "ncclAllReduce of the last bucket (embedding-table gradients: backward produces "
                                            "them last, nothing is left to hide them under)",
                     "note": "standalone, back to back; inside the step it runs on a side stream under backward"}

    # ---- strong scaling: BASELINE.json configs[2] fixes the GLOBAL batch at 256 (256/128/64/32 per GPU at 1/2/4/8)
    strong = None
    if not args.no_strong and args.global_batch % world == 0:
        per = args.global_batch // world
        if per == args.batch:
            strong = {"seq_s": args.batch * world * args.steps / (ms_dev * 1e-3), "ms_per_step": ms_dev / args.steps}
        else:
            sb = to_device(synthetic_batches(4, per, SEQ, 30522, 4, seed=11 + rank))
            for i in range(4):
                float(trainer.train_step(*sb[i % len(sb)]))
            for i in range(30):
                last = trainer.train_step(*sb[i % len(sb)])
            float(last)
            ms_s, _, _ = timed(trainer, sb, args.steps)
            (ms_s,) = timer.max_over_ranks([ms_s])
            strong = {"seq_s": args.global_batch * args.steps / (ms_s * 1e-3), "ms_per_step": ms_s / args.steps}
            if world > 1:
                # the same step without its collective = what ONE GPU does on this per-GPU batch: the difference is the
                # exchange time the step fails to hide, the ratio the scaling efficiency against N independent GPUs
                (nc,) = timer.max_over_ranks([replay_ms(ablate={"polus_comm_allreduce_f32", "polus_comm_allreduce_bf16"}, feed=sb)])
                strong.update(step_ms_without_allreduce=nc, exposed_comm_ms=ms_s / args.steps - nc,
                              efficiency_vs_same_batch_without_comm=nc / (ms_s / args.steps),
                              limiting_collective="ncclAllReduce of the word-embedding gradient pieces (produced last by backward)")
        strong.update(global_batch=args.global_batch, batch_per_gpu=per, scaling="strong")
        try:
            with open(os.path.join(ROOT, "profiles", "r02_strong_baseline.json")) as f:
                base = json.load(f)
            # strong-scaling efficiency in the usual sense: speed-up over ONE GPU on the whole global batch, divided by N
            strong["efficiency_vs_n1_b256"] = strong["seq_s"] / base["n1_b256_seq_s"] / world
            strong["n1_b256_seq_s_source"] = base.get("source")
        except Exception:
            pass
        dbg(f"strong scaling done: {strong}")
    # ---- the same step at round 1's headline batch (128 / GPU), so the two rounds' lines can be compared like for like
    sweep = None
    if world == 1 and args.sweep_batch and args.sweep_batch != args.batch:
        sb = to_device(synthetic_batches(4, args.sweep_batch, SEQ, 30522, 4, seed=21 + rank))
        for i in range(4):
            float(trainer.train_step(*sb[i % len(sb)]))
        for i in range(40):
            last = trainer.train_step(*sb[i % len(sb)])
        float(last)
        ms_s, _, _ = timed(trainer, sb, args.steps)
        sweep = {str(args.sweep_batch): {"seq_s": args.sweep_batch * args.steps / (ms_s * 1e-3), "ms_per_step": ms_s / args.steps}}
    trainer.release_graphs()
    del trainer, dev_batches

    # ---- the two S=512 configurations BASELINE.json names (configs[3], configs[4]); data parallel like the headline
    extra = None
    if not args.no_extra_configs:
        extra = {}
        for name, b in (("cfg4", args.cfg4_batch), ("cfg5", args.cfg5_batch)):
            r = quick_config(name, b, args.steps, timer, world)
            extra[name + "_seq_s"] = r["seq_s"]
            extra[name] = r
            dbg(f"{name} done: {r['seq_s']:.1f} seq/s")
    if rank != 0:
        return
    seqs = args.batch * world * args.steps
    value = seqs / (ms_dev * 1e-3)
    e2e_value = seqs / (ms_e2e * 1e-3)
    line = {"metric": "train_sequences_per_second", "value": value, "unit": "sequences/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(args.batch),
                       "global_batch": args.batch * world, "seq_len": SEQ, "parallelism": f"dp{world}",
                       "preheat_steps": args.preheat_steps,
                       "l2": "per-step working set (weights 0.2 GB bf16 + activations > 3 GB) exceeds the 126 MB L2; no flush needed",
                       "loss_last": loss_dev},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "sequences/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "roofline": roof}
    if allreduce is not None:
        line["allreduce"] = allreduce
    if dp_parity is not None:
        line["dp_parity"] = dp_parity
    if strong is not None:
        line["strong_gb256"] = strong
    if sweep is not None:
        line["batch_sweep"] = sweep
    if extra is not None:
        line["configs"] = extra
    if world == 1 and not args.no_cpu_baseline:
        from oracle import torch_ref
        sps, dt, threads = torch_ref.time_train_steps(batch=args.ref_batch, seq=SEQ, steps=2, warmup=1)
        line["cpu_baseline"] = {"value": sps, "unit": "sequences/s", "cores": threads, "kind": "port",
                                "sample": f"2 timed steps of {args.ref_batch} sequences x {SEQ} tokens (torch-CPU port, fp32)"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="sequences per GPU per step (weak scaling: global batch = batch x N); "
                    "BASELINE.json names the model and sequence length, not the batch: 256 is the best of the 32..256 sweep (DESIGN.md)")
    ap.add_argument("--sweep-batch", type=int, default=128, help="a second per-GPU batch timed briefly at N = 1 (round 1's headline batch)")
    ap.add_argument("--ref-batch", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--preheat-steps", type=int, default=100, help="untimed steps before the timed regions (~2.4 s at batch 128)")
    ap.add_argument("--global-batch", type=int, default=256, help="strong-scaling arm: global batch split over the N GPUs (BASELINE cfg3)")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-dp-parity", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the cfg4 / cfg5 (S=512) throughput lines")
    ap.add_argument("--cfg4-batch", type=int, default=64)
    ap.add_argument("--cfg5-batch", type=int, default=32)
    ap.add_argument("--dump-outputs", metavar="DIR", help="start each timed region from the initial weights and write "
                    "the loss of each region's last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what --impl ours computed")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
