"""Differentiable device ops + the gradient tape.

Plays the role tf.GradientTape / TF's kernel library play for the reference (polus/training.py:173-185):
the trainer records the forward computation on a tape and asks for d(loss)/d(trainable_weights).  Every
op below is one or a few launches of libpolus_b200.so kernels; nothing computes on the host.
Parameter gradients are accumulated straight into the fp32 gradient arena (`Param.grad`), so shared
variables and split-K GEMMs need no extra reduction pass.
"""
import ctypes as C
import math

import numpy as np

from . import _lib, device
from .tensor import BF16, F32, I32, U8, Param, Tensor

# ------------------------------------------------------------------------------------------------
# tape
# ------------------------------------------------------------------------------------------------
_tape_stack = []
_rng_state = {"seed": 0x5EED5EED, "site": 0, "step_ptr": None, "step_buf": None}


def set_seed(seed):
    """Seed of the device dropout streams (reference: polus/utils.py:6-9 set_random_seed)."""
    _rng_state["seed"] = int(seed) & 0xFFFFFFFFFFFFFFFF
    _rng_state["site"] = 0


def reset_dropout_sites():
    _rng_state["site"] = 0


def _next_site():
    _rng_state["site"] += 1
    return _rng_state["site"]


def step_counter():
    """Device uint32 holding optimizer.iterations; dropout counters and the LR schedule read it."""
    if _rng_state["step_ptr"] is None:
        buf = device.Buffer(16, zero=True)
        device.synchronize()
        _rng_state["step_buf"] = buf
        _rng_state["step_ptr"] = buf.ptr
    return _rng_state["step_ptr"]


def set_step(value):
    device.upload(step_counter(), np.array([value, 0, 0, 0], np.uint32))


class Node:
    __slots__ = ("inputs", "output", "backward")

    def __init__(self, inputs, output, backward):
        self.inputs = inputs
        self.output = output
        self.backward = backward


class GradientTape:
    """Same usage as tf.GradientTape in polus/training.py:173-185 (incl. stop_recording)."""

    def __init__(self):
        self.nodes = []
        self.paused = 0

    def __enter__(self):
        _tape_stack.append(self)
        return self

    def __exit__(self, *exc):
        _tape_stack.pop()
        return False

    class _Pause:
        def __init__(self, tape):
            self.tape = tape

        def __enter__(self):
            self.tape.paused += 1

        def __exit__(self, *exc):
            self.tape.paused -= 1
            return False

    def stop_recording(self):
        return GradientTape._Pause(self)

    def gradient(self, loss, weights, on_bucket_ready=None):
        """Back-propagate from a scalar loss.  Returns the gradient tensors of `weights` (views of the
        gradient arena for Params).  on_bucket_ready(chunk, offset, n_elems): called during the sweep as soon as every
        gradient of a contiguous ~64 MB span of the arena is final (the optimizer updates that span on a side stream
        while backward continues, training.BaseTrainer._step_body)."""
        before = None
        if on_bucket_ready is not None:
            before, flush = bucket_schedule(self.nodes, weights, lambda b: on_bucket_ready(b[0], b[1], b[2]))
        grads = run_backward(self.nodes, loss, before)
        if on_bucket_ready is not None:
            flush()
        self.nodes = []
        return [w.grad if isinstance(w, Param) else _materialise(grads.get(id(w))) for w in weights]


def bucket_schedule(nodes, weights, launch):
    """(before_node, flush) for run_backward: `launch(bucket)` fires once backward has passed the EARLIEST forward node
    that reads any parameter of the bucket, i.e. when all its gradients are final and its weights are no longer read."""
    from . import comm
    buckets = comm.plan_buckets(weights)
    first_use = {}
    for idx, node in enumerate(nodes):
        for t in node.inputs:
            if isinstance(t, Param) and id(t) not in first_use:
                first_use[id(t)] = idx
    ready_at = []
    for b in buckets:
        uses = [first_use[id(p)] for p in b[3] if id(p) in first_use]
        ready_at.append(min(uses) if uses else len(nodes))
    pending = sorted(range(len(buckets)), key=lambda i: -ready_at[i])

    def before_node(idx):
        while pending and ready_at[pending[0]] > idx:
            launch(buckets[pending.pop(0)])

    def flush():
        while pending:
            launch(buckets[pending.pop(0)])
    return before_node, flush


def _materialise(g):
    """A gradient slot holds one tensor or a list of not-yet-summed contributions."""
    if isinstance(g, list):
        acc = g[0]
        for t in g[1:]:
            acc = _accumulate(acc, t)
        return acc
    return g


def run_backward(nodes, loss, before_node=None):
    """Reverse sweep over the recorded nodes.  `before_node(idx)` lets the data-parallel tape launch bucket
    allreduces as soon as backward has passed the variables of a bucket.  Contributions to the same tensor
    are kept as a list and summed lazily: a node whose backward carries `pair_ok` (LayerNorm backward)
    consumes two contributions directly, fusing the residual-stream addition into its own pass."""
    root = ones_like(loss)
    root.is_one = True
    grads = {id(loss): root}
    for idx in range(len(nodes) - 1, -1, -1):
        if before_node is not None:
            before_node(idx)
        node = nodes[idx]
        g = grads.pop(id(node.output), None)
        if g is None:
            continue
        if isinstance(g, list) and not (len(g) == 2 and getattr(node.backward, "pair_ok", False)):
            g = _materialise(g)
        in_grads = node.backward(g)
        for t, gi in zip(node.inputs, in_grads):
            if gi is None or t is None or isinstance(t, Param) or not t.requires_grad:
                continue
            prev = grads.get(id(t))
            if prev is None:
                grads[id(t)] = gi
            elif isinstance(prev, list):
                prev.append(gi)
            else:
                grads[id(t)] = [prev, gi]
    side_join()  # weight gradients issued on the background stream are complete from here on
    return grads


_no_grad_depth = [0]


class no_grad:
    """Forward computations whose intermediates must not be kept (frozen encoders: polus/data.py:523-545,
    polus/ir/training.py:47-67 under tape.stop_recording)."""

    def __enter__(self):
        _no_grad_depth[0] += 1

    def __exit__(self, *exc):
        _no_grad_depth[0] -= 1
        return False


def _recording(*inputs):
    if not _tape_stack or _no_grad_depth[0]:
        return None
    tape = _tape_stack[-1]
    if tape.paused:
        return None
    if any(t is not None and t.requires_grad for t in inputs):
        return tape
    return None


def _record(tape, inputs, output, backward):
    output.requires_grad = True
    for t in inputs:
        if t is not None and not isinstance(t, Param):
            t.consumers += 1
    tape.nodes.append(Node(list(inputs), output, backward))
    return output


def _accumulate(a, b):
    if a.dtype == BF16 and b.dtype == BF16:
        out = Tensor(a.shape, BF16)
        _lib.call("polus_add_bf16", a.ptr, b.ptr, out.ptr, a.size, device.stream())
        return out
    a32, b32 = cast(a, F32), cast(b, F32)
    out = Tensor(a.shape, F32)
    _lib.call("polus_binary_f32", 0, a32.ptr, b32.ptr, a.size, b.size, out.ptr, device.stream())
    return out


# ------------------------------------------------------------------------------------------------
# background stream for weight-gradient GEMMs
# ------------------------------------------------------------------------------------------------
# Nothing in backward consumes dW before the optimizer (or the bucket allreduce), while the dgrad chain is strictly
# serial and most of its GEMMs end in a partly filled wave (96 pair-tiles on 74 SM pairs for the 768-wide ones).
# While a step is being captured, wgrad GEMMs are issued on a low-priority side stream, so in the replayed graph
# they run in those tails and next to the memory-bound LayerNorm / activation-gradient kernels.  Only during
# capture: there activation blocks are never recycled (tensor._Pool.trace), so the side stream cannot observe a
# buffer being reused by the main chain.
_side = {"stream": None, "events": [], "next": 0, "dirty": False}


def _side_event():
    i = _side["next"]
    if i == len(_side["events"]):
        ev = C.c_void_p()
        _lib.call("polus_event_create", C.byref(ev))
        _side["events"].append(ev)
    _side["next"] = i + 1
    return _side["events"][i]


def side_active():
    from . import tensor as _t
    return _t._pool.trace is not None


def side_reset():
    """Called when a capture begins: events of an earlier capture may be reused."""
    _side["next"] = 0
    _side["dirty"] = False
    _side["opt_dirty"] = False


def side_fork():
    """Side stream observes everything issued on the main stream so far; returns the side stream."""
    if _side["stream"] is None:
        s = C.c_void_p()
        _lib.call("polus_stream_create", C.byref(s), 2)
        _side["stream"] = s.value
    ev = _side_event()
    _lib.call("polus_event_record", ev, device.stream())
    _lib.call("polus_stream_wait_event", _side["stream"], ev)
    _side["dirty"] = True
    return _side["stream"]


def opt_stream_after(*streams):
    """Stream for early optimizer updates (training._step_body): it first observes everything issued so far on
    `streams`.  Separate from the wgrad side stream so that an update waiting for its allreduce never blocks wgrads."""
    if _side.get("opt") is None:
        s = C.c_void_p()
        _lib.call("polus_stream_create", C.byref(s), 2)
        _side["opt"] = s.value
    for st in streams:
        if st is None:
            continue
        ev = _side_event()
        _lib.call("polus_event_record", ev, st)
        _lib.call("polus_stream_wait_event", _side["opt"], ev)
    _side["opt_dirty"] = True
    return _side["opt"]


def opt_stream_join():
    """Main stream waits for every early optimizer update."""
    if _side.get("opt_dirty"):
        ev = _side_event()
        _lib.call("polus_event_record", ev, _side["opt"])
        _lib.call("polus_stream_wait_event", device.stream(), ev)
        _side["opt_dirty"] = False


def side_stream_if_dirty():
    return _side["stream"] if _side["dirty"] else None


def side_join(stream=None):
    """`stream` (default: main) waits for every wgrad issued on the side stream so far."""
    if not _side["dirty"]:
        return
    ev = _side_event()
    _lib.call("polus_event_record", ev, _side["stream"])
    _lib.call("polus_stream_wait_event", stream if stream is not None else device.stream(), ev)
    if stream is None:
        _side["dirty"] = False


# ------------------------------------------------------------------------------------------------
# basic helpers (not differentiable unless stated)
# ------------------------------------------------------------------------------------------------
def ones_like(t):
    out = Tensor(t.shape, F32)
    _lib.call("polus_fill_f32", out.ptr, 1.0, out.size, device.stream())
    return out if t.dtype == F32 else cast(out, t.dtype)


def zeros(shape, dtype=F32):
    return Tensor(shape, dtype, zero=True)


def cast(x, dtype):
    """Differentiable dtype conversion."""
    if x.dtype == dtype:
        return x
    out = Tensor(x.shape, dtype)
    _lib.call("polus_cast", x.ptr, x.dtype, out.ptr, dtype, x.size, device.stream())
    tape = _recording(x)
    if tape is not None and dtype in (F32, BF16) and x.dtype in (F32, BF16):
        src = x.dtype
        _record(tape, [x], out, lambda g: [cast(g, src)])
    return out


def reshape(x, shape):
    out = x.view(shape)
    tape = _recording(x)
    if tape is not None:
        old = x.shape
        _record(tape, [x], out, lambda g: [g.view(old)])
    return out


def argmax(x, axis=-1):
    """tf.argmax(..., output_type=int32), ties -> lowest index (polus/models.py:148-150)."""
    assert axis in (-1, x.ndim - 1)
    x = cast(x, F32)
    cols = x.shape[-1]
    rows = x.size // cols
    out = Tensor(x.shape[:-1], I32)
    _lib.call("polus_argmax_f32", x.ptr, rows, cols, out.ptr, device.stream())
    return out


def one_hot(idx, depth):
    rows = idx.size
    out = Tensor(tuple(idx.shape) + (depth,), F32)
    _lib.call("polus_one_hot_f32", idx.ptr, rows, depth, out.ptr, device.stream())
    return out


# ------------------------------------------------------------------------------------------------
# GEMM plumbing
# ------------------------------------------------------------------------------------------------
GEMM_PROFILE = None  # list collecting (kind, flops, start_event, stop_event) when bench.py profiles a step


def _operand(t_ptr, ld, mn_major, dtype, bs0=0, bs1=0):
    return _lib.Operand(t_ptr, ld, bs0, bs1, 1 if mn_major else 0, dtype)


def _gemm(M, N, K, A, B, c_ptr, ldc, c_dtype, bias=None, act=0, c2=None, alpha=1.0, accumulate=0, split_k=1,
          batch0=1, batch1=1, cbs0=0, cbs1=0, force_small=False, stream=None, c2_kind=0, emul=None, colsum=None):
    if stream is None:
        stream = device.stream()
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = M, N, K, batch0, batch1
    g.A, g.B = A, B
    g.C, g.ldc, g.cbs0, g.cbs1, g.c_dtype = c_ptr, ldc, cbs0, cbs1, c_dtype
    g.C2, g.bias = c2, bias
    g.alpha, g.act, g.accumulate, g.split_k = alpha, act, accumulate, split_k
    g.c2_kind, g.Emul, g.colsum = c2_kind, emul, colsum
    use_tc = (not force_small and A.dtype == BF16 and B.dtype == BF16
              and _lib.call("polus_gemm_tc_supported", C.byref(g)) == 1)
    prof = GEMM_PROFILE
    if prof is not None:  # bench.py: bracket every launch with CUDA events on the launching stream
        e0, e1 = C.c_void_p(), C.c_void_p()
        _lib.call("polus_event_create", C.byref(e0))
        _lib.call("polus_event_create", C.byref(e1))
        _lib.call("polus_event_record", e0, stream)
    if use_tc:
        _lib.call("polus_gemm_tc", C.byref(g), stream)
    else:
        g.split_k = 1
        _lib.call("polus_gemm_small", C.byref(g), stream)
    if prof is not None:
        _lib.call("polus_event_record", e1, stream)
        prof.append(("tc" if use_tc else "small", 2.0 * M * N * K * batch0 * batch1, e0, e1))
    return "tc" if use_tc else "small"


def _gemm_tc_supported(M, N, K, A, B, c_ptr, ldc, c_dtype, **kw):
    """Would polus_gemm_tc take this problem?  (Same fields as _gemm; used to choose the 8-bit derivative format.)"""
    g = _lib.Gemm()
    g.M, g.N, g.K, g.batch0, g.batch1 = M, N, K, 1, 1
    g.A, g.B = A, B
    g.C, g.ldc, g.cbs0, g.cbs1, g.c_dtype = c_ptr, ldc, 0, 0, c_dtype
    g.C2, g.bias = kw.get("c2"), kw.get("bias")
    g.alpha, g.act, g.accumulate, g.split_k = 1.0, kw.get("act", 0), 0, 1
    g.c2_kind, g.Emul, g.colsum = kw.get("c2_kind", 0), kw.get("emul"), kw.get("colsum")
    return _lib.call("polus_gemm_tc_supported", C.byref(g)) == 1


def _act_code(act):
    if callable(act):
        act = getattr(act, "__name__", None)
    if act not in _lib.ACT:
        raise ValueError(f"unsupported activation {act!r}")
    return _lib.ACT[act]


def linear(x, W, b=None, activation=None, out_dtype=None, defer_bias_grad=False):
    """y = act(x @ W + b) with W in Keras layout [in, out] (tf.keras.layers.Dense).

    bf16 operands with in/out multiples of 8 run on the tcgen05 GEMM; anything else (the K-tag
    projection, the 10-way tutorial head) on the CUDA-core GEMM with fp32 weights."""
    act = _act_code(activation)
    K, N = W.shape
    lead = x.shape[:-1]
    M = x.size // K
    assert x.shape[-1] == K, f"Dense expected last dim {K}, got {x.shape}"
    use_tc = (K % 8 == 0 and N % 8 == 0 and M > 0)
    tape = _recording(x, W, b)
    if use_tc:
        xb = cast(x, BF16)
        y = Tensor(lead + (N,), BF16)
        # with an activation the GEMM epilogue also stores act'(z) (not z): backward is then one multiply, which the
        # dgrad GEMM of the layer that consumes y applies in its own epilogue together with the bias-gradient column
        # sums -- no pass over the [M,N] tensor for GeluGrad / BiasAddGrad.  GELU's derivative goes as 8-bit
        # fixed point (c2_kind = 2) wherever the GEMM takes it: the FFN-up GEMM and the dgrad GEMM that reads it back are
        # bound by SM store bandwidth / multiplier-tile traffic, and a byte per element carries the same aggregate
        # gradient error as bf16 (DESIGN.md section 8)
        d, dkind = None, 1
        if act != 0 and tape is not None:
            opA, opB = _operand(xb.ptr, K, False, BF16), _operand(W.shadow.ptr, N, True, BF16)
            if (act == _lib.ACT["gelu"]
                    and _gemm_tc_supported(M, N, K, opA, opB, y.ptr, N, BF16, bias=b.ptr if b is not None else None, act=act,
                                           c2=y.ptr, c2_kind=2)):
                d, dkind = Tensor(lead + (N,), U8), 2
            else:
                d = Tensor(lead + (N,), BF16)
        _gemm(M, N, K, _operand(xb.ptr, K, False, BF16), _operand(W.shadow.ptr, N, True, BF16),
              y.ptr, N, BF16, bias=b.ptr if b is not None else None, act=act, c2=d.ptr if d is not None else None, c2_kind=dkind)
        if tape is not None:
            if d is not None:
                y.bwd_fuse = (d, b.grad if b is not None else None, dkind)

            def backward(g, xb=xb, d=d):
                g = cast(g, BF16)
                need_dz = act != 0
                if need_dz and g.fused_for == id(y):
                    dz, need_dz, want_bias = g, False, False  # the producer of g already applied act' and summed the bias grad
                else:
                    dz = Tensor(g.shape, BF16) if need_dz else g
                    # defer_bias_grad: the consumer (layernorm_residual with x_bias=b) already added colsum(g) to b.grad
                    want_bias = b is not None and not (defer_bias_grad and act == 0)
                if need_dz or want_bias:
                    _lib.call("polus_act_bwd_colsum", g.ptr, d.ptr if d is not None else None, M, N,
                              (_lib.ACT_DERIV_U8 if dkind == 2 else _lib.ACT_DERIV) if need_dz else 0,
                              dz.ptr if need_dz else None, b.grad.ptr if want_bias else None, None, device.stream())
                # dW[K,N] += x^T dz : A = x (MN-major over K), B = dz (MN-major over N), reduce over M
                _gemm(K, N, M, _operand(xb.ptr, K, True, BF16), _operand(dz.ptr, N, True, BF16),
                      W.grad.ptr, N, F32, accumulate=1, split_k=0, stream=side_fork() if side_active() else None)
                dx = None
                if xb.requires_grad:
                    dx = Tensor(lead + (K,), BF16)
                    fuse = xb.bwd_fuse if (xb.bwd_fuse is not None and xb.consumers == 1) else None
                    opA, opB = _operand(dz.ptr, N, False, BF16), _operand(W.shadow.ptr, N, False, BF16)
                    if fuse is not None and fuse[2] == 2 and not _gemm_tc_supported(M, K, N, opA, opB, dx.ptr, K, BF16, emul=fuse[0].ptr,
                                                                                  colsum=fuse[1].ptr if fuse[1] is not None else None, c2_kind=2):
                        fuse = None   # this GEMM cannot read the 8-bit derivative: the producer's own backward applies it
                    # dx[M,K] = dz[M,N] . W[K,N]^T : both K-major over N  (* act'(z_prev), + bias-grad column sums when fused)
                    kind = _gemm(M, K, N, opA, opB,
                                 dx.ptr, K, BF16, emul=fuse[0].ptr if fuse else None,
                                 colsum=fuse[1].ptr if (fuse and fuse[1] is not None) else None, c2_kind=fuse[2] if fuse else 0)
                    if fuse and kind == "tc":
                        dx.fused_for = id(xb)
                    elif fuse:
                        raise RuntimeError("fused activation backward needs the tcgen05 GEMM path")
                return [dx, None, None]
            _record(tape, [xb, W, b], y, backward)
        return y
    # CUDA-core path (fp32 weights)
    y = Tensor(lead + (N,), out_dtype if out_dtype is not None else F32)
    assert y.dtype == F32
    z = Tensor(lead + (N,), F32) if (act != 0 and tape is not None) else None
    skinny = x.dtype in (F32, BF16) and _lib.call("polus_skinny_supported", K, N) == 1
    if skinny:  # narrow outputs (K-tag projection, 10-way head): one pass over x
        _lib.call("polus_skinny_fwd", x.ptr, x.dtype, W.ptr, b.ptr if b is not None else None, M, K, N, act, y.ptr,
                  z.ptr if z is not None else None, device.stream())
    else:
        _gemm(M, N, K, _operand(x.ptr, K, False, x.dtype), _operand(W.ptr, N, True, F32), y.ptr, N, F32,
              bias=b.ptr if b is not None else None, act=act, c2=z.ptr if z is not None else None, force_small=True)
    if tape is not None:
        def backward(g, z=z):
            g = cast(g, F32)
            if act != 0:
                dz = Tensor(g.shape, F32)
                _lib.call("polus_unary_f32", act, z.ptr, g.ptr, 1, g.size, dz.ptr, 1.0, device.stream())
            else:
                dz = g
            dx = None
            if x.requires_grad:
                dx = Tensor(lead + (K,), x.dtype if x.dtype in (F32, BF16) else F32)
            if skinny:
                _lib.call("polus_skinny_bwd", x.ptr, x.dtype, W.ptr, dz.ptr, M, K, N, dx.ptr if dx is not None else None,
                          dx.dtype if dx is not None else F32, W.grad.ptr, b.grad.ptr if b is not None else None,
                          device.stream())
                return [dx, None, None]
            if b is not None:
                _lib.call("polus_reduce_sum_f32", dz.ptr, M, N, 0, 1.0, b.grad.ptr, 1, device.stream())
            _gemm(K, N, M, _operand(x.ptr, K, True, x.dtype), _operand(dz.ptr, N, True, F32), W.grad.ptr, N, F32,
                  accumulate=1, force_small=True)
            if dx is not None:
                _gemm(M, K, N, _operand(dz.ptr, N, False, F32), _operand(W.ptr, N, False, F32), dx.ptr, K, dx.dtype,
                      force_small=True)
            return [dx, None, None]
        _record(tape, [x, W, b], y, backward)
    return y


def matmul(a, b, transpose_b=False):
    """fp32 2-D matmul for head/score code written against tf.matmul (polus/ir/training.py compute_scores)."""
    a, b = cast(a, F32), cast(b, F32)
    M, K = a.shape
    N = b.shape[0] if transpose_b else b.shape[1]
    y = Tensor((M, N), F32)
    Bop = _operand(b.ptr, b.shape[1], not transpose_b, F32)
    _gemm(M, N, K, _operand(a.ptr, K, False, F32), Bop, y.ptr, N, F32, force_small=True)
    tape = _recording(a, b)
    if tape is not None:
        def backward(g):
            g = cast(g, F32)
            da = db = None
            if a.requires_grad:
                da = Tensor(a.shape, F32)
                # da[M,K] = g[M,N] . Bm[N,K] where Bm = b^T (transpose_b) or b
                _gemm(M, K, N, _operand(g.ptr, N, False, F32),
                      _operand(b.ptr, b.shape[1], transpose_b, F32), da.ptr, K, F32, force_small=True)
            if b.requires_grad:
                db = Tensor(b.shape, F32)
                if transpose_b:  # b [N,K]: db = g^T a
                    _gemm(N, K, M, _operand(g.ptr, N, True, F32), _operand(a.ptr, K, True, F32), db.ptr, K, F32, force_small=True)
                else:  # b [K,N]: db = a^T g
                    _gemm(K, N, M, _operand(a.ptr, K, True, F32), _operand(g.ptr, N, True, F32), db.ptr, N, F32, force_small=True)
            return [da, db]
        _record(tape, [a, b], y, backward)
    return y


# ------------------------------------------------------------------------------------------------
# encoder ops
# ------------------------------------------------------------------------------------------------
def embed_layernorm(ids, token_type_ids, word, pos, type_, gamma, beta, eps=1e-12, p_drop=0.0):
    """HF TFBertEmbeddings (polus/data.py:526-545): LN(word[ids]+pos+type[tt]) -> dropout.  -> bf16 [B,S,H]."""
    Bsz, S = ids.shape
    V, H = word.shape
    n_types = type_.shape[0]
    assert S <= pos.shape[0], f"sequence length {S} exceeds the {pos.shape[0]} learned positions"
    M = Bsz * S
    y = Tensor((Bsz, S, H), BF16)
    z = Tensor((M, H), F32)
    mean, rstd = Tensor((M,), F32), Tensor((M,), F32)
    site = _next_site() if p_drop > 0 else 0
    seed = _rng_state["seed"]
    _lib.call("polus_embed_ln_fwd", ids.ptr, token_type_ids.ptr if token_type_ids is not None else None, word.ptr,
              pos.ptr, type_.ptr, gamma.ptr, beta.ptr, Bsz, S, H, V, n_types, eps, p_drop, seed, site, step_counter(),
              y.ptr, z.ptr, mean.ptr, rstd.ptr, device.stream())
    tape = _recording(word, pos, type_, gamma, beta)
    if tape is not None:
        def backward(g):
            g = cast(g, BF16)
            ws = Tensor((int(_lib.call("polus_embed_ws_floats", Bsz, S, H)),), F32)
            _lib.call("polus_embed_ln_bwd", g.ptr, z.ptr, mean.ptr, rstd.ptr, gamma.ptr, ids.ptr,
                      token_type_ids.ptr if token_type_ids is not None else None, Bsz, S, H, V, n_types, p_drop, seed,
                      site, step_counter(), word.grad.ptr, pos.grad.ptr, type_.grad.ptr, gamma.grad.ptr, beta.grad.ptr,
                      ws.ptr, device.stream())
            return [None] * 5
        _record(tape, [word, pos, type_, gamma, beta], y, backward)
    return y


def layernorm_residual(x, res, gamma, beta, eps=1e-12, p_drop=0.0, x_bias=None):
    """y = LN(dropout(x) + res)  (HF TFBertSelfOutput / TFBertOutput).  x is consumed (overwritten by z).
    x_bias: bias Param of the Dense layer that produced x (called with defer_bias_grad=True): its gradient,
    colsum(d x), is accumulated by this op's backward kernel instead of a separate pass."""
    H = x.shape[-1]
    M = x.size // H
    x = cast(x, BF16)
    if res is not None:
        res = cast(res, BF16)
    y = Tensor(x.shape, BF16)
    mean, rstd = Tensor((M,), F32), Tensor((M,), F32)
    site = _next_site() if p_drop > 0 else 0
    seed = _rng_state["seed"]
    tape = _recording(x, res, gamma, beta)
    # dropout decisions, one byte per 8 elements, handed to backward (saves it the Philox regeneration)
    keep = Tensor((M * (H // 8),), U8) if (p_drop > 0 and tape is not None) else None
    _lib.call("polus_ln_res_fwd", x.ptr, res.ptr if res is not None else None, gamma.ptr, beta.ptr, M, H, eps, p_drop,
              seed, site, step_counter(), y.ptr, mean.ptr, rstd.ptr, keep.ptr if keep is not None else None, device.stream())
    if tape is not None:
        z = x  # now holds dropout(x) + res

        def backward(g):
            g2 = None
            if isinstance(g, list):  # two contributions to d(y): summed inside the kernel
                g, g2 = cast(g[0], BF16), cast(g[1], BF16)
            else:
                g = cast(g, BF16)
            dx = Tensor(x.shape, BF16)
            if res is None:
                dres = None
            elif p_drop > 0:
                dres = Tensor(x.shape, BF16)
            else:
                dres = dx  # identical values: write once
            _lib.call("polus_ln_res_bwd", g.ptr, g2.ptr if g2 is not None else None, z.ptr, mean.ptr, rstd.ptr, gamma.ptr,
                      M, H, p_drop, seed, site, step_counter(), dx.ptr, dres.ptr if dres is not None else None,
                      gamma.grad.ptr, beta.grad.ptr, x_bias.grad.ptr if x_bias is not None else None,
                      keep.ptr if keep is not None else None, device.stream())
            return [dx, dres, None, None]
        backward.pair_ok = True
        _record(tape, [x, res, gamma, beta], y, backward)
    return y


def attention(qkv, mask, n_heads, p_drop=0.0, qkv_bias=None):
    """Multi-head self-attention core on the packed projection qkv [B,S,3H] (q|k|v column blocks):
    softmax(QK^T/sqrt(dh) + (1-mask)*-10000) V  ->  ctx [B,S,H]   (HF TFBertSelfAttention; mask constant
    from polus/models.py:175-195).  The fused kernels wherever polus_attention_supported(S, dh) accepts the shape,
    the GEMM + softmax path otherwise."""
    Bsz, S, H3 = qkv.shape
    H = H3 // 3
    dh = H // n_heads
    assert dh % 8 == 0 and S % 8 == 0, "attention needs head_dim and sequence length multiples of 8"
    qkv = cast(qkv, BF16)
    if _lib.call("polus_attention_supported", S, dh) == 1:
        return _attention_fused(qkv, mask, n_heads, p_drop, qkv_bias)
    return _attention_unfused(qkv, mask, n_heads, p_drop)


def attention_takes_bias_grad(S, head_dim):
    """True when ops.attention(..., qkv_bias=b) will accumulate b's gradient itself (fused kernels): the caller then
    builds the QKV projection with defer_bias_grad=True."""
    return bool(head_dim % 8 == 0 and S % 8 == 0 and _lib.call("polus_attention_supported", S, head_dim) == 1)


def _attention_unfused(qkv, mask, n_heads, p_drop):
    """Any S and head_dim (multiples of 8), qkv in bf16.  Three batched tcgen05 GEMM launches + one softmax launch; the
    head split/merge transposes of the reference are folded into the TMA tensor maps."""
    Bsz, S, H3 = qkv.shape
    H = H3 // 3
    dh = H // n_heads
    nb = Bsz * n_heads
    scale = 1.0 / math.sqrt(dh)
    q_ptr, k_ptr, v_ptr = qkv.ptr, qkv.ptr + H * 2, qkv.ptr + 2 * H * 2
    ld, bs0, bs1 = H3, dh, S * H3  # batch0 = head, batch1 = batch
    scores = Tensor((nb, S, S), BF16)
    _gemm(S, S, dh, _operand(q_ptr, ld, False, BF16, bs0, bs1), _operand(k_ptr, ld, False, BF16, bs0, bs1),
          scores.ptr, S, BF16, batch0=n_heads, batch1=Bsz, cbs0=S * S, cbs1=S * S * n_heads)
    tape = _recording(qkv)
    P = scores  # softmax in place
    Pd = Tensor((nb, S, S), BF16) if p_drop > 0 else P
    site = _next_site() if p_drop > 0 else 0
    seed = _rng_state["seed"]
    _lib.call("polus_softmax_fwd", scores.ptr, mask.ptr if mask is not None else None, Bsz, n_heads, S, S, scale,
              p_drop, seed, site, step_counter(), P.ptr, Pd.ptr, device.stream())
    ctx = Tensor((Bsz, S, H), BF16)
    _gemm(S, dh, S, _operand(Pd.ptr, S, False, BF16, S * S, S * S * n_heads), _operand(v_ptr, ld, True, BF16, bs0, bs1),
          ctx.ptr, H, BF16, batch0=n_heads, batch1=Bsz, cbs0=dh, cbs1=S * H)
    if tape is not None:
        def backward(g):
            g = cast(g, BF16)  # dctx [B,S,H]
            dqkv = Tensor((Bsz, S, H3), BF16)
            dq_ptr, dk_ptr, dv_ptr = dqkv.ptr, dqkv.ptr + H * 2, dqkv.ptr + 2 * H * 2
            gO = lambda ptr: _operand(ptr, H, False, BF16, dh, S * H)   # dctx as [S, dh] K-major per head
            # dPd[S,S'] = dctx[S,dh] . V[S',dh]^T
            dP = Tensor((nb, S, S), BF16)
            _gemm(S, S, dh, gO(g.ptr), _operand(v_ptr, ld, False, BF16, bs0, bs1), dP.ptr, S, BF16,
                  batch0=n_heads, batch1=Bsz, cbs0=S * S, cbs1=S * S * n_heads)
            # dS in place of dP; Pd (dropped probabilities) in place of P
            _lib.call("polus_softmax_bwd", P.ptr, dP.ptr, Bsz, n_heads, S, S, scale, p_drop, seed, site,
                      step_counter(), device.stream())
            Pd_b = P
            pop = lambda ptr, mn: _operand(ptr, S, mn, BF16, S * S, S * S * n_heads)
            # dV[S',dh] = Pd^T[S',S] . dctx[S,dh]
            _gemm(S, dh, S, pop(Pd_b.ptr, True), _operand(g.ptr, H, True, BF16, dh, S * H), dv_ptr, H3, BF16,
                  batch0=n_heads, batch1=Bsz, cbs0=dh, cbs1=S * H3)
            # dQ[S,dh] = dS[S,S'] . K[S',dh]
            _gemm(S, dh, S, pop(dP.ptr, False), _operand(k_ptr, ld, True, BF16, bs0, bs1), dq_ptr, H3, BF16,
                  batch0=n_heads, batch1=Bsz, cbs0=dh, cbs1=S * H3)
            # dK[S',dh] = dS^T[S',S] . Q[S,dh]
            _gemm(S, dh, S, pop(dP.ptr, True), _operand(q_ptr, ld, True, BF16, bs0, bs1), dk_ptr, H3, BF16,
                  batch0=n_heads, batch1=Bsz, cbs0=dh, cbs1=S * H3)
            return [dqkv]
        _record(tape, [qkv], ctx, backward)
    return ctx


def _attention_fused(qkv, mask, n_heads, p_drop, qkv_bias=None):
    """One kernel per direction: scores and probabilities stay in TMEM / shared memory (csrc/attention.cu)."""
    Bsz, S, H3 = qkv.shape
    H = H3 // 3
    dh = H // n_heads
    ctx = Tensor((Bsz, S, H), BF16)
    lse = Tensor((Bsz, n_heads, S), F32)
    site = _next_site() if p_drop > 0 else 0
    seed = _rng_state["seed"]
    mptr = mask.ptr if mask is not None else None
    keep = Tensor((int(_lib.call("polus_attention_keepbits_words", Bsz, S, n_heads)),), I32) if p_drop > 0 else None
    kptr = keep.ptr if keep is not None else None
    _lib.call("polus_attention_fwd", qkv.ptr, mptr, Bsz, S, n_heads, dh, p_drop, seed, site, step_counter(), ctx.ptr,
              lse.ptr, kptr, device.stream())
    tape = _recording(qkv)
    if tape is not None:
        def backward(g, _alive=(keep, mask)):  # the closure uses raw pointers: keep their owners out of the pool
            g = cast(g, BF16)
            dqkv = Tensor((Bsz, S, H3), BF16)
            _lib.call("polus_attention_bwd", qkv.ptr, mptr, ctx.ptr, g.ptr, lse.ptr, Bsz, S, n_heads, dh, p_drop, seed, site,
                      step_counter(), kptr, dqkv.ptr, qkv_bias.grad.ptr if qkv_bias is not None else None, device.stream())
            return [dqkv]
        _record(tape, [qkv], ctx, backward)
    return ctx


def dropout(x, p_drop):
    """tf.keras.layers.Dropout in training mode (polus/ner/models.py:58)."""
    if p_drop <= 0:
        return x
    x = cast(x, BF16)
    assert x.size % 8 == 0
    y = Tensor(x.shape, BF16)
    site, seed = _next_site(), _rng_state["seed"]
    _lib.call("polus_dropout", x.ptr, y.ptr, x.size, p_drop, seed, site, step_counter(), device.stream())
    tape = _recording(x)
    if tape is not None:
        def backward(g):
            g = cast(g, BF16)
            dx = Tensor(x.shape, BF16)
            _lib.call("polus_dropout", g.ptr, dx.ptr, g.size, p_drop, seed, site, step_counter(), device.stream())
            return [dx]
        _record(tape, [x], y, backward)
    return y


def gather_rows(x, first, step, n_rows):
    """out[i] = x2d[first + i*step]  (e.g. h[:,0,:] pooling, polus/models.py:216)."""
    cols = x.shape[-1]
    esz = device.dtype_size(x.dtype)
    out = Tensor((n_rows, cols), x.dtype)
    _lib.call("polus_gather_rows", x.ptr, cols * esz, cols * esz, first, step, n_rows, out.ptr, device.stream())
    tape = _recording(x)
    if tape is not None:
        def backward(g):
            g = cast(g, BF16)
            dx = Tensor(x.shape, BF16, zero=True)
            _lib.call("polus_scatter_rows_add_bf16", g.ptr, cols, first, step, n_rows, dx.ptr, device.stream())
            return [dx if x.dtype == BF16 else cast(dx, x.dtype)]
        _record(tape, [x], out, backward)
    return out


# ------------------------------------------------------------------------------------------------
# losses
# ------------------------------------------------------------------------------------------------
def crf_nll_loss(emissions, tags, transitions, lens=None, sample_weights=None):
    """mean_b(w_b * -crf_log_likelihood)  (polus/layers.py:86-126 via tensorflow_addons)."""
    emissions = cast(emissions, F32)
    Bsz, T, K = emissions.shape
    loss = Tensor((), F32)
    nll = Tensor((Bsz,), F32)
    gemis = Tensor(emissions.shape, F32)
    tape = _recording(emissions, transitions)
    is_param = isinstance(transitions, Param)
    gtrans = Tensor(transitions.shape, F32, zero=True) if tape is not None else None  # the kernel accumulates into it
    _lib.call("polus_crf_nll", emissions.ptr, tags.ptr, lens.ptr if lens is not None else None, transitions.ptr,
              sample_weights.ptr if sample_weights is not None else None, Bsz, T, K, nll.ptr, loss.ptr, gemis.ptr,
              gtrans.ptr if tape is not None else None, device.stream())
    if tape is not None:
        def backward(g):
            # The kernel produced d loss / d(emissions, transitions) with the forward pass.  In polus the loss is the
            # root of the tape (training.py:180-185, g == 1); a user loss that scales or combines it (0.5*crf + aux)
            # arrives here with its own upstream gradient, applied as a scalar broadcast.
            ge, gt = (gemis, gtrans) if g.is_one else (_scale_by(gemis, g), _scale_by(gtrans, g))
            if is_param:  # accumulated in BACKWARD: evaluating the loss twice, or only in forward, leaves .grad alone
                _lib.call("polus_binary_f32", 0, transitions.grad.ptr, gt.ptr, gt.size, gt.size, transitions.grad.ptr,
                          device.stream())
            return [ge, None if is_param else gt]
        _record(tape, [emissions, transitions], loss, backward)
    return loss


def _scale_by(x, g):
    """x * g for a scalar upstream gradient g (device tensor), no tape."""
    out = Tensor(x.shape, F32)
    _lib.call("polus_binary_f32", 2, x.ptr, cast(g, F32).ptr, x.size, 1, out.ptr, device.stream())
    return out


def crf_decode(emissions, transitions, lens=None):
    emissions = cast(emissions, F32)
    Bsz, T, K = emissions.shape
    tags = Tensor((Bsz, T), I32)
    score = Tensor((Bsz,), F32)
    _lib.call("polus_crf_decode", emissions.ptr, lens.ptr if lens is not None else None, transitions.ptr, Bsz, T, K,
              tags.ptr, score.ptr, device.stream())
    return tags, score


def cross_entropy(kind, logits, labels, class_weights=None, negative_weight=0.0):
    logits = cast(logits, F32)
    Cn = logits.shape[-1]
    rows = logits.size // Cn
    loss = Tensor((), F32)
    glog = Tensor(logits.shape, F32)
    _lib.call("polus_xent", kind, logits.ptr, labels.ptr, class_weights.ptr if class_weights is not None else None,
              float(negative_weight), rows, Cn, loss.ptr, glog.ptr, device.stream())
    tape = _recording(logits)
    if tape is not None:
        _record(tape, [logits], loss, lambda g: [glog if g.is_one else _scale_by(glog, g)])
    return loss


# ------------------------------------------------------------------------------------------------
# fp32 element-wise / reductions (score functions and custom losses of polus.ir users)
# ------------------------------------------------------------------------------------------------
def _binary(op, a, b):
    a = cast(a, F32)
    if not isinstance(b, Tensor):
        scalar = float(b)
        b = Tensor((1,), F32)
        _lib.call("polus_fill_f32", b.ptr, scalar, 1, device.stream())
    b = cast(b, F32)
    assert a.size % b.size == 0
    out = Tensor(a.shape, F32)
    _lib.call("polus_binary_f32", op, a.ptr, b.ptr, a.size, b.size, out.ptr, device.stream())
    tape = _recording(a, b)
    if tape is not None:
        def backward(g):
            ga = gb = None
            if op == 0:
                ga, gb_full = g, g
            elif op == 1:
                ga, gb_full = g, unary("neg", g)
            elif op == 2:
                ga, gb_full = _binary(2, g, b), _binary(2, g, a)
            else:
                ga = _binary(3, g, b)
                gb_full = unary("neg", _binary(3, _binary(2, g, out), b))
            if b.requires_grad:
                if b.size == a.size:
                    gb = gb_full
                else:  # broadcast over leading rows
                    gb = Tensor(b.shape, F32)
                    _lib.call("polus_reduce_sum_f32", gb_full.ptr, a.size // b.size, b.size, 0, 1.0, gb.ptr, 0, device.stream())
            return [ga if a.requires_grad else None, gb]
        _record(tape, [a, b], out, backward)
    return out


def add(a, b):
    return _binary(0, a, b)


def sub(a, b):
    return _binary(1, a, b)


def mul(a, b):
    return _binary(2, a, b)


def div(a, b):
    return _binary(3, a, b)


def unary(name, x, alpha=1.0):
    code = _lib.UNARY[name]
    x = cast(x, F32)
    out = Tensor(x.shape, F32)
    _lib.call("polus_unary_f32", code, x.ptr, None, 0, x.size, out.ptr, alpha, device.stream())
    tape = _recording(x)
    if tape is not None:
        def backward(g):
            dx = Tensor(x.shape, F32)
            _lib.call("polus_unary_f32", code, x.ptr, cast(g, F32).ptr, 1, x.size, dx.ptr, alpha, device.stream())
            return [dx]
        _record(tape, [x], out, backward)
    return out


def reduce_sum(x, axis=None, mean=False):
    """Sum (or mean) over everything (axis=None) or over the last axis (axis=-1)."""
    x = cast(x, F32)
    if axis is None:
        rows, cols = 1, x.size
        out_shape = ()
    else:
        assert axis in (-1, x.ndim - 1)
        cols = x.shape[-1]
        rows = x.size // cols
        out_shape = x.shape[:-1]
    scale = 1.0 / cols if mean else 1.0
    out = Tensor(out_shape, F32)
    _lib.call("polus_reduce_sum_f32", x.ptr, rows, cols, 1, scale, out.ptr, 0, device.stream())
    tape = _recording(x)
    if tape is not None:
        def backward(g):
            # broadcast g back over the reduced axis: dx[r, c] = g[r] * scale
            ones = Tensor((rows, cols), F32)
            _lib.call("polus_fill_f32", ones.ptr, scale, ones.size, device.stream())
            dx = Tensor(x.shape, F32)
            # dx = ones * g (row broadcast): use binary with transposed roles via per-row scaling
            gcol = cast(g, F32)
            _broadcast_rows_mul(ones, gcol, rows, cols, dx)
            return [dx]
        _record(tape, [x], out, backward)
    return out


def _broadcast_rows_mul(mat, vec, rows, cols, out):
    """out[r, c] = mat[r, c] * vec[r]  -- expressed as a K=1 outer product on the CUDA-core GEMM."""
    if rows == 1:
        _lib.call("polus_binary_f32", 2, mat.ptr, vec.ptr, mat.size, 1, out.ptr, device.stream())
        return
    onesrow = Tensor((cols,), F32)
    _lib.call("polus_fill_f32", onesrow.ptr, 1.0, cols, device.stream())
    tmp = Tensor((rows, cols), F32)
    _gemm(rows, cols, 1, _operand(vec.ptr, 1, False, F32), _operand(onesrow.ptr, 1, False, F32), tmp.ptr, cols, F32,
          force_small=True)
    _lib.call("polus_binary_f32", 2, mat.ptr, tmp.ptr, mat.size, tmp.size, out.ptr, device.stream())


def reduce_mean(x, axis=None):
    return reduce_sum(x, axis=axis, mean=True)


def slice_rows(x, first, n):
    """Contiguous row slice x[first:first+n] of a 1-D / 2-D fp32 tensor (view; gradient scattered back)."""
    x = cast(x, F32)
    cols = 1 if x.ndim == 1 else x.shape[-1]
    shape = (n,) if x.ndim == 1 else (n, cols)
    out = Tensor(shape, F32, ptr=x.ptr + first * cols * 4, block=x.block)
    tape = _recording(x)
    if tape is not None:
        def backward(g):
            dx = Tensor(x.shape, F32, zero=True)
            _lib.call("polus_memcpy_d2d", dx.ptr + first * cols * 4, cast(g, F32).ptr, n * cols * 4, device.stream())
            return [dx]
        _record(tape, [x], out, backward)
    return out


def gather_cols0(x):
    """Column 0 of a 2-D fp32 tensor as a vector (score heads padded to 8 outputs)."""
    x = cast(x, F32)
    rows, cols = x.shape
    sel = Tensor((cols, 1), F32, zero=True)
    _lib.call("polus_fill_f32", sel.ptr, 1.0, 1, device.stream())
    out = matmul(x, sel)
    return reshape(out, (rows,))


_const_cache = {}


def constant_arange(n):
    """int32 [0..n) on the device, created once per n (host uploads are not allowed while a step is being
    captured, so constants are built on the first, op-by-op, call and reused afterwards)."""
    t = _const_cache.get(("arange", n))
    if t is None:
        t = _const_cache[("arange", n)] = Tensor.from_numpy(np.arange(n, dtype=np.int32), I32)
    return t


def clip_by_global_norm(grads, clip_norm):
    """tf.clip_by_global_norm for a post_process_grads hook (polus/training.py:187-189): every gradient is scaled by
    clip_norm / max(global_norm, clip_norm), in place, with no host round trip (usable inside the captured step).
    Returns (grads, global_norm_squared device scalar)."""
    sumsq = Tensor((1,), F32, zero=True)
    st = device.stream()
    live = [g for g in grads if g is not None]
    for g in live:
        assert g.dtype == F32, "clip_by_global_norm works on the fp32 gradient arena views"
        _lib.call("polus_sumsq_f32", g.ptr, g.size, sumsq.ptr, st)
    for g in live:
        _lib.call("polus_scale_by_clip", g.ptr, g.size, sumsq.ptr, float(clip_norm), st)
    return grads, sumsq
