"""Device tensors, the activation pool and the flat parameter arena.

The reference keeps variables inside Keras layers and lets TF's allocator own activations
(SURVEY.md §8b "Ownership").  Here libpolus_b200.so owns all device memory; Python holds handles:

* `Tensor`     -- (ptr, shape, dtype) view of device memory, optionally attached to the autograd tape.
* `Param`      -- a trainable slice of the `ParamArena`: fp32 master, fp32 gradient, bf16 shadow (the
                  GEMM operand), laid out contiguously in creation order so that one fused Adam launch
                  and a handful of contiguous NCCL buckets cover every variable
                  (polus/training.py:185-191 does this per variable, ~200 launches).
* activation buffers come from a size-bucketed pool; while a train step is being captured into a
  CUDA graph they are pinned to that trace (never recycled while the graph can replay).
"""
import ctypes as C

import numpy as np

from . import _lib, device

F32, BF16, I32, U8 = _lib.F32, _lib.BF16, _lib.I32, _lib.U8
_NP = {F32: np.float32, BF16: np.uint16, I32: np.int32, U8: np.uint8}
_NAMES = {F32: "float32", BF16: "bfloat16", I32: "int32", U8: "uint8"}


def _round_size(n):
    if n <= 1 << 20:
        return max(256, (n + 255) & ~255)
    return (n + (1 << 21) - 1) & ~((1 << 21) - 1)


class _Pool:
    """Caching allocator: freed blocks are kept per rounded size and handed out again."""

    def __init__(self):
        self.free = {}
        self.trace = None  # list collecting blocks while a step is being traced

    def take(self, nbytes):
        size = _round_size(int(nbytes))
        lst = self.free.get(size)
        if lst:
            ptr = lst.pop()
        else:
            p = C.c_void_p()
            try:
                _lib.call("polus_malloc", C.byref(p), size)
            except _lib.PolusOOM:
                self.release_cached()
                _lib.call("polus_malloc", C.byref(p), size)
            ptr = p.value
        return ptr, size

    def give(self, ptr, size):
        self.free.setdefault(size, []).append(ptr)

    def release_cached(self):
        for lst in self.free.values():
            for ptr in lst:
                _lib.load().polus_free(ptr)
        self.free = {}


_pool = _Pool()


class Block:
    """One pooled allocation; returns to the pool when the last Tensor using it dies."""

    __slots__ = ("ptr", "size", "pinned")

    def __init__(self, nbytes):
        device.stream()  # make sure the device is initialised
        self.ptr, self.size = _pool.take(nbytes)
        self.pinned = False
        if _pool.trace is not None:
            _pool.trace.append(self)
            self.pinned = True

    def __del__(self):
        try:
            if not self.pinned and self.ptr:
                _pool.give(self.ptr, self.size)
        except Exception:
            pass


def begin_trace():
    _pool.trace = []
    return _pool.trace


def end_trace():
    _pool.trace = None


class Tensor:
    __slots__ = ("ptr", "shape", "dtype", "block", "requires_grad", "node", "name", "consumers", "bwd_fuse", "fused_for",
                 "is_one", "__weakref__")

    def __init__(self, shape, dtype, ptr=None, block=None, zero=False):
        self.shape = tuple(int(s) for s in shape)
        self.dtype = dtype
        self.requires_grad = False
        self.node = None
        self.name = None
        self.consumers = 0     # tape nodes that read this tensor (ops._record)
        self.bwd_fuse = None   # (act' tensor, bias-grad tensor): the consumer's dgrad GEMM may apply them in its epilogue
        self.fused_for = None  # id() of the activation output whose backward this gradient already includes
        self.is_one = False    # the tape's root gradient (d loss / d loss == 1): loss ops skip the multiply
        if ptr is None:
            block = Block(max(self.nbytes, 16))
            ptr = block.ptr
            if zero and self.nbytes:
                _lib.call("polus_memset", ptr, 0, self.nbytes, device.stream())
        self.ptr = ptr
        self.block = block

    # ------------------------------------------------------------------ properties
    @property
    def size(self):
        n = 1
        for s in self.shape:
            n *= s
        return n

    @property
    def nbytes(self):
        return self.size * device.dtype_size(self.dtype)

    @property
    def ndim(self):
        return len(self.shape)

    def __repr__(self):
        return f"Tensor(shape={self.shape}, dtype={_NAMES[self.dtype]})"

    # ------------------------------------------------------------------ host transfer
    @staticmethod
    def from_numpy(arr, dtype=None):
        arr = np.asarray(arr)
        if dtype is None:
            if arr.dtype in (np.float32, np.float64, np.float16):
                dtype = F32
            elif arr.dtype == np.uint8 or arr.dtype == np.bool_:
                dtype = U8
            else:
                dtype = I32
        if dtype == BF16:
            host = device.f32_to_bf16_bits(arr.astype(np.float32))
        else:
            host = np.ascontiguousarray(arr, dtype=_NP[dtype])
        t = Tensor(arr.shape, dtype)
        if host.nbytes:
            device.upload(t.ptr, host)
        return t

    def numpy(self):
        """Host copy (synchronises the stream).  bf16 comes back as float32."""
        raw = device.download(self.ptr, self.shape, _NP[self.dtype])
        if self.dtype == BF16:
            return device.bf16_bits_to_f32(raw).reshape(self.shape)
        return raw

    def view(self, shape):
        """Alias with a new shape (no copy, not recorded on the tape -- use ops.reshape for that)."""
        shape = list(shape)
        if -1 in shape:
            known = 1
            for s in shape:
                if s != -1:
                    known *= s
            shape[shape.index(-1)] = self.size // max(known, 1)
        t = Tensor(shape, self.dtype, ptr=self.ptr, block=self.block)
        assert t.size == self.size, f"cannot view {self.shape} as {tuple(shape)}"
        return t

    def __float__(self):
        assert self.size == 1
        return float(self.numpy().reshape(-1)[0])

    def __format__(self, spec):
        if self.size == 1:
            return format(float(self), spec)
        return repr(self)


# ------------------------------------------------------------------------------------------------
# parameter arena
# ------------------------------------------------------------------------------------------------
class ArenaChunk:
    _created = 0

    def __init__(self, capacity):
        # creation order: the rank-invariant sort key for anything that orders chunks across processes (id() and device
        # addresses differ from rank to rank, and collectives must be issued in the same order everywhere)
        ArenaChunk._created += 1
        self.index = ArenaChunk._created
        self.capacity = int(capacity)
        self.used = 0
        self.p = device.Buffer(self.capacity * 4, zero=True)
        self.g = device.Buffer(self.capacity * 4, zero=True)
        self.pb = device.Buffer(self.capacity * 2, zero=True)
        self.decay = None  # host-side uint8 mask, uploaded by the optimizer on demand
        self.host_decay = np.zeros(self.capacity, np.uint8)


class ParamArena:
    """Flat storage for every trainable variable of the process, in creation order."""

    DEFAULT_CHUNK = 128 * 1024 * 1024  # parameters per chunk (BERT-base + head = 109.6 M fits in one)

    def __init__(self):
        self.chunks = []
        self.params = []

    def allocate(self, n):
        n_al = (n + 63) & ~63  # keep every variable 256-byte aligned (TMA / float4 friendly)
        for ch in self.chunks:
            if ch.used + n_al <= ch.capacity:
                break
        else:
            ch = ArenaChunk(max(self.DEFAULT_CHUNK if self.chunks else self._first_chunk(n_al), n_al))
            self.chunks.append(ch)
        off = ch.used
        ch.used += n_al
        return ch, off

    def _first_chunk(self, n_al):
        import os
        return int(os.environ.get("POLUS_ARENA_PARAMS", self.DEFAULT_CHUNK))


_arena = None


def arena():
    global _arena
    if _arena is None:
        _arena = ParamArena()
    return _arena


def reset_arena():
    """Drop every parameter (tests / HPO trials that rebuild models from scratch)."""
    global _arena
    _arena = None


class Param(Tensor):
    """Trainable variable: fp32 master + fp32 grad + bf16 shadow at the same arena offset."""

    __slots__ = ("chunk", "offset", "grad", "shadow", "decay")

    def __init__(self, value, name=None, decay=True):
        value = np.ascontiguousarray(value, dtype=np.float32)
        ch, off = arena().allocate(value.size)
        Tensor.__init__(self, value.shape, F32, ptr=ch.p.ptr + off * 4, block=ch)
        self.chunk, self.offset = ch, off
        self.grad = Tensor(value.shape, F32, ptr=ch.g.ptr + off * 4, block=ch)
        self.shadow = Tensor(value.shape, BF16, ptr=ch.pb.ptr + off * 2, block=ch)
        self.requires_grad = True
        self.name = name
        self.decay = decay
        ch.host_decay[off:off + value.size] = 1 if decay else 0
        arena().params.append(self)
        self.assign(value)

    def assign(self, value):
        value = np.ascontiguousarray(value, dtype=np.float32).reshape(self.shape)
        device.upload(self.ptr, value)
        device.upload(self.shadow.ptr, device.f32_to_bf16_bits(value))

    def read_value(self):
        return self.numpy()
