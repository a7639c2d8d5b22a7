"""ctypes binding of libpolus_b200.so (the C ABI declared in include/polus_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this module raises.
The reference has no FFI (SURVEY.md §8b); INTEGRATION.md shows how polus itself would bind this ABI.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("POLUS_LIB") or os.path.join(_HERE, "libpolus_b200.so")  # POLUS_LIB: A/B builds of the same ABI

F32, BF16, I32, U8 = 0, 1, 2, 3
ACT = {None: 0, "linear": 0, "none": 0, "gelu": 1, "relu": 2, "swish": 3, "silu": 3, "tanh": 4, "mish": 5}
ACT_DERIV = 100  # polus_act_bwd_colsum: `z` already holds act'(pre-activation) (written by the forward GEMM, c2_kind = 1)
ACT_DERIV_U8 = 101  # ... as 8-bit fixed point (c2_kind = 2)
UNARY = {"exp": 16, "log": 17, "softplus": 18, "sigmoid": 19, "neg": 20, "square": 21, "scale": 22,
         "gelu": 1, "relu": 2, "swish": 3, "tanh": 4, "mish": 5, "identity": 0}


class PolusError(RuntimeError):
    pass


class PolusOOM(MemoryError):
    pass


class Operand(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("ld", C.c_int64), ("bs0", C.c_int64), ("bs1", C.c_int64),
                ("mn_major", C.c_int32), ("dtype", C.c_int32)]


class Gemm(C.Structure):
    _fields_ = [("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
                ("batch0", C.c_int32), ("batch1", C.c_int32),
                ("A", Operand), ("B", Operand),
                ("C", C.c_void_p), ("ldc", C.c_int64), ("cbs0", C.c_int64), ("cbs1", C.c_int64),
                ("c_dtype", C.c_int32), ("C2", C.c_void_p), ("bias", C.c_void_p),
                ("alpha", C.c_float), ("act", C.c_int32), ("accumulate", C.c_int32),
                ("split_k", C.c_int32), ("c2_kind", C.c_int32), ("Emul", C.c_void_p), ("colsum", C.c_void_p)]


class AdamCfg(C.Structure):
    _fields_ = [("lr", C.c_float), ("schedule", C.c_int32), ("warmup_steps", C.c_int32),
                ("decay_steps", C.c_int32), ("end_lr", C.c_float), ("beta1", C.c_float),
                ("beta2", C.c_float), ("eps", C.c_float), ("weight_decay", C.c_float),
                ("grad_scale", C.c_float)]


p, i32, i64, u32, u64, f32, sz = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64, C.c_float, C.c_size_t

# name -> argtypes (return type is int status unless listed in _RET)
_SIGS = {
    "polus_version": [],
    "polus_init": [i32],
    "polus_device_count": [C.POINTER(i32)],
    "polus_device_info": [C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(sz)],
    "polus_malloc": [C.POINTER(p), sz],
    "polus_free": [p],
    "polus_host_alloc": [C.POINTER(p), sz],
    "polus_host_free": [p],
    "polus_memcpy_h2d": [p, p, sz, p],
    "polus_memcpy_d2h": [p, p, sz, p],
    "polus_memcpy_d2d": [p, p, sz, p],
    "polus_memset": [p, i32, sz, p],
    "polus_stream_create": [C.POINTER(p), i32],
    "polus_stream_destroy": [p],
    "polus_stream_sync": [p],
    "polus_device_sync": [],
    "polus_event_create": [C.POINTER(p)],
    "polus_event_destroy": [p],
    "polus_event_record": [p, p],
    "polus_event_sync": [p],
    "polus_event_elapsed_ms": [p, p, C.POINTER(f32)],
    "polus_stream_wait_event": [p, p],
    "polus_graph_begin": [p],
    "polus_graph_end": [p, C.POINTER(p)],
    "polus_graph_launch": [p, p],
    "polus_graph_destroy": [p],
    "polus_launch_count": [],
    "polus_profiler_start": [],
    "polus_profiler_stop": [],
    "polus_profiler_range_push": [C.c_char_p],
    "polus_profiler_range_pop": [],
    "polus_gemm_tc": [C.POINTER(Gemm), p],
    "polus_gemm_small": [C.POINTER(Gemm), p],
    "polus_gemm_tc_supported": [C.POINTER(Gemm)],
    "polus_skinny_supported": [i32, i32],
    "polus_skinny_fwd": [p, i32, p, p, i32, i32, i32, i32, p, p, p],
    "polus_skinny_bwd": [p, i32, p, p, i32, i32, i32, p, i32, p, p, p],
    "polus_embed_ln_fwd": [p, p, p, p, p, p, p, i32, i32, i32, i32, i32, f32, f32, u64, u32, p, p, p, p, p, p],
    "polus_embed_ln_bwd": [p, p, p, p, p, p, p, i32, i32, i32, i32, i32, f32, u64, u32, p, p, p, p, p, p, p, p],
    "polus_embed_ws_floats": [i32, i32, i32],
    "polus_embed_ln_fwd_pos": [p, p, p, p, p, p, p, i32, i32, i32, i32, i32, f32, f32, u64, u32, p, p, p, p, p, p, i32, p],
    "polus_embed_ln_bwd_pos": [p, p, p, p, p, p, p, i32, i32, i32, i32, i32, f32, u64, u32, p, p, p, p, p, p, p, p, i32, p],
    "polus_position_ids": [p, i32, i32, i32, p, p],
    "polus_add_bf16": [p, p, p, i64, p],
    "polus_ln_res_fwd": [p, p, p, p, i32, i32, f32, f32, u64, u32, p, p, p, p, p, p],
    "polus_ln_res_bwd": [p, p, p, p, p, p, i32, i32, f32, u64, u32, p, p, p, p, p, p, p, p],
    "polus_ln_ws_floats": [i32],
    "polus_softmax_fwd": [p, p, i32, i32, i32, i32, f32, f32, u64, u32, p, p, p, p],
    "polus_softmax_bwd": [p, p, i32, i32, i32, i32, f32, f32, u64, u32, p, p],
    "polus_attention_supported": [i32, i32],
    "polus_attention_keepbits_words": [i32, i32, i32],
    "polus_attention_fwd": [p, p, i32, i32, i32, i32, f32, u64, u32, p, p, p, p, p],
    "polus_attention_bwd": [p, p, p, p, p, i32, i32, i32, i32, f32, u64, u32, p, p, p, p, p],
    "polus_act_bwd_colsum": [p, p, i32, i32, i32, p, p, p, p],
    "polus_colsum_ws_floats": [i32],
    "polus_dropout": [p, p, i64, f32, u64, u32, p, p],
    "polus_crf_nll": [p, p, p, p, p, i32, i32, i32, p, p, p, p, p],
    "polus_crf_decode": [p, p, p, i32, i32, i32, p, p, p],
    "polus_crf_mask_transitions": [p, p, i32, p, p],
    "polus_crf_sample_weights": [p, p, f32, i32, i32, i32, p, p],
    "polus_xent": [i32, p, p, p, f32, i32, i32, p, p, p],
    "polus_gather_positions": [p, p, i32, i32, i32, i32, p, p],
    "polus_scatter_positions_add": [p, p, i32, i32, i32, i32, p, p],
    "polus_vocab_xent": [p, i32, i32, i64, p, p, p, p, p, p],
    "polus_colsum_bf16": [p, i32, i32, i64, p, p],
    "polus_adam": [p, p, p, p, p, p, i64, C.POINTER(AdamCfg), p, p, i32, p],
    "polus_cast": [p, i32, p, i32, i64, p],
    "polus_fill_f32": [p, f32, i64, p],
    "polus_binary_f32": [i32, p, p, i64, i64, p, p],
    "polus_unary_f32": [i32, p, p, i32, i64, p, f32, p],
    "polus_reduce_sum_f32": [p, i32, i32, i32, f32, p, i32, p],
    "polus_argmax_f32": [p, i32, i32, p, p],
    "polus_one_hot_f32": [p, i32, i32, p, p],
    "polus_confusion_matrix": [p, p, i64, i32, p, p],
    "polus_gather_rows": [p, i64, i64, i64, i64, i64, p, p],
    "polus_scatter_rows_add_bf16": [p, i64, i64, i64, i64, p, p],
    "polus_sumsq_f32": [p, i64, p, p],
    "polus_scale_by_clip": [p, i64, p, f32, p],
    "polus_comm_unique_id": [p],
    "polus_comm_init": [i32, i32, p],
    "polus_comm_init_cfg": [i32, i32, p, i32],
    "polus_comm_size": [],
    "polus_comm_rank": [],
    "polus_comm_allreduce_f32": [p, i64, p],
    "polus_comm_allreduce_bf16": [p, p, i64, p],
    "polus_comm_broadcast": [p, sz, i32, p],
    "polus_comm_allgather": [p, p, sz, p],
    "polus_comm_destroy": [],
}
_RET = {"polus_launch_count": C.c_int64, "polus_ln_ws_floats": sz, "polus_colsum_ws_floats": sz,
        "polus_embed_ws_floats": sz, "polus_attention_keepbits_words": sz}
# functions whose int return is a value, not a status
_VALUE_RET = {"polus_version", "polus_gemm_tc_supported", "polus_skinny_supported", "polus_attention_supported", "polus_attention_keepbits_words", "polus_comm_size", "polus_comm_rank",
              "polus_launch_count", "polus_ln_ws_floats", "polus_colsum_ws_floats", "polus_embed_ws_floats"}

EXPORTS = ["polus_last_error"] + list(_SIGS)

_lib = None


def load():
    """Load the shared library (once). Raises PolusError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PolusError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(polus_b200 has no CPU fallback)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    lib.polus_last_error.restype = C.c_char_p
    lib.polus_last_error.argtypes = []
    for name, args in _SIGS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:  # reported by missing_exports(); calling it raises below
            continue
        fn.argtypes = args
        fn.restype = _RET.get(name, C.c_int)
    _lib = lib
    return lib


def missing_exports():
    """Symbols include/polus_b200.h declares that the loaded library does not export."""
    lib = load()
    out = []
    for name in EXPORTS:
        try:
            getattr(lib, name)
        except AttributeError:
            out.append(name)
    return out


def last_error():
    return load().polus_last_error().decode("utf-8", "replace")


# POLUS_ABLATE=name[,name...]: profiling aid (tools/ablate_step.py) -- the listed entry points become no-ops, so the
# step time without them gives their true marginal cost inside the replayed graph.  Results are garbage by design.
_ABLATE = frozenset(n for n in os.environ.get("POLUS_ABLATE", "").split(",") if n)


_ONLY = None  # set_only(): every kernel entry point NOT in this set becomes a no-op (bench.py's GEMM-only replay)
_PLUMBING = ("polus_malloc", "polus_free", "polus_host_", "polus_memcpy", "polus_memset", "polus_stream_", "polus_device_",
             "polus_event_", "polus_graph_", "polus_launch_count", "polus_profiler_", "polus_init", "polus_version",
             "polus_comm_init", "polus_comm_unique_id", "polus_comm_size", "polus_comm_rank", "polus_comm_destroy")


def set_only(names):
    """Profiling aid: keep memory/stream/graph plumbing and the listed kernel entry points, skip every other one
    (None restores normal operation).  Used to replay the step's GEMM launches alone, in order, on the step's own
    buffers, for the roofline figure; results of such a replay are garbage by design."""
    global _ONLY
    _ONLY = None if names is None else frozenset(names)


def call(name, *args):
    """Call a status-returning entry point; raise the matching Python exception on failure."""
    if _ABLATE and name in _ABLATE:
        return 0
    if _ONLY is not None and name not in _ONLY and name not in _VALUE_RET and not name.startswith(_PLUMBING):
        return 0
    rc = getattr(load(), name)(*args)
    if name in _VALUE_RET:
        return rc
    if rc != 0:
        msg = f"{name} failed ({rc}): {last_error()}"
        if rc == -4:
            raise PolusOOM(msg)
        if rc in (-1, -5):
            raise ValueError(msg)
        raise PolusError(msg)
    return 0
