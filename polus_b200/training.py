"""polus.training (reference polus/training.py:14-397): BaseTrainer / ClassifierTrainer.

Same constructor, attributes, override points and loop as the reference; `train_step` is where the
device work happens.  The reference wraps it in `@tf.function` (one static graph per input signature,
retraced on new shapes, training.py:150-151,171); here the first call with a given signature runs the
step once under CUDA stream capture -- forward, loss, backward, gradient allreduce, optimizer -- and
every later call copies the batch into the graph's input buffers and replays it with one launch.
The returned loss is a lazy handle: it syncs only when a callback formats or does arithmetic on it
(SURVEY.md §3.2), so the host loop never stalls the GPU by itself.
"""
import ctypes as C
import os
import weakref

import numpy as np

from . import PolusContext, _lib, device, hvd as _hvd, logger, ops, tensor
from .callbacks import CallbackCoordinator, Profiler
from .tensor import BF16, F32, I32, Tensor


class LazyLoss:
    """Scalar loss of one step, living in a pinned host slot filled by an async D2H copy."""

    __slots__ = ("_slot", "_event", "_value", "__weakref__")

    def __init__(self, slot_array, event):
        self._slot, self._event, self._value = slot_array, event, None

    def _get(self):
        if self._value is None:
            _lib.call("polus_event_sync", self._event)
            self._value = float(self._slot[0])
        return self._value

    def numpy(self):
        return np.float32(self._get())

    def __float__(self):
        return self._get()

    def __format__(self, spec):
        return format(self._get(), spec)

    def __repr__(self):
        return f"LazyLoss({self._get()})"

    def __mul__(self, o):
        return self._get() * o

    __rmul__ = __mul__

    def __add__(self, o):
        return self._get() + o

    __radd__ = __add__

    def __sub__(self, o):
        return self._get() - o

    def __rsub__(self, o):
        return o - self._get()

    def __truediv__(self, o):
        return self._get() / o

    def __lt__(self, o):
        return self._get() < float(o)

    def __gt__(self, o):
        return self._get() > float(o)

    def __array__(self, dtype=None, copy=None):
        return np.asarray(self._get(), dtype=dtype or np.float32)


_LOSS_RING = 256


def _flatten_inputs(inputs):
    """(structure, leaves): leaves are numpy arrays / Tensors in a deterministic order."""
    leaves = []

    def walk(x):
        if isinstance(x, dict):
            return {k: walk(x[k]) for k in x}
        if isinstance(x, (list, tuple)):
            return type(x)(walk(v) for v in x)
        if x is None:
            return None
        leaves.append(x)
        return ("leaf", len(leaves) - 1)
    return walk(list(inputs)), leaves


def _rebuild(struct, leaves):
    if isinstance(struct, dict):
        return {k: _rebuild(v, leaves) for k, v in struct.items()}
    if isinstance(struct, tuple) and len(struct) == 2 and struct[0] == "leaf":
        return leaves[struct[1]]
    if isinstance(struct, (list, tuple)):
        return type(struct)(_rebuild(v, leaves) for v in struct)
    return struct


def _leaf_dtype(x):
    if isinstance(x, Tensor):
        return x.dtype
    a = np.asarray(x)
    if a.dtype.kind == "f":
        return F32
    if a.dtype == np.uint8 or a.dtype == np.bool_:
        return tensor.U8
    return I32


_STAGE_SLOTS = 3   # pinned / device staging ring of the input feed
_copy_stream = [None]


def _h2d_stream():
    if _copy_stream[0] is None:
        st = C.c_void_p()
        _lib.call("polus_stream_create", C.byref(st), 0)
        _copy_stream[0] = st.value
    return _copy_stream[0]


def _new_event():
    ev = C.c_void_p()
    _lib.call("polus_event_create", C.byref(ev))
    return ev.value


class _CompiledStep:
    """One captured CUDA graph + its static input buffers (one per input signature).

    Input feed (host batches): the graph reads fixed device buffers.  Each step's numpy leaves are copied into one slot
    of a ring of pinned host buffers, shipped by an async H2D copy on a dedicated copy stream into that slot's device
    staging buffers -- overlapping the previous step's compute -- and moved into the graph's inputs by a device-to-device
    copy on the compute stream right before the replay.  A slot is rewritten only after the event recorded behind its
    D2D copy has completed, so the host can run ahead of the device without overwriting a batch still in flight."""

    def __init__(self, trainer, struct, leaves):
        self.struct = struct
        self.inputs = []   # device tensors the graph reads
        self.host_leaf = []
        for x in leaves:
            dt = _leaf_dtype(x)
            shape = x.shape if isinstance(x, Tensor) else np.asarray(x).shape
            self.inputs.append(Tensor(shape, dt))
            self.host_leaf.append(not isinstance(x, Tensor))
        self.staging = None    # [slot][leaf] pinned host arrays (created on the first host-fed step)
        self.dev_stage = None  # [slot][leaf] device staging tensors
        self.slot_done = [None] * _STAGE_SLOTS   # event behind the D2D copies that consumed the slot
        self.slot_h2d = [None] * _STAGE_SLOTS    # event behind the slot's H2D copies (copy stream)
        self.pos = 0
        self.h2d_bytes = 0
        self.blocks = None
        self.graph = None
        self.loss = None
        self.trainer = trainer

    def _ensure_staging(self):
        if self.staging is None:
            self.staging = [[device.PinnedArray(t.shape, tensor._NP[t.dtype]) for t in self.inputs] for _ in range(_STAGE_SLOTS)]
            self.dev_stage = [[Tensor(t.shape, t.dtype) for t in self.inputs] for _ in range(_STAGE_SLOTS)]
            for k in range(_STAGE_SLOTS):
                self.slot_done[k], self.slot_h2d[k] = _new_event(), _new_event()
            self._slot_used = [False] * _STAGE_SLOTS

    def feed(self, leaves):
        st = device.stream()
        host = [i for i, x in enumerate(leaves) if not isinstance(x, Tensor)]
        for i, (x, t) in enumerate(zip(leaves, self.inputs)):
            if isinstance(x, Tensor) and x.ptr != t.ptr:
                _lib.call("polus_memcpy_d2d", t.ptr, x.ptr, t.nbytes, st)
        self.h2d_bytes = 0
        if not host:
            return
        self._ensure_staging()
        k = self.pos
        self.pos = (k + 1) % _STAGE_SLOTS
        if self._slot_used[k]:
            _lib.call("polus_event_sync", self.slot_done[k])  # the batch that used this slot has reached the graph inputs
        self._slot_used[k] = True
        cs = _h2d_stream()
        for i in host:
            pin, t = self.staging[k][i], self.inputs[i]
            np.copyto(pin.array, np.asarray(leaves[i]), casting="unsafe")
            _lib.call("polus_memcpy_h2d", self.dev_stage[k][i].ptr, pin.ptr, t.nbytes, cs)
            self.h2d_bytes += t.nbytes
        _lib.call("polus_event_record", self.slot_h2d[k], cs)
        _lib.call("polus_stream_wait_event", st, self.slot_h2d[k])
        for i in host:
            _lib.call("polus_memcpy_d2d", self.inputs[i].ptr, self.dev_stage[k][i].ptr, self.inputs[i].nbytes, st)
        _lib.call("polus_event_record", self.slot_done[k], st)

    def capture(self):
        st = device.stream()
        ops.reset_dropout_sites()
        ops.side_reset()
        self.blocks = tensor.begin_trace()
        try:
            _lib.call("polus_graph_begin", st)
            g = C.c_void_p()
            try:
                self.loss = self.trainer._step_body(*_rebuild(self.struct, self.inputs))
            except Exception as e:
                try:  # leave capture mode so the stream stays usable, then report the real cause
                    _lib.call("polus_graph_end", st, C.byref(g))
                except Exception:
                    pass
                raise RuntimeError("the training step could not be captured into a CUDA graph (an op in the model / loss "
                                   "needs a host<->device sync, e.g. creating a tensor from numpy inside the step); "
                                   "set POLUS_EAGER=1 to run op by op") from e
            ops.side_join()
            ops.opt_stream_join()
            _lib.call("polus_graph_end", st, C.byref(g))
            self.graph = g.value
        finally:
            tensor.end_trace()

    def launch(self):
        _lib.call("polus_graph_launch", self.graph, device.stream())

    def release(self):
        """Destroy the graph and hand its activation blocks back to the pool (they were pinned to this trace)."""
        device.device_sync()
        if self.graph is not None:
            _lib.call("polus_graph_destroy", self.graph)
            self.graph = None
        for b in self.blocks or []:
            b.pinned = False
        self.blocks = None
        self.loss = None


class BaseTrainer:
    """Abstraction of a gradient-descent training procedure (reference training.py:14-338)."""

    def __init__(self, model, optimizer, loss, metrics=[], post_process_logits=None, post_process_grads=None):
        if self.__class__.__name__ == "BaseTrainer":
            raise Exception("This is an abstraction that cannot be instantiated")
        super().__init__()
        self.model = model
        self.loss = loss
        self.optimizer = optimizer
        self.post_process_logits = post_process_logits
        self.post_process_grads = post_process_grads
        self.metrics = metrics
        self.early_stop = False
        self.train_config = {}
        self.step_counter = 0
        if not hasattr(self, "trainable_weights"):
            logger.warning(f"Since no specific trainable_weights were defined during the {self.__class__.__name__} "
                           f"instantiation, the trainer will optimizer all the variables found on the model instance")
            self.trainable_weights = model.trainable_weights
            self._auto_weights = True  # Keras models may create variables lazily: re-read after the first forward
        self.use_horovod = PolusContext().is_horovod_enabled()
        self.hvd = _hvd()
        if self.use_horovod:
            if hasattr(optimizer, "learning_rate"):
                _new_lr = optimizer.learning_rate.read_value() * self.hvd.size()
                optimizer.learning_rate.assign(_new_lr)
                logger.info(f"The learning rate was adjusted to account for the multiGPU training, local lr is {_new_lr}")
            else:
                logger.info("It was not possible to change the learning rate to adjusted for the multiGPU training, "
                            "please make the attention to multiply the learning rate by hvd.size()")
            # Horovod op=Average (training.py:182): NCCL sums, the optimizer kernel divides
            if hasattr(optimizer, "grad_scale"):
                optimizer.grad_scale = 1.0 / self.hvd.size()
        # POLUS_EAGER=1 runs every step op-by-op (debugging); default is capture + replay
        self.use_graph = os.environ.get("POLUS_EAGER", "0") != "1"
        self._compiled = {}
        self._warm = set()
        self._loss_ring = None
        self._ring_pos = 0
        self.last_h2d_bytes = 0

    def __str__(self):
        return 'Trainer'

    def forward_without_grads(self, *inputs):
        return inputs

    def forward_with_grads(self, *inputs):
        raise NotImplementedError("forward_with_grads function must be implemented in order to compute a loss value for optimization")

    # -------------------------------------------------------------------------------- the step
    def _step_body(self, *inputs):
        """The computation polus/training.py:173-193 traces: forward, loss, backward, allreduce, update."""
        with ops.GradientTape() as tape:
            with tape.stop_recording():
                inputs = self.forward_without_grads(*inputs)
            inputs = self.forward_with_grads(*inputs)
            loss_value = self.loss(*inputs)
        if getattr(self, "_auto_weights", False) and hasattr(self.model, "trainable_weights"):
            # Keras-style lazy build: some variables exist only after the first call
            current = self.model.trainable_weights
            if len(current) != len(self.trainable_weights):
                self.trainable_weights = current
        tape = self.hvd.DistributedGradientTape(tape)
        # without a gradient post-processing hook nothing reads the full gradient list before the update, so each
        # contiguous span of the arena is updated as soon as backward has finished with it (captured steps only)
        early = None
        if (self.post_process_grads is None and ops.side_active()
                and hasattr(self.optimizer, "apply_span_early")):
            early = self.optimizer.apply_span_early
        grads = tape.gradient(loss_value, self.trainable_weights, on_bucket_ready=early) if early is not None \
            else tape.gradient(loss_value, self.trainable_weights)
        if self.post_process_grads is not None:
            grads = self.post_process_grads(grads)
        self.optimizer.apply_gradients(zip(grads, self.trainable_weights))
        return loss_value

    def _lazy_loss(self, loss_tensor):
        if self._loss_ring is None:
            self._loss_ring = device.PinnedArray((_LOSS_RING, 4), np.float32)
            self._loss_events = []
            self._loss_owner = [None] * _LOSS_RING   # weakref to the LazyLoss currently reading each slot
            for _ in range(_LOSS_RING):
                ev = C.c_void_p()
                _lib.call("polus_event_create", C.byref(ev))
                self._loss_events.append(ev.value)
        i = self._ring_pos
        self._ring_pos = (i + 1) % _LOSS_RING
        # a handle from _LOSS_RING steps ago that some callback still holds unread (EarlyStop / ConsoleLogCallback keep
        # them until the epoch ends) takes its value now, before its slot and event are reused
        prev = self._loss_owner[i]() if self._loss_owner[i] is not None else None
        if prev is not None:
            prev._get()
        st = device.stream()
        _lib.call("polus_memcpy_d2h", self._loss_ring.ptr + i * 16, loss_tensor.ptr, 4, st)
        _lib.call("polus_event_record", self._loss_events[i], st)
        out = LazyLoss(self._loss_ring.array[i], self._loss_events[i])
        self._loss_owner[i] = weakref.ref(out)
        return out

    def train_step(self, *inputs):
        """One optimisation step on one batch; returns the (lazy) scalar loss of that batch."""
        if hasattr(self.optimizer, "sync_hyper"):
            self.optimizer.sync_hyper()   # lr / grad_scale assigned since the last step reach the device before this one
        struct, leaves = _flatten_inputs(inputs)
        key = (repr(struct), tuple((tuple(x.shape) if isinstance(x, Tensor) else np.asarray(x).shape, _leaf_dtype(x))
                                   for x in leaves))
        if not self.use_graph or key not in self._warm:
            # First call per signature runs op by op: it builds lazily-created variables, optimizer
            # slots and per-kernel attributes (all of which need host<->device syncs that a stream
            # capture forbids).  The second call captures, later calls replay.
            self._warm.add(key)
            ops.reset_dropout_sites()
            dev = [x if isinstance(x, Tensor) else Tensor.from_numpy(np.asarray(x), _leaf_dtype(x)) for x in leaves]
            self.last_h2d_bytes = sum(t.nbytes for t, x in zip(dev, leaves) if not isinstance(x, Tensor))
            return self._lazy_loss(self._step_body(*_rebuild(struct, dev)))
        step = self._compiled.get(key)
        if step is None:
            logger.debug("train_step was traced (more than a few traces means the step is receiving inputs with "
                         "different shapes or dtypes)")
            step = _CompiledStep(self, struct, leaves)
            step.feed(leaves)
            step.capture()
            self._compiled[key] = step
        else:
            step.feed(leaves)
        step.launch()
        self.last_h2d_bytes = step.h2d_bytes
        return self._lazy_loss(step.loss)

    def release_graphs(self):
        """Forget every captured step (new shapes re-capture): frees the activation memory pinned to those graphs."""
        for step in self._compiled.values():
            step.release()
        self._compiled = {}
        self._warm = set()

    def lr_finder(self, tf_dataset, use_lr_found=False):
        pass

    def changing_train_config(self, **config):
        for k, v in config.items():
            self.train_config[k] = v

    def broadcast_init_vars(self):
        self.hvd.broadcast_variables(self.trainable_weights, root_rank=0)
        self.hvd.broadcast_variables(self.optimizer.variables(), root_rank=0)

    # -------------------------------------------------------------------------------- the loop
    def train(self, tf_dataset=None, epochs=None, callbacks=[], train_map_f=None, steps=None, **kwargs):
        if tf_dataset is None:
            if "tf_dataset" in self.train_config:
                tf_dataset = self.train_config["tf_dataset"]
            else:
                raise ValueError("You need to pass a training dataset to the trainer.train method")
        if epochs is None:
            if "epochs" in self.train_config:
                epochs = self.train_config["epochs"]
            else:
                raise ValueError("You need to pass the epochs variable to the trainer.train method")
        if len(callbacks) == 0 and "callbacks" in self.train_config:
            callbacks = self.train_config["callbacks"]
        if train_map_f is None and "train_map_f" in self.train_config:
            train_map_f = self.train_config["train_map_f"]
        if steps is None and "steps" in self.train_config:
            steps = self.train_config["steps"]

        if steps is None:
            if hasattr(tf_dataset, "cardinality"):
                N_STEPS = tf_dataset.cardinality()
            elif hasattr(tf_dataset, "__len__"):
                N_STEPS = len(tf_dataset)
            else:
                N_STEPS = -2  # tf.data UNKNOWN_CARDINALITY
        else:
            N_STEPS = steps

        if "custom_data_transform_f" in kwargs:
            train_map_f = kwargs.pop("custom_data_transform_f")

        if os.getenv("POLUS_PROFILER", 'False').lower() in ('true', '1', 't', 'y', 'yes'):
            logger.info("POLUS_PROFILER env was set to True, so the Profiler callback was added to training")
            profiler_step_range = list(map(int, os.getenv("POLUS_PROFILER_RANGE", '10:20').split(":")))
            callbacks = list(callbacks) + [Profiler(steps_interval=profiler_step_range)]

        if not isinstance(callbacks, CallbackCoordinator):
            callbacks = CallbackCoordinator(callbacks, trainer=self, epochs=epochs, steps=N_STEPS)
        self.callbacks = callbacks
        self.callbacks.on_train_begin()

        for epoch in range(epochs):
            self.callbacks.on_epoch_begin(epoch)
            _iter = iter(tf_dataset)
            step = 0
            while True:
                self.callbacks.on_train_batch_begin(epoch, step)
                data = next(_iter, None)
                if data is None:
                    break
                if train_map_f is not None:
                    data = train_map_f(data)
                if step == 0 and self.use_horovod:
                    self.broadcast_init_vars()
                loss = self.train_step(*data)
                self.callbacks.on_train_batch_end(epoch, step, loss)
                self.step_counter += 1
                step += 1
                if self.early_stop:
                    break
            self.callbacks.on_epoch_end(epoch)
            if self.early_stop:
                break
        self.callbacks.on_train_end()


class ClassifierTrainer(BaseTrainer):
    """Standard classifier trainer (reference training.py:341-397)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)

    def forward_with_grads(self, x, y):
        if isinstance(x, dict):
            logits = self.model(**x, training=True)
        else:
            logits = self.model(x, training=True)
        if self.post_process_logits is not None:
            logits = self.post_process_logits(logits)
        return y, logits
