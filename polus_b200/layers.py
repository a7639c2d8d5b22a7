"""polus.layers.CRF (reference polus/layers.py:6-140) on the CRF kernels of libpolus_b200.so."""
import numpy as np

from . import _lib, device, nn, ops
from .tensor import F32, I32, Tensor


MAX_TAGS = 128  # the largest K that polus_crf_nll / polus_crf_decode accept


class CRF(nn.Layer):
    """Linear-chain CRF output layer.

    Same wiring as the reference: owns `transitions [K,K]` (glorot_uniform), optional
    `mask_impossible_transitions`; `call` returns the emissions unchanged in the training phase and
    the one-hot Viterbi path otherwise (layers.py:65-84); `loss` / `loss_sample_weights` are the
    negative mean log-likelihoods of layers.py:86-126.  `sequence_lengths` defaults to the full
    length for every row (layers.py:74-76) and is remembered for the loss, as in the reference.
    Difference: in the training phase the reference also runs crf_decode and discards the result;
    that dead work is skipped here.
    """

    def __init__(self, output_dim, sparse_target=True, mask_impossible_transitions=None, **kwargs):
        super().__init__(name=kwargs.get("name"))
        self.output_dim = int(output_dim)
        self.sparse_target = sparse_target
        self.sequence_lengths = None
        self.transitions = None
        self.mask_impossible_transitions = mask_impossible_transitions
        self._mask_t = None

    def build(self, input_shape):
        if self.output_dim > MAX_TAGS:
            raise ValueError(f"CRF supports at most {MAX_TAGS} tags in this port (got output_dim={self.output_dim}); "
                             "the reference layer (tensorflow_addons) has no such limit")
        if input_shape is not None:
            assert len(input_shape) == 3
            if input_shape[-1] != self.output_dim:
                raise ValueError("The last dimension of the input shape must be equal to output shape. "
                                 "Use a linear layer if needed.")
        self.transitions = self.add_weight("transitions", nn.glorot_uniform((self.output_dim, self.output_dim)),
                                           decay=False)
        if self.mask_impossible_transitions is not None:
            self._mask_t = Tensor.from_numpy(np.asarray(self.mask_impossible_transitions, np.float32), F32)

    def get_transitions(self):
        """T*mask + float(int32(1-mask)*-10000) (layers.py:56-63), differentiable wrt T."""
        if self._mask_t is None:
            return self.transitions
        K = self.output_dim
        out = Tensor((K, K), F32)
        _lib.call("polus_crf_mask_transitions", self.transitions.ptr, self._mask_t.ptr, K, out.ptr, device.stream())
        tape = ops._recording(self.transitions)
        if tape is not None:
            mask, trans = self._mask_t, self.transitions

            def backward(g):
                gm = ops.mul(g, mask)
                _lib.call("polus_binary_f32", 0, trans.grad.ptr, gm.ptr, K * K, K * K, trans.grad.ptr, device.stream())
                return [None]
            ops._record(tape, [trans], out, backward)
        return out

    def call(self, inputs, sequence_lengths=None, training=None, **kwargs):
        seq = ops.cast(nn.as_tensor(inputs), F32)
        assert seq.ndim == 3
        if sequence_lengths is not None:
            sl = nn.as_tensor(sequence_lengths, I32)
            assert sl.ndim == 2 and sl.shape[1] == 1
            self.sequence_lengths = sl.view((sl.shape[0],))
        else:
            self.sequence_lengths = None  # == full length for every row
        if training:
            return seq
        tags, _ = ops.crf_decode(seq, self.get_transitions(), self.sequence_lengths)
        return ops.one_hot(tags, self.output_dim)

    def _tags(self, y_true):
        y_true = nn.as_tensor(y_true)
        if y_true.ndim == 3:  # one-hot, as the reference expects (layers.py:93)
            return ops.argmax(y_true)
        return ops.cast(y_true, I32) if y_true.dtype != I32 else y_true

    @property
    def loss(self):
        def crf_loss(y_true, y_pred):
            return ops.crf_nll_loss(y_pred, self._tags(y_true), self.get_transitions(), self.sequence_lengths)
        return crf_loss

    def loss_sample_weights(self, mask_positive_classes, negative_weight):
        mask_t = Tensor.from_numpy(np.asarray(mask_positive_classes, np.float32), F32)

        def crf_loss(y_true, y_pred):
            y_true = nn.as_tensor(y_true)
            assert y_true.ndim == 3, "loss_sample_weights needs one-hot labels (layers.py:116)"
            B, T, K = y_true.shape
            w = Tensor((B,), F32)
            _lib.call("polus_crf_sample_weights", ops.cast(y_true, F32).ptr, mask_t.ptr, float(negative_weight), B, T, K,
                      w.ptr, device.stream())
            return ops.crf_nll_loss(y_pred, self._tags(y_true), self.get_transitions(), self.sequence_lengths, w)
        return crf_loss

    def compute_output_shape(self, input_shape):
        return tuple(input_shape[:2]) + (self.output_dim,)

    def get_config(self):
        return {"output_dim": self.output_dim, "sparse_target": self.sparse_target, "name": self.name}
