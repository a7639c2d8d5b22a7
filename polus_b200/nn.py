"""Keras-shaped layers and models on top of polus_b200.ops.

The reference builds its models from tf.keras layers and HuggingFace TF BERT blocks
(polus/models.py:135-216, polus/ner/models.py:26-67, tutorials/classifier_example.py:44-48).  These
classes keep the same names, constructor arguments and call convention (`model(x, training=True)`,
`.trainable_weights`, `.get_weights()/.set_weights()` in Keras order) so user scripts read the same,
while every computation is a libpolus_b200.so kernel.
"""
import math

import numpy as np

from . import ops
from .tensor import BF16, F32, I32, Param, Tensor

_seed_state = {"rng": np.random.Generator(np.random.PCG64(42))}


def set_initializer_seed(seed):
    """Deterministic host-side weight init (numpy PCG64) -- the same arrays are handed to the oracle
    in parity tests, which is how 'same random-init weights' is achieved without TF."""
    _seed_state["rng"] = np.random.Generator(np.random.PCG64(int(seed)))


def _rng():
    return _seed_state["rng"]


def glorot_uniform(shape):
    fan_in, fan_out = shape[0], shape[-1]
    limit = math.sqrt(6.0 / (fan_in + fan_out))
    return _rng().uniform(-limit, limit, size=shape).astype(np.float32)


def truncated_normal(shape, stddev=0.02):
    """tf.keras TruncatedNormal (HF get_initializer(0.02)): resample beyond 2 sigma."""
    x = _rng().standard_normal(size=shape)
    bad = np.abs(x) > 2.0
    while bad.any():
        x[bad] = _rng().standard_normal(size=int(bad.sum()))
        bad = np.abs(x) > 2.0
    return (x * stddev).astype(np.float32)


def as_tensor(x, dtype=None):
    if isinstance(x, Tensor):
        return x
    return Tensor.from_numpy(np.asarray(x), dtype)


# ------------------------------------------------------------------------------------------------
class Layer:
    _counter = {}

    def __init__(self, name=None, **kwargs):
        cls = self.__class__.__name__.lower()
        n = Layer._counter.get(cls, 0)
        Layer._counter[cls] = n + 1
        self._name = name or (cls if n == 0 else f"{cls}_{n}")
        self.built = False
        self.trainable = True
        self._params = []
        self._input_shape = kwargs.get("input_shape")

    @property
    def name(self):
        return self._name

    def add_weight(self, name, value, decay=True):
        p = Param(value, name=f"{self._name}/{name}", decay=decay)
        self._params.append(p)
        return p

    def build(self, input_shape):
        pass

    def compute_output_shape(self, input_shape):
        return tuple(input_shape)

    def _maybe_build(self, x):
        if not self.built:
            self.build(x.shape if isinstance(x, Tensor) else None)
            self.built = True

    def sublayers(self):
        return []

    @property
    def weights(self):
        out = list(self._params)
        for l in self.sublayers():
            out.extend(l.weights)
        return out

    @property
    def trainable_weights(self):
        if not self.trainable:
            return []
        out = list(self._params)
        for l in self.sublayers():
            out.extend(l.trainable_weights)
        return out

    @property
    def trainable_variables(self):
        return self.trainable_weights

    def get_weights(self):
        return [w.numpy() for w in self.weights]

    def set_weights(self, values):
        ws = self.weights
        assert len(ws) == len(values), f"{self.name}: expected {len(ws)} arrays, got {len(values)}"
        for w, v in zip(ws, values):
            w.assign(v)

    def call(self, x, training=False):
        raise NotImplementedError

    def __call__(self, *args, training=False, **kwargs):
        if args:
            self._maybe_build(args[0])
        else:
            self._maybe_build(next(iter(kwargs.values())))
        return self.call(*args, training=training, **kwargs)


class Dense(Layer):
    """tf.keras.layers.Dense: kernel [in, units] glorot_uniform, zero bias."""

    def __init__(self, units, activation=None, use_bias=True, input_shape=None, kernel_initializer="glorot_uniform",
                 name=None, **kwargs):
        super().__init__(name=name, input_shape=input_shape)
        self.units = int(units)
        self.activation = activation
        self.use_bias = use_bias
        self.kernel_initializer = kernel_initializer
        self.kernel = self.bias = None

    def build(self, input_shape):
        fan_in = int(input_shape[-1])
        if self.kernel_initializer == "glorot_uniform":
            k = glorot_uniform((fan_in, self.units))
        elif self.kernel_initializer == "bert":
            k = truncated_normal((fan_in, self.units))
        else:
            k = np.asarray(self.kernel_initializer((fan_in, self.units)), np.float32)
        self.kernel = self.add_weight("kernel", k)
        if self.use_bias:
            self.bias = self.add_weight("bias", np.zeros(self.units, np.float32), decay=False)

    def compute_output_shape(self, input_shape):
        return tuple(input_shape[:-1]) + (self.units,)

    def call(self, x, training=False):
        return ops.linear(as_tensor(x), self.kernel, self.bias, self.activation)


class Dropout(Layer):
    def __init__(self, rate, input_shape=None, name=None, **kwargs):
        super().__init__(name=name, input_shape=input_shape)
        self.rate = float(rate)

    def call(self, x, training=False):
        return ops.dropout(as_tensor(x), self.rate) if training and self.rate > 0 else as_tensor(x)


class Flatten(Layer):
    def __init__(self, input_shape=None, name=None, **kwargs):
        super().__init__(name=name, input_shape=input_shape)

    def compute_output_shape(self, input_shape):
        n = 1
        for s in input_shape[1:]:
            n *= s
        return (input_shape[0], n)

    def call(self, x, training=False):
        x = as_tensor(x)
        return ops.reshape(x, (x.shape[0], -1))


class Model(Layer):
    """Minimal tf.keras.Model: layers discovered from attributes in definition order."""

    def __init__(self, *args, name=None, **kwargs):
        super().__init__(name=name)

    def sublayers(self):
        seen, out = set(), []
        for v in self.__dict__.values():
            items = v if isinstance(v, (list, tuple)) else [v]
            for it in items:
                if isinstance(it, Layer) and id(it) not in seen and it is not self:
                    seen.add(id(it))
                    out.append(it)
        return out

    @property
    def layers(self):
        return self.sublayers()

    def _maybe_build(self, x):
        self.built = True


class Sequential(Model):
    def __init__(self, layers=None, name=None, **kwargs):
        super().__init__(name=name)
        self._layers = list(layers or [])
        # Keras builds a Sequential eagerly when its first layer declares input_shape, so
        # model.trainable_weights is populated before the first call (the reference trainer reads it
        # at construction, polus/training.py:85).
        if self._layers and self._layers[0]._input_shape is not None:
            shape = (None,) + tuple(self._layers[0]._input_shape)
            for l in self._layers:
                if not l.built:
                    l.build(shape)
                    l.built = True
                shape = l.compute_output_shape(shape)

    def add(self, layer):
        self._layers.append(layer)

    def sublayers(self):
        return list(self._layers)

    def call(self, x, training=False):
        x = as_tensor(x)
        for l in self._layers:
            x = l(x, training=training)
        return x


# ------------------------------------------------------------------------------------------------
# BERT blocks (HF TFBertEmbeddings / TFBertLayer / TFBertPooler semantics; see SURVEY.md §8a)
# ------------------------------------------------------------------------------------------------
class BertConfig:
    def __init__(self, vocab_size=30522, hidden_size=768, num_hidden_layers=12, num_attention_heads=12,
                 intermediate_size=3072, max_position_embeddings=512, type_vocab_size=2, hidden_dropout_prob=0.1,
                 attention_probs_dropout_prob=0.1, layer_norm_eps=1e-12, initializer_range=0.02, model_type="bert",
                 pad_token_id=0, **kwargs):
        self.model_type = model_type
        self.pad_token_id = pad_token_id
        self.vocab_size = vocab_size
        self.hidden_size = hidden_size
        self.num_hidden_layers = num_hidden_layers
        self.num_attention_heads = num_attention_heads
        self.intermediate_size = intermediate_size
        self.max_position_embeddings = max_position_embeddings
        self.type_vocab_size = type_vocab_size
        self.hidden_dropout_prob = hidden_dropout_prob
        self.attention_probs_dropout_prob = attention_probs_dropout_prob
        self.layer_norm_eps = layer_norm_eps
        self.initializer_range = initializer_range
        self._name_or_path = kwargs.get("name_or_path", "random-init")

    @property
    def roberta_positions(self):
        """RoBERTa-family checkpoints number positions from pad_token_id + 1 and send pad tokens to pad_token_id."""
        return self.model_type in ROBERTA_MODEL_TYPES


ROBERTA_MODEL_TYPES = ("roberta", "xlm-roberta", "camembert")


class BertEmbeddings(Layer):
    def __init__(self, config, name="embeddings"):
        super().__init__(name=name)
        c = self.config = config
        sd = c.initializer_range
        self.word = self.add_weight("word_embeddings/weight", truncated_normal((c.vocab_size, c.hidden_size), sd))
        self.token_type = self.add_weight("token_type_embeddings/embeddings", truncated_normal((c.type_vocab_size, c.hidden_size), sd))
        self.position = self.add_weight("position_embeddings/embeddings", truncated_normal((c.max_position_embeddings, c.hidden_size), sd))
        self.ln_gamma = self.add_weight("LayerNorm/gamma", np.ones(c.hidden_size, np.float32), decay=False)
        self.ln_beta = self.add_weight("LayerNorm/beta", np.zeros(c.hidden_size, np.float32), decay=False)
        self.built = True

    def call(self, input_ids, token_type_ids=None, training=False, position_ids=None):
        """position_ids: int32 [B,S] (HF semantics).  Without them a BERT config uses position s for token s and a
        RoBERTa-family config derives them from input_ids on the device (pad tokens -> pad_token_id)."""
        c = self.config
        ids = as_tensor(input_ids, I32)
        tt = as_tensor(token_type_ids, I32) if token_type_ids is not None else None
        if position_ids is not None:
            pos_ids = as_tensor(position_ids, I32)
        elif c.roberta_positions:
            S = ids.shape[1]
            if S + c.pad_token_id + 1 > c.max_position_embeddings:
                raise ValueError(f"sequence length {S} needs position ids up to {S + c.pad_token_id} (pad_token_id "
                                 f"{c.pad_token_id} + 1 + S - 1), beyond the {c.max_position_embeddings} learned positions")
            pos_ids = ops.position_ids_from_input_ids(ids, c.pad_token_id)
        else:
            pos_ids = None
        p = c.hidden_dropout_prob if training else 0.0
        return ops.embed_layernorm(ids, tt, self.word, self.position, self.token_type, self.ln_gamma, self.ln_beta,
                                   c.layer_norm_eps, p, position_ids=pos_ids)


class BertLayer(Layer):
    """One post-LN transformer block.  Parameters (creation order): Wqkv [H,3H] (q|k|v), bqkv, Wo, bo,
    LN1 gamma/beta, W1 [H,I], b1, W2 [I,H], b2, LN2 gamma/beta."""

    def __init__(self, config, name=None):
        super().__init__(name=name)
        c = self.config = config
        H, I, sd = c.hidden_size, c.intermediate_size, c.initializer_range
        assert H % c.num_attention_heads == 0
        qkv = np.concatenate([truncated_normal((H, H), sd) for _ in range(3)], axis=1)
        self.Wqkv = self.add_weight("attention/self/qkv/kernel", qkv)
        self.bqkv = self.add_weight("attention/self/qkv/bias", np.zeros(3 * H, np.float32), decay=False)
        self.Wo = self.add_weight("attention/output/dense/kernel", truncated_normal((H, H), sd))
        self.bo = self.add_weight("attention/output/dense/bias", np.zeros(H, np.float32), decay=False)
        self.ln1_g = self.add_weight("attention/output/LayerNorm/gamma", np.ones(H, np.float32), decay=False)
        self.ln1_b = self.add_weight("attention/output/LayerNorm/beta", np.zeros(H, np.float32), decay=False)
        self.W1 = self.add_weight("intermediate/dense/kernel", truncated_normal((H, I), sd))
        self.b1 = self.add_weight("intermediate/dense/bias", np.zeros(I, np.float32), decay=False)
        self.W2 = self.add_weight("output/dense/kernel", truncated_normal((I, H), sd))
        self.b2 = self.add_weight("output/dense/bias", np.zeros(H, np.float32), decay=False)
        self.ln2_g = self.add_weight("output/LayerNorm/gamma", np.ones(H, np.float32), decay=False)
        self.ln2_b = self.add_weight("output/LayerNorm/beta", np.zeros(H, np.float32), decay=False)
        self.built = True

    def call(self, hidden_states, attention_mask=None, training=False, **unused):
        """attention_mask: int32 [B,S] (1 = attend).  The additive (1-m)*-10000 form of
        polus/models.py:175-195 is applied inside the softmax kernel."""
        c = self.config
        x = ops.cast(as_tensor(hidden_states), BF16)
        pa = c.attention_probs_dropout_prob if training else 0.0
        ph = c.hidden_dropout_prob if training else 0.0
        # fused attention backward also sums the QKV bias gradient from the dQ|dK|dV tiles it holds in shared memory
        fuse_b = ops.attention_takes_bias_grad(x.shape[-2], c.hidden_size // c.num_attention_heads)
        qkv = ops.linear(x, self.Wqkv, self.bqkv, defer_bias_grad=fuse_b)
        ctx = ops.attention(qkv, attention_mask, c.num_attention_heads, pa, qkv_bias=self.bqkv if fuse_b else None)
        # the two Dense layers feeding a LayerNorm leave their bias gradient to the LayerNorm backward kernel
        ao = ops.linear(ctx, self.Wo, self.bo, defer_bias_grad=True)
        h1 = ops.layernorm_residual(ao, x, self.ln1_g, self.ln1_b, c.layer_norm_eps, ph, x_bias=self.bo)
        a = ops.linear(h1, self.W1, self.b1, "gelu")
        o = ops.linear(a, self.W2, self.b2, defer_bias_grad=True)
        y = ops.layernorm_residual(o, h1, self.ln2_g, self.ln2_b, c.layer_norm_eps, ph, x_bias=self.b2)
        return (y,)

    # Keras/HF variable order: query k,b; key k,b; value k,b; attn-out k,b; LN g,b; inter k,b; out k,b; LN g,b
    def get_weights(self):
        H = self.config.hidden_size
        Wqkv, bqkv = self.Wqkv.numpy(), self.bqkv.numpy()
        out = []
        for i in range(3):
            out += [Wqkv[:, i * H:(i + 1) * H].copy(), bqkv[i * H:(i + 1) * H].copy()]
        out += [w.numpy() for w in (self.Wo, self.bo, self.ln1_g, self.ln1_b, self.W1, self.b1, self.W2, self.b2,
                                    self.ln2_g, self.ln2_b)]
        return out

    def set_weights(self, values):
        assert len(values) == 16, f"BertLayer expects 16 arrays (Keras order), got {len(values)}"
        self.Wqkv.assign(np.concatenate([values[0], values[2], values[4]], axis=1))
        self.bqkv.assign(np.concatenate([values[1], values[3], values[5]]))
        for w, v in zip((self.Wo, self.bo, self.ln1_g, self.ln1_b, self.W1, self.b1, self.W2, self.b2, self.ln2_g,
                         self.ln2_b), values[6:]):
            w.assign(v)


class BertPooler(Layer):
    def __init__(self, config, name="pooler"):
        super().__init__(name=name)
        self.dense = Dense(config.hidden_size, activation="tanh", kernel_initializer="bert", name="pooler/dense")

    def sublayers(self):
        return [self.dense]

    def call(self, hidden_states, training=False):
        B, S, H = hidden_states.shape
        first = ops.gather_rows(ops.reshape(hidden_states, (B * S, H)), 0, S, B)
        return self.dense(first, training=training)


class BertOutput(dict):
    """dict + attribute access, like HF's TFBaseModelOutputWithPooling (polus/models.py:215-216)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __getitem__(self, k):
        if isinstance(k, int):
            return list(self.values())[k]
        return dict.__getitem__(self, k)


class BertEncoder(Layer):
    def __init__(self, config, name="encoder"):
        super().__init__(name=name)
        self.layer = [BertLayer(config, name=f"encoder/layer_._{i}") for i in range(config.num_hidden_layers)]
        self.built = True

    def sublayers(self):
        return list(self.layer)


class BertMainLayer(Layer):
    def __init__(self, config, add_pooling_layer=True, name="bert"):
        super().__init__(name=name)
        self.config = config
        self.embeddings = BertEmbeddings(config)
        self.encoder = BertEncoder(config)
        self.pooler = BertPooler(config) if add_pooling_layer else None
        self.built = True

    def sublayers(self):
        return [self.embeddings, self.encoder] + ([self.pooler] if self.pooler else [])


class BertModel(Model):
    """Stand-in for transformers.TFBertModel (random init; pretrained import is a §8f 'next' row).
    `model.layers[0].encoder.layer` is the list polus/models.py:260-264 slices."""

    def __init__(self, config=None, add_pooling_layer=True, name="tf_bert_model", **kwargs):
        super().__init__(name=name)
        self.config = config or BertConfig(**kwargs)
        self.bert = BertMainLayer(self.config, add_pooling_layer)

    def sublayers(self):
        return [self.bert]

    def call(self, input_ids=None, attention_mask=None, token_type_ids=None, training=False, position_ids=None, **unused):
        ids = as_tensor(input_ids, I32)
        mask = as_tensor(attention_mask, I32) if attention_mask is not None else None
        h = self.bert.embeddings(ids, token_type_ids, training=training, position_ids=position_ids)
        for layer in self.bert.encoder.layer:
            h = layer(h, attention_mask=mask, training=training)[0]
        out = BertOutput(last_hidden_state=h)
        if self.bert.pooler is not None:
            out["pooler_output"] = self.bert.pooler(h, training=training)
        else:
            B, S, H = h.shape
            out["pooler_output"] = ops.gather_rows(ops.reshape(h, (B * S, H)), 0, S, B)
        return out


class BertLMPredictionHead(Layer):
    """HF `cls.predictions` (BERT) / `lm_head` (RoBERTa family): Dense(H, H, gelu) -> LayerNorm -> logits against the TIED
    word-embedding table plus an output bias [V].  `word_embeddings` is the encoder's word Param, not a copy: the decoder
    reads its bf16 shadow and adds its gradient into the same fp32 slice as the embedding lookup.
    Parameters (Keras order): transform kernel [H,H], transform bias, LN gamma, LN beta, output bias [V]."""

    def __init__(self, config, word_embeddings, name="cls/predictions"):
        super().__init__(name=name)
        c = self.config = config
        H, V = c.hidden_size, c.vocab_size
        assert tuple(word_embeddings.shape) == (V, H), "the decoder is tied to a [vocab_size, hidden_size] table"
        self.word = word_embeddings
        self.kernel = self.add_weight("transform/dense/kernel", truncated_normal((H, H), c.initializer_range))
        self.dense_bias = self.add_weight("transform/dense/bias", np.zeros(H, np.float32), decay=False)
        self.ln_gamma = self.add_weight("transform/LayerNorm/gamma", np.ones(H, np.float32), decay=False)
        self.ln_beta = self.add_weight("transform/LayerNorm/beta", np.zeros(H, np.float32), decay=False)
        self.bias = self.add_weight("bias", np.zeros(V, np.float32), decay=False)
        self.built = True

    def call(self, hidden_states, training=False):
        """hidden_states [R, H] (the gathered masked positions) -> bf16 logits [R, V] (ops.VocabLogits)."""
        t = ops.linear(as_tensor(hidden_states), self.kernel, self.dense_bias, "gelu")
        t = ops.layernorm_residual(t, None, self.ln_gamma, self.ln_beta, self.config.layer_norm_eps)
        return ops.vocab_projection(t, self.word, self.bias)
