"""polus.models (reference polus/models.py:18-295): model utilities + the split-BERT encoder."""
import json
import os
import pickle
import sys
from functools import wraps

import numpy as np

from . import logger, nn, ops
from .nn import BertConfig, BertModel, BertOutput  # noqa: F401  (re-exported for user scripts)
from .tensor import BF16, I32, Tensor
from .utils import complex_json_deserializer, complex_json_serializer, flatten_dict, merge_dicts


def load_model(file_name_w_ext, change_config={}, external_module=None):
    """Rebuild a model from `<name>.cfg` (+ `.init`, weights) written by SavableModel.save
    (reference models.py:18-50).  Weights come from `<name>.h5` -- the reference's format, datasets weight0..N of the root
    group, read with h5py when it is installed and with the package's own HDF5 reader (h5lite) otherwise -- or from the
    `<name>.npz` files round 1 of this package wrote."""
    file_name = os.path.splitext(file_name_w_ext)[0]
    with open(file_name_w_ext, "r") as f:
        cfg = complex_json_deserializer(json.load(f))
    cfg["model"] = merge_dicts(cfg["model"], change_config)
    module = external_module if external_module is not None else sys.modules[__name__]
    model = getattr(module, cfg['func_name'])(**cfg)
    if os.path.exists(file_name + ".init"):
        with open(file_name + ".init", "rb") as f:
            args, kwargs = pickle.load(f)
        model.init_from_data(*args, **kwargs)
    if os.path.exists(file_name + ".h5"):
        try:
            import h5py
            with h5py.File(file_name + ".h5", 'r') as f:
                model.set_weights([f['weight' + str(i)][:] for i in range(len(f.keys()))])
        except ImportError:
            from . import h5lite
            model.set_weights(h5lite.read_weights(file_name + ".h5"))
    else:
        with np.load(file_name + ".npz") as z:
            model.set_weights([z[f"weight{i}"] for i in range(len(z.files))])
    return model


def resolve_activation(activation_name):
    return activation_name  # "mish" is a native activation code here (reference maps it to tfa)


def from_config(func):
    """Factory decorator: flattens the nested config, records func_name + config for save/load
    (reference models.py:60-82)."""
    @wraps(func)
    def function_wrapper(**kwargs):
        if "model" in kwargs and "activation" in kwargs["model"]:
            _activation = kwargs["model"]["activation"]
            kwargs["model"]["activation"] = resolve_activation(_activation)
        model = func(**flatten_dict(kwargs))
        kwargs['func_name'] = func.__name__
        if "model" in kwargs and "activation" in kwargs["model"]:
            kwargs["model"]["activation"] = _activation
        model._name = func.__name__
        model.savable_config = kwargs
        return model
    return function_wrapper


class PolusModel(nn.Model):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)

    def init_from_data(self, *args, **kwargs):
        self._init = (args, kwargs)
        return self(*args, **kwargs)

    def set_name(self, name):
        self._name = name


class SavableModel(PolusModel):
    def save(self, base_path=os.path.join(".polus_cache", "saved_models"), extension=""):
        """`<base>/<name><ext>.cfg` (complex JSON) + `.init` (pickle) + weights in get_weights() order
        (reference models.py:112-133): datasets weight0..N of `<name>.h5`, through h5py when it is installed, else through
        h5lite (same on-disk layout: version-0 superblock, symbol-table root group, contiguous datasets)."""
        os.makedirs(base_path, exist_ok=True)
        path = os.path.join(base_path, self.name + extension)
        with open(path + ".cfg", "w") as f:
            json.dump(complex_json_serializer(getattr(self, "savable_config", {"model": {}})), f)
        if hasattr(self, "_init"):
            with open(path + ".init", "wb") as f:
                pickle.dump(self._init, f)
        weights = self.get_weights()
        try:
            import h5py
            with h5py.File(path + ".h5", 'w') as f:
                for i, w in enumerate(weights):
                    f.create_dataset('weight' + str(i), data=w)
        except ImportError:
            from . import h5lite
            h5lite.write_weights(path + ".h5", weights)


class SequentialSavableModel(nn.Sequential, SavableModel):
    def __init__(self, layers, **kwargs):
        nn.Sequential.__init__(self, layers, **kwargs)


class PolusClassifier(SavableModel):
    def inference(self, x):
        """argmax(model(x), -1) as int32 (reference models.py:148-150)."""
        return ops.argmax(self(x), axis=-1)


class SequentialPolusClassifier(nn.Sequential, PolusClassifier):
    def __init__(self, layers, **kwargs):
        nn.Sequential.__init__(self, layers, **kwargs)


class TFBertSplited(PolusModel):
    """Trainable top-k BERT layers over precomputed hidden states (reference models.py:164-216).

    call(hidden_states [B,S,H], attention_mask [B,S] int32, training) -> last_hidden_state and
    pooler_output = h[:,0,:] (no pooler dense, models.py:216).  `training` reaches the layers as
    `run_in_training_mode & training` (models.py:213)."""

    def __init__(self, bert_layers, *args, run_in_training_mode=True, **kwargs):
        super().__init__(*args, **kwargs)
        self.layer = list(bert_layers)
        self.run_in_training_mode = run_in_training_mode

    def sublayers(self):
        return list(self.layer)

    def call(self, hidden_states, attention_mask=None, training=False):
        h = ops.cast(nn.as_tensor(hidden_states), BF16)
        mask = nn.as_tensor(attention_mask, I32) if attention_mask is not None else None
        for layer_module in self.layer:
            h = layer_module(h, attention_mask=mask, training=bool(self.run_in_training_mode and training))[0]
        B, S, H = h.shape
        return BertOutput(last_hidden_state=h, pooler_output=ops.gather_rows(ops.reshape(h, (B * S, H)), 0, S, B))


def split_bert_model(bert_model, index_layer, init_models=False, return_pre_bert_model=True, return_post_bert_model=True):
    """Cut a BertModel at `index_layer`: layers [index:] become a trainable TFBertSplited, layers
    [:index] stay in `bert_model` (reference models.py:242-295)."""
    assert return_pre_bert_model or return_post_bert_model
    n = bert_model.config.num_hidden_layers
    assert n > index_layer > -n and index_layer != 0
    encoder = bert_model.layers[0].encoder
    post_model = None
    if return_post_bert_model:
        post_model = TFBertSplited(encoder.layer[index_layer:])
    if return_pre_bert_model:
        del encoder.layer[index_layer:]
        bert_model.config.num_hidden_layers = len(encoder.layer)
    if return_pre_bert_model and return_post_bert_model:
        return bert_model, post_model
    return bert_model if return_pre_bert_model else post_model


def bert_model_from_checkpoint(bert_model_checkpoint):
    """Offline stand-in for `TFAutoModel.from_pretrained(checkpoint)` (reference models.py:225-229, data.py:526-530, which
    download from the HuggingFace hub).  `bert_model_checkpoint` may be
      * a BertModel (returned as is), a BertConfig or a dict of BertConfig fields (random init), or
      * a directory holding `config.json` and, optionally, weights: `weights.npz` (arrays weight0..N in get_weights()
        order, what SavableModel.save writes) or a HuggingFace snapshot's `model.safetensors` (imported with
        polus_b200.pretrained.load_hf_bert_weights; task heads such as `cls.*` are ignored).  `model_type` and
        `pad_token_id` of config.json are kept, so a RoBERTa, XLM-RoBERTa or CamemBERT snapshot gets its position ids."""
    if isinstance(bert_model_checkpoint, BertModel):
        return bert_model_checkpoint
    if isinstance(bert_model_checkpoint, BertConfig):
        return BertModel(bert_model_checkpoint)
    if isinstance(bert_model_checkpoint, dict):
        return BertModel(BertConfig(**bert_model_checkpoint))
    path = str(bert_model_checkpoint)
    if not os.path.isdir(path):
        raise ValueError(f"cannot resolve checkpoint {bert_model_checkpoint!r} offline: pass a BertModel, a BertConfig, a dict "
                         f"or a directory with config.json (+ weights.npz or model.safetensors)")
    with open(os.path.join(path, "config.json")) as f:
        bert_model = BertModel(BertConfig(**json.load(f)))
    npz, st = os.path.join(path, "weights.npz"), os.path.join(path, "model.safetensors")
    if os.path.exists(npz):
        with np.load(npz) as z:
            bert_model.set_weights([z[f"weight{i}"] for i in range(len(z.files))])
    elif os.path.exists(st):
        from .pretrained import load_hf_bert_weights
        load_hf_bert_weights(bert_model, st, strict=True)
    else:
        logger.warning(f"{path} holds no weights.npz / model.safetensors: the encoder keeps its random initialisation")
    return bert_model


def split_bert_model_from_checkpoint(bert_model_checkpoint, index_layer, init_models=False, return_pre_bert_model=True,
                                     return_post_bert_model=True):
    """The reference downloads a HF checkpoint here (models.py:225-229); offline resolution: bert_model_from_checkpoint."""
    bert_model = bert_model_from_checkpoint(bert_model_checkpoint)
    return split_bert_model(bert_model, index_layer, init_models=init_models,
                            return_pre_bert_model=return_pre_bert_model, return_post_bert_model=return_post_bert_model)
