"""Import of HuggingFace BERT checkpoints into polus_b200.nn.BertModel (SURVEY.md §8f rank 3).

The reference gets pretrained encoders from `TFAutoModel.from_pretrained(checkpoint)` (polus/data.py:526-530,
polus/models.py:225-229).  Here the weights come from a HuggingFace *state dict* -- a `.safetensors` file, a `.npz`, or a
mapping name -> array -- with the torch naming (`bert.` prefix optional; RoBERTa, XLM-RoBERTa and CamemBERT checkpoints
use the same names under a `roberta.` prefix).  A model with a masked-LM head (polus_b200.mlm.BertMaskedLMModel) also
takes the head: `cls.predictions.{transform.dense, transform.LayerNorm, bias}` (BERT) or `lm_head.{dense, layer_norm,
bias}` (RoBERTa family); the decoder is tied to the word embeddings.  For any other model the heads are left unused:

    embeddings.word_embeddings.weight            [V, H]          encoder.layer.N.attention.output.dense.weight  [H, H]
    embeddings.position_embeddings.weight        [P, H]          encoder.layer.N.attention.output.LayerNorm.*
    embeddings.token_type_embeddings.weight      [T, H]          encoder.layer.N.intermediate.dense.weight      [I, H]
    embeddings.LayerNorm.{weight,bias}                           encoder.layer.N.output.dense.weight            [H, I]
    encoder.layer.N.attention.self.{query,key,value}.{weight [H, H], bias}    encoder.layer.N.output.LayerNorm.*
    pooler.dense.{weight,bias}

torch `Linear.weight` is [out, in]; the kernels here keep the Keras layout [in, out] and fuse q|k|v into one [H, 3H]
variable (DESIGN.md §3), so every dense weight is transposed and the three projections are concatenated.
"""
import numpy as np


def _load_state(source):
    if isinstance(source, dict):
        return {k: np.asarray(v) for k, v in source.items()}
    path = str(source)
    if path.endswith(".safetensors"):
        from safetensors.numpy import load_file
        return load_file(path)
    if path.endswith(".npz"):
        with np.load(path) as z:
            return {k: z[k] for k in z.files}
    raise ValueError(f"unsupported checkpoint {path!r}: expected .safetensors, .npz or a dict")


def load_hf_bert_weights(model, source, strict=True):
    """Copy a HuggingFace BERT or RoBERTa-family state dict into `model` (a polus_b200.nn.BertModel, its BertMainLayer, or
    a BertMaskedLMModel, whose head is filled too; a checkpoint without a head raises KeyError then, unless
    strict=False, which keeps the model's freshly initialised head -- e.g. MLM training from an encoder-only snapshot).  Returns the list of state-dict keys that were not used (heads such
    as `cls.*` or `lm_head.*` of an encoder-only model)."""
    state = _load_state(source)
    strip = lambda k: k.split(".", 1)[1] if k.startswith(("bert.", "roberta.")) else k
    # LayerNorm.gamma / .beta: the TF-era names, which HF still reads and, after reading them, writes back
    legacy = lambda k: k.replace("LayerNorm.gamma", "LayerNorm.weight").replace("LayerNorm.beta", "LayerNorm.bias")
    state = {legacy(strip(k)): v for k, v in state.items()}
    used = set()

    def get(name):
        if name not in state:
            raise KeyError(f"checkpoint has no tensor {name!r}")
        used.add(name)
        return np.asarray(state[name], dtype=np.float32)

    head = getattr(model, "cls", None)
    main = model.bert if head is not None else model
    main = getattr(main, "bert", main)
    cfg = main.config
    emb = main.embeddings
    for param, name in ((emb.word, "embeddings.word_embeddings.weight"), (emb.position, "embeddings.position_embeddings.weight"),
                        (emb.token_type, "embeddings.token_type_embeddings.weight"), (emb.ln_gamma, "embeddings.LayerNorm.weight"),
                        (emb.ln_beta, "embeddings.LayerNorm.bias")):
        value = get(name)
        if value.shape != tuple(param.shape):
            raise ValueError(f"{name}: checkpoint shape {value.shape} != model shape {tuple(param.shape)} "
                             f"(vocab/positions/hidden of the BertConfig must match the checkpoint)")
        param.assign(value)
    for i, layer in enumerate(main.encoder.layer):
        p = f"encoder.layer.{i}."
        qkv_w = np.concatenate([get(p + f"attention.self.{n}.weight").T for n in ("query", "key", "value")], axis=1)
        qkv_b = np.concatenate([get(p + f"attention.self.{n}.bias") for n in ("query", "key", "value")])
        pairs = ((layer.Wqkv, qkv_w), (layer.bqkv, qkv_b),
                 (layer.Wo, get(p + "attention.output.dense.weight").T), (layer.bo, get(p + "attention.output.dense.bias")),
                 (layer.ln1_g, get(p + "attention.output.LayerNorm.weight")), (layer.ln1_b, get(p + "attention.output.LayerNorm.bias")),
                 (layer.W1, get(p + "intermediate.dense.weight").T), (layer.b1, get(p + "intermediate.dense.bias")),
                 (layer.W2, get(p + "output.dense.weight").T), (layer.b2, get(p + "output.dense.bias")),
                 (layer.ln2_g, get(p + "output.LayerNorm.weight")), (layer.ln2_b, get(p + "output.LayerNorm.bias")))
        for param, value in pairs:
            if value.shape != tuple(param.shape):
                raise ValueError(f"layer {i}: checkpoint shape {value.shape} != model shape {tuple(param.shape)}")
            param.assign(np.ascontiguousarray(value))
    if main.pooler is not None and "pooler.dense.weight" in state:
        if main.pooler.dense.kernel is None:
            main.pooler.dense.build((None, main.config.hidden_size))
            main.pooler.dense.built = True
        main.pooler.dense.kernel.assign(np.ascontiguousarray(get("pooler.dense.weight").T))
        main.pooler.dense.bias.assign(get("pooler.dense.bias"))
    if head is not None and (strict or "lm_head.bias" in state or "cls.predictions.bias" in state):
        _load_head(head, state, get, used)   # strict=False and no head in the checkpoint: the head keeps its init
    unused = sorted(k for k in state if k not in used and not k.endswith("position_ids"))
    if strict and any(k.startswith(("embeddings.", "encoder.")) for k in unused):
        raise ValueError(f"checkpoint tensors without a destination (more layers than the model?): {unused[:5]}")
    del cfg
    return unused


# masked-LM head names: (transform dense, transform LayerNorm, output bias, decoder) per family
_HEAD_NAMES = {"bert": ("cls.predictions.transform.dense", "cls.predictions.transform.LayerNorm", "cls.predictions.bias",
                        "cls.predictions.decoder"),
               "roberta": ("lm_head.dense", "lm_head.layer_norm", "lm_head.bias", "lm_head.decoder")}


def _head_family(config):
    return "roberta" if config.roberta_positions else "bert"


def _load_head(head, state, get, used):
    if "lm_head.bias" in state:
        dense, ln, bias, dec = _HEAD_NAMES["roberta"]
    elif "cls.predictions.bias" in state:
        dense, ln, bias, dec = _HEAD_NAMES["bert"]
    else:
        raise KeyError("checkpoint has no masked-LM head (cls.predictions.* or lm_head.*)")
    for param, value in ((head.kernel, get(dense + ".weight").T), (head.dense_bias, get(dense + ".bias")),
                         (head.ln_gamma, get(ln + ".weight")), (head.ln_beta, get(ln + ".bias")), (head.bias, get(bias))):
        if value.shape != tuple(param.shape):
            raise ValueError(f"masked-LM head: checkpoint shape {value.shape} != model shape {tuple(param.shape)}")
        param.assign(np.ascontiguousarray(value))
    # HF ties decoder.weight to the word embeddings and decoder.bias to the output bias; save_pretrained omits both
    for name, tied in ((dec + ".weight", "embeddings.word_embeddings.weight"), (dec + ".bias", bias)):
        if name in state:
            if not np.array_equal(get(name), get(tied)):
                raise ValueError(f"{name} differs from {tied}: untied masked-LM decoders are not supported")


def export_hf_bert_weights(model):
    """The inverse mapping: a HuggingFace-named state dict (numpy) of `model` -- what `safetensors.numpy.save_file` or
    `torch.load_state_dict` expect.  A BertMaskedLMModel's head is emitted under its family's names (without the tied
    decoder, as HF's save_pretrained writes it)."""
    head = getattr(model, "cls", None)
    if head is not None:
        out = export_hf_bert_weights(model.bert)
        dense, ln, bias, _ = _HEAD_NAMES[_head_family(head.config)]
        out.update({dense + ".weight": np.ascontiguousarray(head.kernel.numpy().T), dense + ".bias": head.dense_bias.numpy(),
                    ln + ".weight": head.ln_gamma.numpy(), ln + ".bias": head.ln_beta.numpy(), bias: head.bias.numpy()})
        return out
    main = getattr(model, "bert", model)
    emb = main.embeddings
    H = main.config.hidden_size
    out = {"embeddings.word_embeddings.weight": emb.word.numpy(), "embeddings.position_embeddings.weight": emb.position.numpy(),
           "embeddings.token_type_embeddings.weight": emb.token_type.numpy(), "embeddings.LayerNorm.weight": emb.ln_gamma.numpy(),
           "embeddings.LayerNorm.bias": emb.ln_beta.numpy()}
    for i, layer in enumerate(main.encoder.layer):
        p = f"encoder.layer.{i}."
        w, b = layer.Wqkv.numpy(), layer.bqkv.numpy()
        for j, n in enumerate(("query", "key", "value")):
            out[p + f"attention.self.{n}.weight"] = np.ascontiguousarray(w[:, j * H:(j + 1) * H].T)
            out[p + f"attention.self.{n}.bias"] = b[j * H:(j + 1) * H].copy()
        out[p + "attention.output.dense.weight"] = np.ascontiguousarray(layer.Wo.numpy().T)
        out[p + "attention.output.dense.bias"] = layer.bo.numpy()
        out[p + "attention.output.LayerNorm.weight"] = layer.ln1_g.numpy()
        out[p + "attention.output.LayerNorm.bias"] = layer.ln1_b.numpy()
        out[p + "intermediate.dense.weight"] = np.ascontiguousarray(layer.W1.numpy().T)
        out[p + "intermediate.dense.bias"] = layer.b1.numpy()
        out[p + "output.dense.weight"] = np.ascontiguousarray(layer.W2.numpy().T)
        out[p + "output.dense.bias"] = layer.b2.numpy()
        out[p + "output.LayerNorm.weight"] = layer.ln2_g.numpy()
        out[p + "output.LayerNorm.bias"] = layer.ln2_b.numpy()
    if main.pooler is not None:
        out["pooler.dense.weight"] = np.ascontiguousarray(main.pooler.dense.kernel.numpy().T)
        out["pooler.dense.bias"] = main.pooler.dense.bias.numpy()
    return out


def save_hf_checkpoint(model, directory):
    """Write a HuggingFace snapshot of `model` (a BertModel or a BertMaskedLMModel): `config.json` and `model.safetensors`
    with the family's prefix (`bert.` or `roberta.`).  The directory loads back through
    polus_b200.models.bert_model_from_checkpoint (e.g. as the encoder of an NER model) and through HF's
    BertForMaskedLM / RobertaForMaskedLM.from_pretrained."""
    import json
    import os
    from safetensors.numpy import save_file
    head = getattr(model, "cls", None)
    main = getattr(model.bert if head is not None else model, "bert", model)
    c = main.config
    family = _head_family(c)
    prefix = "roberta." if family == "roberta" else "bert."
    state = {}
    for k, v in export_hf_bert_weights(model).items():
        key = k if k.startswith(("cls.", "lm_head.")) else prefix + k
        state[key] = np.ascontiguousarray(v, dtype=np.float32)
    arch = {"bert": "BertForMaskedLM" if head is not None else "BertModel",
            "roberta": "RobertaForMaskedLM" if head is not None else "RobertaModel"}[family]
    config = {"architectures": [arch], "model_type": c.model_type, "vocab_size": c.vocab_size,
              "hidden_size": c.hidden_size, "num_hidden_layers": c.num_hidden_layers,
              "num_attention_heads": c.num_attention_heads, "intermediate_size": c.intermediate_size,
              "hidden_act": "gelu", "hidden_dropout_prob": c.hidden_dropout_prob,
              "attention_probs_dropout_prob": c.attention_probs_dropout_prob,
              "max_position_embeddings": c.max_position_embeddings, "type_vocab_size": c.type_vocab_size,
              "initializer_range": c.initializer_range, "layer_norm_eps": c.layer_norm_eps, "pad_token_id": c.pad_token_id,
              "tie_word_embeddings": True}
    os.makedirs(directory, exist_ok=True)
    with open(os.path.join(directory, "config.json"), "w") as f:
        json.dump(config, f, indent=2)
    save_file(state, os.path.join(directory, "model.safetensors"))
