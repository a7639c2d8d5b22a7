"""Masked-language-model training of BERT and RoBERTa-family encoders (HF BertForMaskedLM / RobertaForMaskedLM).

Continued MLM training on in-domain text is how BioBERT-style encoders are adapted before an NER or IR head is trained on
them.  The inputs follow Google's TF BERT pretraining data: `masked_lm_positions`, `masked_lm_ids` and
`masked_lm_weights`, each [B, P] with P = max_predictions_per_seq.  Only the P gathered rows per sequence are projected
onto the vocabulary, so every shape is static and the step captures into one CUDA graph.

    model = bert_mlm(vocab_size=..., ...)            # or BertMaskedLMModel(config), then load_hf_bert_weights
    ids, pos, lm_ids, lm_w = mask_tokens(ids, mask, vocab_size=..., mask_token_id=..., special_token_ids=...,
                                         max_predictions=20, rng=rng)
    x = {"input_ids": ids, "attention_mask": mask, "token_type_ids": tt, "masked_lm_positions": pos}
    y = {"masked_lm_ids": lm_ids, "masked_lm_weights": lm_w}
    ClassifierTrainer(model, optimizer, model.loss).train_step(x, y)
"""
import numpy as np

from . import nn, ops
from .models import BertConfig, BertModel, SavableModel, from_config
from .tensor import F32, I32


class BertMaskedLMModel(SavableModel):
    """BertModel(add_pooling_layer=False) + BertLMPredictionHead tied to its word embeddings.
    model(input_ids=..., attention_mask=..., token_type_ids=..., masked_lm_positions=..., training=...) -> bf16 logits
    [B*P, V] (ops.VocabLogits: rows padded to a multiple of 8 columns; generic ops refuse it, and model.loss overwrites
    it with its gradient).  get_weights(): the encoder's, then the head's (transform kernel and bias, LN gamma and beta, output bias)."""

    def __init__(self, config=None, name="bert_mlm", **kwargs):
        super().__init__(name=name)
        self.config = config or BertConfig(**kwargs)
        self.bert = BertModel(self.config, add_pooling_layer=False)
        self.cls = nn.BertLMPredictionHead(self.config, self.bert.bert.embeddings.word)
        self.last_predictions = None

    def sublayers(self):
        return [self.bert, self.cls]

    def call(self, input_ids=None, attention_mask=None, token_type_ids=None, masked_lm_positions=None, training=False,
             position_ids=None, **unused):
        if masked_lm_positions is None:
            raise ValueError("BertMaskedLMModel needs masked_lm_positions [B, P]")
        h = self.bert(input_ids=input_ids, attention_mask=attention_mask, token_type_ids=token_type_ids, training=training,
                      position_ids=position_ids)["last_hidden_state"]
        hm = ops.gather_positions(h, nn.as_tensor(masked_lm_positions, I32))
        return self.cls(hm, training=training)

    def loss(self, y, logits):
        """Weighted mean NLL of masked_lm_ids over the masked_lm_weights (HF's mean over labelled positions for 0/1
        weights).  The argmax of every row is kept in `last_predictions` (masked-token accuracy without another pass).
        Under data parallelism each replica normalises by its own sum of weights, as TF BERT's pretraining does per
        replica; the averaged gradient equals the whole batch's when the replicas' batches carry equal sums of weights
        (e.g. the same number of masked tokens per row)."""
        ids = nn.as_tensor(y["masked_lm_ids"], I32)
        w = nn.as_tensor(y["masked_lm_weights"], F32)
        loss, self.last_predictions = ops.vocab_cross_entropy(logits, ids.view((ids.size,)), w.view((w.size,)))
        return loss

    def inference(self, x):
        """Predicted token ids at the masked positions, int32 [B, P]; x is the dict the model is called with."""
        if not isinstance(x, dict) or "masked_lm_positions" not in x:
            raise ValueError("inference(x) takes the model's input dict, masked_lm_positions included")
        pos = nn.as_tensor(x["masked_lm_positions"], I32)
        return ops.vocab_argmax(self(**x)).view(tuple(pos.shape))


@from_config
def bert_mlm(**kwargs):
    cfg_keys = ("vocab_size", "hidden_size", "num_hidden_layers", "num_attention_heads", "intermediate_size",
                "max_position_embeddings", "type_vocab_size", "hidden_dropout_prob", "attention_probs_dropout_prob",
                "layer_norm_eps", "initializer_range", "model_type", "pad_token_id")
    return BertMaskedLMModel(BertConfig(**{k: kwargs[k] for k in cfg_keys if k in kwargs}))


def mask_tokens(input_ids, attention_mask, *, vocab_size, mask_token_id, special_token_ids, max_predictions,
                mlm_probability=0.15, rng):
    """Dynamic masking on the host, Google create_pretraining_data.py rules, vectorised over the batch.

    Candidates are attended tokens that are not in `special_token_ids`.  Each row masks
    n = min(max_predictions, max(1, round(mlm_probability * #candidates))) of them (0 without candidates), chosen
    uniformly without replacement and sorted; 80 % become mask_token_id, 10 % a uniform random id, 10 % stay.
    Returns (input_ids with the replacements, masked_lm_positions, masked_lm_ids, masked_lm_weights): int32 [B,S] and
    three [B, max_predictions] arrays (int32, int32, float32); slots beyond n hold position 0, id 0 and weight 0."""
    ids = np.asarray(input_ids)
    mask = np.asarray(attention_mask)
    if ids.ndim != 2 or mask.shape != ids.shape:
        raise ValueError(f"input_ids and attention_mask must both be [B, S], got {ids.shape} and {mask.shape}")
    P = int(max_predictions)
    if P < 1:
        raise ValueError(f"max_predictions must be >= 1, got {max_predictions}")
    if not 0.0 < mlm_probability <= 1.0:
        raise ValueError(f"mlm_probability must be in (0, 1], got {mlm_probability}")
    B, S = ids.shape
    cand = (mask != 0) & ~np.isin(ids, np.asarray(list(special_token_ids), dtype=ids.dtype))
    n_cand = cand.sum(axis=1)
    n = np.minimum(P, np.maximum(1, np.rint(mlm_probability * n_cand).astype(np.int64)))
    n = np.where(n_cand == 0, 0, np.minimum(n, n_cand))
    keys = np.where(cand, rng.random((B, S)), 2.0)
    order = np.argsort(keys, axis=1, kind="stable")[:, :P]          # candidates in random order first
    if order.shape[1] < P:
        order = np.pad(order, ((0, 0), (0, P - order.shape[1])))
    take = np.arange(P)[None, :] < n[:, None]
    pos = np.sort(np.where(take, order, S), axis=1)                  # chosen positions ascending, unused slots last
    take = pos < S
    pos = np.where(take, pos, 0).astype(np.int32)
    rows = np.arange(B)[:, None]
    labels = np.where(take, ids[rows, pos], 0).astype(np.int32)
    r = rng.random((B, P))
    random_ids = rng.integers(0, vocab_size, (B, P))
    repl = np.where(r < 0.8, mask_token_id, np.where(r < 0.9, random_ids, labels))
    out = ids.astype(np.int32, copy=True)
    bsel, psel = np.nonzero(take)
    out[bsel, pos[bsel, psel]] = repl[bsel, psel]
    return out, pos, labels, take.astype(np.float32)
