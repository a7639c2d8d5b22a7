"""polus.ner.models (reference polus/ner/models.py:7-67) + the assembled BERT-NER model of BASELINE.json."""
from .. import nn, ops
from ..layers import CRF
from ..models import BertConfig, BertModel, SavableModel, from_config, resolve_activation
from ..tensor import I32


class NERBertModel(SavableModel):
    def inference(self, x):
        """argmax over the CRF layer's one-hot Viterbi output = the Viterbi tags, int32 [B,S]
        (reference ner/models.py:12-15)."""
        return ops.argmax(self(x), axis=-1)


class SequentialNERBertModel(nn.Sequential, NERBertModel):
    def __init__(self, layers, **kwargs):
        nn.Sequential.__init__(self, layers, **kwargs)


@from_config
def baselineNER_MLP_CRF(sequence_length=256, output_classes=3, hidden_space=128, activation="swish", **kwargs):
    """Dense(768->hidden, act) -> Dense(hidden->K) -> CRF over 768-d embeddings (ner/models.py:26-44)."""
    crf_layer = CRF(output_classes)
    model = SequentialNERBertModel([
        nn.Dense(hidden_space, input_shape=(sequence_length, 768), activation=activation),
        nn.Dense(output_classes),
        crf_layer,
    ])
    model.loss = crf_layer.loss
    model.loss_sample_weights = crf_layer.loss_sample_weights
    return model


@from_config
def baselineNER_MLP_Dropout_CRF(sequence_length=256, output_classes=3, hidden_space=128, droupout_p=0.1,
                                activation="swish", **kwargs):
    """Dropout(p) -> Dense -> Dense -> CRF (ner/models.py:46-67; `droupout_p` spelling is the reference's)."""
    activation = resolve_activation(activation)
    crf_layer = CRF(output_classes)
    model = SequentialNERBertModel([
        nn.Dropout(droupout_p, input_shape=(sequence_length, 768)),
        nn.Dense(hidden_space, activation=activation),
        nn.Dense(output_classes),
        crf_layer,
    ])
    model.loss = crf_layer.loss
    model.loss_sample_weights = crf_layer.loss_sample_weights
    return model


class BertNERModel(NERBertModel):
    """BERT encoder + NER head + CRF in one trainable model: the configuration BASELINE.json quotes
    ("BERT-base polus.ner token classification + CRF, seq 256").  The reference assembles it from
    build_bert_embeddings / TFBertSplited (polus/data.py:523-545, polus/models.py:164-216) feeding a
    baselineNER_* head; here every layer is trainable, so the full 137.7 GFLOP/sequence step runs.
    Called as model(input_ids=..., attention_mask=..., token_type_ids=..., training=...)."""

    def __init__(self, config=None, output_classes=4, hidden_space=128, droupout_p=0.1, activation="swish",
                 name="bert_ner_crf", **kwargs):
        super().__init__(name=name)
        self.config = config or BertConfig(**kwargs)
        self.bert = BertModel(self.config, add_pooling_layer=False)
        self.dropout = nn.Dropout(droupout_p)
        self.hidden = nn.Dense(hidden_space, activation=activation)
        self.out = nn.Dense(output_classes)
        self.crf = CRF(output_classes)
        self.loss = self.crf.loss
        self.loss_sample_weights = self.crf.loss_sample_weights

    def sublayers(self):
        return [self.bert, self.dropout, self.hidden, self.out, self.crf]

    def emissions(self, input_ids=None, attention_mask=None, token_type_ids=None, training=False, position_ids=None):
        h = self.bert(input_ids=input_ids, attention_mask=attention_mask, token_type_ids=token_type_ids,
                      training=training, position_ids=position_ids)["last_hidden_state"]
        h = self.dropout(h, training=training)
        return self.out(self.hidden(h, training=training), training=training)

    def call(self, input_ids=None, attention_mask=None, token_type_ids=None, training=False, position_ids=None, **unused):
        e = self.emissions(input_ids, attention_mask, token_type_ids, training=training, position_ids=position_ids)
        return self.crf(e, training=training)

    def inference(self, x):
        out = self(**x) if isinstance(x, dict) else self(x)
        return ops.argmax(out, axis=-1)


@from_config
def bert_ner_crf(output_classes=4, hidden_space=128, droupout_p=0.1, activation="swish", **kwargs):
    cfg_keys = ("vocab_size", "hidden_size", "num_hidden_layers", "num_attention_heads", "intermediate_size",
                "max_position_embeddings", "type_vocab_size", "hidden_dropout_prob", "attention_probs_dropout_prob",
                "layer_norm_eps", "model_type", "pad_token_id")
    cfg = BertConfig(**{k: kwargs[k] for k in cfg_keys if k in kwargs})
    return BertNERModel(cfg, output_classes=output_classes, hidden_space=hidden_space, droupout_p=droupout_p,
                        activation=activation)
