"""Drop-in ``MISA`` model class for the reference's ``Solver`` (SURVEY.md section 8b, row B1).

Same constructor (one ``config`` object), same ``forward(sentences, video, acoustic, lengths,
bert_sent, bert_sent_type, bert_sent_mask) -> (scores, labels)`` signature, same parameter /
``state_dict`` key names and registration order (so the same ``torch.manual_seed`` gives the same
initial weights and reference checkpoints load), and the same post-forward attributes the
reference's ``get_*_loss`` functions read (reference src/models.py:15-285, src/solver.py:63-99,
154, 373-462).  The torch modules created here are *parameter containers only*: none of their
``forward`` methods is ever called.  All arithmetic runs in ``libmmda_b200.so`` through
:class:`mmda_b200.engine.MisaEngine`; there is no CPU or eager-PyTorch fallback.
"""
from __future__ import annotations

import math
import warnings

import torch
import torch.nn as nn

from .config import activation_name

MODS = ("t", "v", "a")
_TORCH_ACT = {"leakyrelu": nn.LeakyReLU, "relu": nn.ReLU, "tanh": nn.Tanh, "sigmoid": nn.Sigmoid,
              "elu": nn.ELU, "hardshrink": nn.Hardshrink, "hardtanh": nn.Hardtanh, "rrelu": nn.RReLU}


class BiLSTMParams(nn.Module):
    """Parameter container with ``nn.LSTM(input, hidden, bidirectional=True)``'s names, shapes,
    registration order and U(-1/sqrt(H), 1/sqrt(H)) init (so RNG consumption matches).
    ``gates=3`` gives ``nn.GRU``'s shapes (rows r,z,n) under the same names."""

    def __init__(self, input_size: int, hidden_size: int, gates: int = 4):
        super().__init__()
        self.input_size, self.hidden_size, self.gates = input_size, hidden_size, gates
        for suffix in ("", "_reverse"):
            self.register_parameter(f"weight_ih_l0{suffix}",
                                    nn.Parameter(torch.empty(gates * hidden_size, input_size)))
            self.register_parameter(f"weight_hh_l0{suffix}",
                                    nn.Parameter(torch.empty(gates * hidden_size, hidden_size)))
            self.register_parameter(f"bias_ih_l0{suffix}", nn.Parameter(torch.empty(gates * hidden_size)))
            self.register_parameter(f"bias_hh_l0{suffix}", nn.Parameter(torch.empty(gates * hidden_size)))
        stdv = 1.0 / math.sqrt(hidden_size) if hidden_size > 0 else 0
        for w in self.parameters():
            nn.init.uniform_(w, -stdv, stdv)

    def forward(self, *a, **k):
        raise RuntimeError("BiLSTMParams holds parameters only; the recurrence runs in libmmda_b200")


def _named_seq(**mods) -> nn.Sequential:
    s = nn.Sequential()
    for name, m in mods.items():
        s.add_module(name, m)
    return s


class MISA(nn.Module):
    """MISA for multi-label emotion classification on B200 (reference src/models.py:15)."""

    OUTPUT_ATTRS = ("utt_t_orig", "utt_v_orig", "utt_a_orig", "utt_private_t", "utt_private_v",
                    "utt_private_a", "utt_shared_t", "utt_shared_v", "utt_shared_a", "utt_t",
                    "utt_v", "utt_a", "utt_t_recon", "utt_v_recon", "utt_a_recon", "tcp",
                    "shared_or_private_p_t", "shared_or_private_p_v", "shared_or_private_p_a",
                    "shared_or_private_s")

    def __init__(self, config):
        super().__init__()
        self.config = config
        d = config.hidden_size
        self.text_size, self.visual_size, self.acoustic_size = (
            config.embedding_size, config.visual_size, config.acoustic_size)
        self.input_sizes = [self.text_size, self.visual_size, self.acoustic_size]
        self.hidden_sizes = [int(s) for s in self.input_sizes]
        self.output_size = config.num_classes
        self.dropout_rate = config.dropout
        self.act_name = activation_name(config.activation)
        act_mod = _TORCH_ACT[self.act_name]()          # container entry only (keeps key layout)

        if getattr(config, "extractor", "lstm") == "transformer":
            raise NotImplementedError("extractor='transformer' exits in the reference too "
                                      "(src/models.py:33-36)")
        self.rnncell = "lstm" if getattr(config, "rnncell", "lstm") == "lstm" else "gru"   # models.py:39
        ng = 4 if self.rnncell == "lstm" else 3
        if d % 2:
            raise ValueError("hidden_size must be even (2 attention heads)")

        sz = dict(zip(MODS, self.hidden_sizes))
        if config.use_bert:
            from transformers import BertConfig, BertModel
            # bert-base-uncased geometry; weights are random-init (no network), SURVEY.md row O1
            self.bertmodel = BertModel(BertConfig(output_hidden_states=True))
        else:
            self.embed = nn.Embedding(len(config.word2id), sz["t"])
            self.trnn1 = BiLSTMParams(sz["t"], sz["t"], ng)
            self.trnn2 = BiLSTMParams(2 * sz["t"], sz["t"], ng)
        self.vrnn1 = BiLSTMParams(sz["v"], sz["v"], ng)
        self.vrnn2 = BiLSTMParams(2 * sz["v"], sz["v"], ng)
        self.arnn1 = BiLSTMParams(sz["a"], sz["a"], ng)
        self.arnn2 = BiLSTMParams(2 * sz["a"], sz["a"], ng)

        for m in MODS:
            fan_in = 768 if (m == "t" and config.use_bert) else 4 * sz[m]
            setattr(self, f"project_{m}", _named_seq(**{
                f"project_{m}": nn.Linear(fan_in, d),
                f"project_{m}_activation": act_mod,
                f"project_{m}_layer_norm": nn.LayerNorm(d)}))
        for m, tag in zip(MODS, ("1", "1", "3")):
            setattr(self, f"private_{m}", _named_seq(**{
                f"private_{m}_{tag}": nn.Linear(d, d),
                f"private_{m}_activation_{tag}": nn.Sigmoid()}))
        self.shared = _named_seq(shared_1=nn.Linear(d, d), shared_activation_1=nn.Sigmoid())
        for m in MODS:
            setattr(self, f"recon_{m}", _named_seq(**{f"recon_{m}_1": nn.Linear(d, d)}))
        if not getattr(config, "use_cmd_sim", True):      # adversarial branch, models.py:122-127
            self.discriminator = _named_seq(
                discriminator_layer_1=nn.Linear(d, d),
                discriminator_layer_1_activation=act_mod,
                discriminator_layer_1_dropout=nn.Dropout(config.dropout),
                discriminator_layer_2=nn.Linear(d, len(self.hidden_sizes)))
        self.sp_discriminator = _named_seq(sp_discriminator_layer_1=nn.Linear(d, 4))
        self.confidence = _named_seq(confidence_layer_1=nn.Linear(6 * d, 6),
                                     confidence_layer_activation=nn.Sigmoid())
        self.classifier = _named_seq(
            classifier_layer=nn.Linear(6 * d, config.num_classes),
            classifier_layer_dropout=nn.Dropout(config.dropout),
            classifier_layer_activation=nn.Sigmoid())
        self.tlayer_norm = nn.LayerNorm((2 * sz["t"],))
        self.vlayer_norm = nn.LayerNorm((2 * sz["v"],))
        self.alayer_norm = nn.LayerNorm((2 * sz["a"],))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            self.transformer_encoder = nn.TransformerEncoder(
                nn.TransformerEncoderLayer(d_model=d, nhead=2), num_layers=1)

        self._engine = None
        self.domain_label_t = self.domain_label_v = self.domain_label_a = None

    # -- plumbing ---------------------------------------------------------------------------
    @property
    def engine(self):
        if self._engine is None:
            from .engine import MisaEngine
            object.__setattr__(self, "_engine", MisaEngine(self))
        return self._engine

    def param_names_without_grad(self):
        """Parameters the reference leaves at ``grad=None`` after ``loss.backward()``
        (SURVEY.md hard part 7): the shared/private discriminator always, the confidence head
        unless ``use_confidNet``."""
        skip = ["sp_discriminator."]
        if not getattr(self.config, "use_confidNet", False):
            skip.append("confidence.")
        if getattr(self.config, "use_bert", False):
            skip += ["tlayer_norm.", "bertmodel.pooler."]
        return [n for n, _ in self.named_parameters() if any(n.startswith(s) for s in skip)]

    # -- reference src/models.py:282-285 -----------------------------------------------------
    def forward(self, sentences, video, acoustic, lengths, bert_sent=None, bert_sent_type=None,
                bert_sent_mask=None):
        from .engine import misa_apply
        out = misa_apply(self, sentences, video, acoustic, lengths, bert_sent, bert_sent_type,
                         bert_sent_mask)
        for k in self.OUTPUT_ATTRS:
            object.__setattr__(self, k, out[k])
        for m in MODS:      # models.py:219-231
            object.__setattr__(self, f"domain_label_{m}", out.get(f"domain_label_{m}"))
        return out["scores"], out["labels"]
