"""Which attention core the BERT encoder (mmda_b200/bert.py) launches at each sequence length, on
a stubbed library: the shared-memory resident kernels wherever they ran before, the tiled kernels
(no S x S buffer) only beyond the resident limits (S > 84 with a backward, S > 116 without)."""
import collections

import pytest
import torch

from mmda_b200 import MISA, mosei_config
from mmda_b200._lib import LIB

RESIDENT = ("mmda_bert_attention_forward", "mmda_bert_attention_backward",
            "mmda_bert_attention_forward_mma", "mmda_bert_attention_backward_mma")


class _StubLib:
    def __init__(self):
        self.calls = []
    def __call__(self, name, *args):
        self.calls.append(name)
        return 0


def _raw(name):
    if name == "mmda_bert_attention_resident_max_seq":
        return lambda backward: 84 if backward else 116
    return lambda *a: 4096


@pytest.fixture
def dryrun(monkeypatch):
    import mmda_b200.engine as E
    stub = _StubLib()
    monkeypatch.setattr(E, "_DRYRUN", True)
    monkeypatch.setattr(LIB, "call", stub)
    monkeypatch.setattr(LIB, "raw", _raw)
    return stub


def _step(precision, seq_len, B=4):
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=50, batch_size=B, use_bert=True, precision=precision)
    torch.manual_seed(0)
    model = MISA(cfg).train()
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=seq_len)
    tr = FusedTrainer(model)
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels, b.bert_sent, b.bert_sent_type,
            b.bert_sent_mask)
    return tr, b


@pytest.mark.parametrize("precision,sfx", [("fp32", "_tiled"), ("bf16", "_tiled_mma")])
def test_long_training_step_goes_tiled(dryrun, precision, sfx):
    tr, b = _step(precision, 128)
    B, S = b.bert_sent.shape
    assert S == 130
    c = collections.Counter(dryrun.calls)
    assert c["mmda_bert_attention_forward" + sfx] == 12
    assert c["mmda_bert_attention_backward" + sfx] == 12
    assert not any(c[n] for n in RESIDENT), {n: c[n] for n in RESIDENT}
    other = "_tiled" if sfx == "_tiled_mma" else "_tiled_mma"
    assert c["mmda_bert_attention_forward" + other] == c["mmda_bert_attention_backward" + other] == 0
    ws = tr.eng.ws
    assert not [n for n in ws if n.startswith("bert_probs_")]
    for l in range(12):
        assert ws[f"bert_lse_{l}"].numel() == B * 12 * S
    assert ws["bert_att_delta"].numel() == B * 12 * S


@pytest.mark.parametrize("precision,seq_len,fwd", [
    ("fp32", 50, "mmda_bert_attention_forward"),          # C4 shape: unchanged
    ("bf16", 50, "mmda_bert_attention_forward_mma"),
    ("fp32", 82, "mmda_bert_attention_forward"),          # S = 84: the resident backward's limit
    ("bf16", 70, "mmda_bert_attention_forward"),          # bf16 at 65..84: the fp32 resident pair
])
def test_training_steps_that_fit_stay_resident(dryrun, precision, seq_len, fwd):
    tr, _ = _step(precision, seq_len)
    c = collections.Counter(dryrun.calls)
    assert c[fwd] == 12 and c[fwd.replace("forward", "backward")] == 12
    assert not any(n for n in c if "_tiled" in n)
    assert "bert_lse_0" not in tr.eng.ws


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_forward_resident_up_to_116(dryrun, precision):
    from mmda_b200.synthetic import batch_for
    cfg = mosei_config(vocab_size=50, batch_size=3, use_bert=True, precision=precision)
    torch.manual_seed(0)
    model = MISA(cfg).eval()
    be = model.engine.bert
    sfx = "_tiled_mma" if precision == "bf16" else "_tiled"
    for seq_len, want in ((98, "mmda_bert_attention_forward"),
                          (114, "mmda_bert_attention_forward"),
                          (115, "mmda_bert_attention_forward" + sfx),
                          (128, "mmda_bert_attention_forward" + sfx)):
        b = batch_for(cfg, seed=2, lengths="ragged", seq_len=seq_len)
        dryrun.calls.clear()
        be.forward(b.bert_sent, b.bert_sent_type, b.bert_sent_mask, train=False, drop=False, seed=0)
        c = collections.Counter(n for n in dryrun.calls if n.startswith("mmda_bert_attention"))
        assert c == {want: 12}, (seq_len + 2, c)
    assert not [n for n in model.engine.ws if n.startswith(("bert_probs_", "bert_lse_"))]
