"""CPU dry run of the deterministic mode (torch.use_deterministic_algorithms): with the flag on no
launch of a step uses an order-dependent reduction; with it off the launch sequence is the one of a
run that never touched the flag.  The stubbed library records (entry, args, stream role)."""
import pytest
import torch

from mmda_b200 import MISA, mosei_config
from mmda_b200._lib import LIB

ATOMIC_ENTRIES = {"mmda_colsum", "mmda_layernorm_backward", "mmda_embedding_backward",
                  "mmda_loss_phase2", "mmda_loss_phase4a", "mmda_loss_dxn",
                  "mmda_layernorm_backward_dropout", "mmda_bert_embed_backward"}


@pytest.fixture
def launches(monkeypatch):
    import mmda_b200.engine as E
    calls = []

    def stub(name, *args):
        calls.append((name, args[:-1], args[-1]))
        return 0
    monkeypatch.setattr(E, "_DRYRUN", True)
    monkeypatch.setattr(LIB, "call", stub)
    monkeypatch.setattr(LIB, "raw", lambda name: (lambda *a: 4096))
    yield calls
    torch.use_deterministic_algorithms(False)


def _order_dependent(name, a):
    if name in ATOMIC_ENTRIES:
        return True
    if name == "mmda_sgemm":       # (ta, tb, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, bias2, act, split_k, c_ilv)
        beta, act, split_k = a[10], a[15], a[16]
        return split_k >= 2 or (split_k == 0 and act == 0 and beta == 1.0)
    if name == "mmda_gemm_tc":     # (..., mode, split_k, c_ilv)
        return a[-3] == 1 and a[-2] != 1
    return False


def _trainer(variant, seed=0):
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=80, batch_size=12, use_confidNet=True, **variant)
    torch.manual_seed(seed)
    model = MISA(cfg).train()
    return cfg, model, FusedTrainer(model)


def _step(tr, cfg, seed=1, lengths="ragged"):
    from mmda_b200.synthetic import batch_for
    b = batch_for(cfg, seed=seed, lengths=lengths, seq_len=7)
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels)


VARIANTS = [{}, {"rnncell": "gru"}, {"use_cmd_sim": False}]


@pytest.mark.parametrize("lengths", ["ragged", "full"])
@pytest.mark.parametrize("variant", VARIANTS, ids=["default", "gru", "adversarial"])
def test_fused_step_uses_no_order_dependent_reduction(launches, variant, lengths):
    cfg, model, tr = _trainer(variant)
    torch.use_deterministic_algorithms(True)
    launches.clear()
    _step(tr, cfg, lengths=lengths)
    bad = [(n, a, r) for n, a, r in launches if _order_dependent(n, a)]
    assert not bad, bad[:5]
    names = [n for n, _, _ in launches]
    for entry in ("mmda_colsum_det", "mmda_layernorm_backward_det", "mmda_embedding_backward_det",
                  "mmda_loss_phase2_det", "mmda_loss_phase4a_det", "mmda_loss_dxn_det"):
        assert entry in names, entry
    # shared.shared_1: one partial per head stream, summed by one launch on the caller's stream
    d = cfg.hidden_size
    sums = [(a, r) for n, a, r in launches if n == "mmda_fixed_order_sum" and a[-1] == d * d]
    assert len(sums) == 1 and sums[0][1] == 0 and sums[0][0][1] == 3, sums


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_bert_step_uses_no_order_dependent_reduction(launches, precision):
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=50, batch_size=4, use_bert=True, precision=precision)
    torch.manual_seed(0)
    model = MISA(cfg).train()
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=8)
    tr = FusedTrainer(model)
    torch.use_deterministic_algorithms(True)
    launches.clear()
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels, b.bert_sent, b.bert_sent_type,
            b.bert_sent_mask)
    bad = [(n, a, r) for n, a, r in launches if _order_dependent(n, a)]
    assert not bad, bad[:5]
    names = {n for n, _, _ in launches}
    assert {"mmda_bert_embed_backward_det", "mmda_layernorm_backward_dropout_det",
            "mmda_gemm_tc_det", "mmda_colsum_det"} <= names


def test_level1_and_eval_use_no_order_dependent_reduction(launches):
    from mmda_b200.evaluate import evaluate
    from mmda_b200.synthetic import batch_for
    cfg = mosei_config(vocab_size=80, batch_size=12, use_confidNet=True)
    torch.manual_seed(0)
    model = MISA(cfg).train()
    b = batch_for(cfg, seed=3, lengths="ragged", seq_len=7)
    torch.use_deterministic_algorithms(True)
    launches.clear()
    out = model(b.sentences, b.visual, b.acoustic, b.lengths)
    loss = sum(v.float().sum() for v in out if torch.is_tensor(v) and v.requires_grad)
    loss.backward()
    evaluate(model, [b])
    assert any(n == "mmda_layernorm_backward_det" for n, _, _ in launches)
    bad = [(n, a, r) for n, a, r in launches if _order_dependent(n, a)]
    assert not bad, bad[:5]


def _normalised(calls):
    """pointer arguments (CPU addresses in the dry run) -> order of first appearance"""
    ids = {}
    out = []
    for n, a, r in calls:
        out.append((n, tuple(ids.setdefault(x, f"p{len(ids)}") if isinstance(x, int) and x > 1 << 22
                             else x for x in a), r))
    return out


@pytest.mark.parametrize("variant", VARIANTS, ids=["default", "gru", "adversarial"])
def test_flag_off_restores_the_launch_sequence(launches, variant):
    cfg, _, tr = _trainer(variant)
    _step(tr, cfg, seed=1)
    launches.clear()
    _step(tr, cfg, seed=2)
    never = _normalised(launches)

    cfg, _, tr = _trainer(variant)
    torch.use_deterministic_algorithms(True)
    _step(tr, cfg, seed=1)
    torch.use_deterministic_algorithms(False)
    launches.clear()
    _step(tr, cfg, seed=2)
    assert _normalised(launches) == never
    assert not any(n.endswith("_det") or n == "mmda_fixed_order_sum" for n, _, _ in launches)
