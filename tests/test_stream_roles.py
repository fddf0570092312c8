"""CPU dry run of a fused (level-2) step: where each C-ABI launch goes.  The dry run takes the GPU's
path through the stream helper (Kernels.side) and binds each launch to the role name of its
stream, 0 being the caller's stream; the stubbed library records (entry, role)."""
import collections

import pytest
import torch

from mmda_b200 import MISA, mosei_config
from mmda_b200._lib import LIB

EARLY_LOSS = ("mmda_loss_phase2", "mmda_loss_gram", "mmda_loss_dxn", "mmda_loss_phase4a",
              "mmda_loss_phase4b")


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
    return calls


@pytest.mark.parametrize("variant", [{}, {"rnncell": "gru"}, {"use_cmd_sim": False}],
                         ids=["default", "gru", "adversarial"])
def test_launch_streams_of_a_fused_step(launches, variant):
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=80, batch_size=12, use_confidNet=True, **variant)
    torch.manual_seed(0)
    model = MISA(cfg).train()
    H = model.engine.H
    assert len(set(H.values())) == 3          # the hidden size tells the modality apart
    mod = {h: m for m, h in H.items()}
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=7)
    tr = FusedTrainer(model)
    launches.clear()
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels)
    cell = variant.get("rnncell", "lstm")
    seen = collections.Counter()

    # each modality's recurrences (forward, BPTT) on that modality's stream
    for name, a, role in launches:
        if name == f"mmda_{cell}_forward":
            assert role == mod[a[-3]], (name, a[-3], role)         # (.., B, H, Tmax, train)
            seen["fwd", role] += 1
        elif name == f"mmda_{cell}_backward":
            assert role == mod[a[-2]], (name, a[-2], role)         # (.., B, H, Tmax)
            seen["bptt", role] += 1
    assert all(seen[k, m] == 2 for k in ("fwd", "bptt") for m in "tva"), seen

    # the hoisted LSTM weight gradients: one stream per (modality, layer, direction), h_prev shift
    # on the first direction's
    wg = collections.defaultdict(list)
    for name, a, role in launches:
        if name == "mmda_gemm_tc" and a[-1] > 0:                   # c_ilv = H: gate-interleaved dW
            assert a[-3] == 1 and role[:2] == ("wg", mod[a[-1]]), (a, role)   # mode 1: accumulate
            wg[role].append(name)
        elif name == "mmda_colsum" and a[-1] > 0:                  # ilv = H: bias gradients
            assert role[:2] == ("wg", mod[a[-1]]), (a, role)
            wg[role].append(name)
        elif name == "mmda_lstm_shift_h":
            assert role[0] == "wg" and role[3] == 0, role
            wg[role].append(name)
        elif name in ("mmda_lstm_backward", "mmda_gru_backward", "mmda_embedding_backward"):
            assert not isinstance(role, tuple)
    assert len(wg) == 12 and {r[2] for r in wg} == {f"{c}rnn{i}" for c in "tva" for i in (1, 2)}
    for role, names in wg.items():
        assert names == ["mmda_lstm_shift_h"] * (role[3] == 0) + ["mmda_gemm_tc"] * 2 + \
            ["mmda_colsum"], (role, names)

    # dense weight gradients (dW += dy^T x) on the leaf stream of the stream that launched the
    # layer's backward; the data gradients stay on the launching stream
    leaf_parents = set()
    for name, a, role in launches:
        if name == "mmda_sgemm":
            ta, beta = a[0], a[10]
            if ta == 1:
                assert beta == 1.0 and isinstance(role, tuple) and role[0] == "leaf", (a, role)
                leaf_parents.add(role[1])
            else:
                assert not (isinstance(role, tuple) and role[0] == "leaf"), (a, role)
    assert leaf_parents == {None, "t", "v", "a"}          # None: the caller's stream

    # the token-only part of the losses on the loss stream, the rest on the caller's
    by_name = collections.defaultdict(list)
    for name, a, role in launches:
        if name.startswith("mmda_loss_"):
            mode = a[-1] if name in ("mmda_loss_phase1", "mmda_loss_finalize") else None
            by_name[name, mode].append(role)
    assert by_name["mmda_loss_phase1", 1] == by_name["mmda_loss_finalize", 1] == ["loss"]
    assert all(by_name[n, None] == ["loss"] for n in EARLY_LOSS)
    assert by_name["mmda_loss_phase1", 2] == by_name["mmda_loss_finalize", 2] == [0]
    assert by_name["mmda_loss_grad_misc", None] == [0]
    if not cfg.use_cmd_sim:
        assert by_name["mmda_loss_domain", None] == [0]

    assert launches[-1][0] == "mmda_adam_clip_step" and launches[-1][2] == 0
