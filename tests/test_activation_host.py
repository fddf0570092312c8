"""Host side of the ELU / Hardshrink / Hardtanh / RReLU activations (reference activation_dict,
src/config.py:24-27): config mapping and refusals, parameter layout against the oracle, the ids
the three layers share, and where a fused step launches the training-mode RReLU kernels (CPU dry
run with a stubbed library, as in test_stream_roles.py)."""
import os
import re

import pytest
import torch
import torch.nn as nn

from mmda_b200 import MISA, MisaConfig, mosei_config
from mmda_b200._lib import HEADER, LIB
from mmda_b200.config import ACTIVATIONS, activation_name

NEW = {"elu": nn.ELU, "hardshrink": nn.Hardshrink, "hardtanh": nn.Hardtanh, "rrelu": nn.RReLU}
CSRC = os.path.join(os.path.dirname(HEADER), "..", "mmda_b200", "csrc")


@pytest.mark.parametrize("name", sorted(NEW))
def test_mapping_of_class_instance_and_name(name):
    cls = NEW[name]
    assert activation_name(cls) == name
    assert activation_name(cls()) == name
    assert activation_name(cls.__name__) == name
    assert activation_name(name.upper()) == name


def test_instances_with_other_arguments_are_refused():
    for act in (nn.ELU(alpha=2.0), nn.Hardtanh(-2.0, 2.0), nn.Hardtanh(max_val=0.5),
                nn.RReLU(0.1, 0.3), nn.RReLU(upper=0.5), nn.Hardshrink(0.3)):
        with pytest.raises(ValueError, match="only torch's defaults"):
            activation_name(act)
        with pytest.raises(ValueError):
            MISA(MisaConfig(vocab_size=10, activation=act))
    # inplace does not change the values
    assert activation_name(nn.ELU(inplace=True)) == "elu"
    assert activation_name(nn.Hardtanh(inplace=True)) == "hardtanh"
    # unchanged: a LeakyReLU instance is taken whatever its slope, other classes stay refused
    assert activation_name(nn.LeakyReLU(0.2)) == "leakyrelu"
    for act in (nn.ReLU6, nn.CELU, nn.SELU, nn.GELU, "prelu"):
        with pytest.raises(ValueError):
            activation_name(act)


def test_prelu_is_refused_with_the_supported_list():
    for act in (nn.PReLU, nn.PReLU(), "PReLU"):
        with pytest.raises(ValueError) as e:
            activation_name(act)
        for name in ("elu", "hardshrink", "hardtanh", "leakyrelu", "relu", "rrelu", "tanh"):
            assert repr(name) in str(e.value)


@pytest.mark.parametrize("use_cmd_sim", [True, False], ids=["cmd", "adversarial"])
@pytest.mark.parametrize("name", sorted(NEW))
def test_state_dict_layout_matches_the_oracle(name, use_cmd_sim):
    from oracle.misa_oracle import OracleMISA
    cfg = MisaConfig(vocab_size=40, embedding_size=12, visual_size=5, acoustic_size=6,
                     hidden_size=16, activation=NEW[name], use_cmd_sim=use_cmd_sim)
    mine, ref = MISA(cfg).state_dict(), OracleMISA(cfg).state_dict()
    assert list(mine) == list(ref)
    assert all(mine[k].shape == ref[k].shape for k in ref)
    # the activation module is registered under the reference's names and holds no parameter
    model = MISA(cfg)
    assert isinstance(model.project_t.project_t_activation, NEW[name])
    assert not any("activation" in k for k in mine)


def test_activation_ids_agree_across_python_cuda_and_the_header():
    header = dict((k.lower(), int(v)) for k, v in
                  re.findall(r"#define MMDA_ACT_(\w+) (\d+)", open(HEADER).read()))
    enum_src = re.search(r"enum : int \{([^}]*)\}", open(os.path.join(CSRC, "common.cuh")).read()).group(1)
    cuda = dict((k.lower(), int(v)) for k, v in re.findall(r"ACT_(\w+) = (\d+)", enum_src))
    assert header == cuda == ACTIVATIONS
    for name in NEW:
        assert name in ACTIVATIONS


# ---- CPU dry run of a fused step ------------------------------------------------------------
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


def _fused_step(launches, train=True, **kw):
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=80, batch_size=12, use_confidNet=True, **kw)
    torch.manual_seed(0)
    model = MISA(cfg).train(train)
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=7)
    tr = FusedTrainer(model)
    launches.clear()
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels)
    return list(launches), tr, cfg


@pytest.mark.parametrize("use_cmd_sim", [True, False], ids=["cmd", "adversarial"])
def test_rrelu_launches_of_a_fused_step(launches, use_cmd_sim):
    from mmda_b200.engine import SID_RRELU_DISC, SID_RRELU_PROJECT
    ref, _, _ = _fused_step(launches, use_cmd_sim=use_cmd_sim)
    got, tr, cfg = _fused_step(launches, use_cmd_sim=use_cmd_sim, activation="rrelu")
    B, d = cfg.batch_size, cfg.hidden_size
    state = tr.state.data_ptr()
    rr = [(n, a, role) for n, a, role in got if n.startswith("mmda_rrelu_")]
    # (x | dy, y, ld, rows, cols, seed, seed_dev, stream id): the heads' forward and backward on
    # their modality's stream, the discriminator's on the caller's
    want = {("mmda_rrelu_forward", SID_RRELU_PROJECT + i, m) for i, m in enumerate("tva")} | \
        {("mmda_rrelu_backward", SID_RRELU_PROJECT + i, m) for i, m in enumerate("tva")}
    if not use_cmd_sim:
        want |= {(f"mmda_rrelu_{w}", SID_RRELU_DISC + i, 0) for i in range(3)
                 for w in ("forward", "backward")}
    assert {(n, a[-1], role) for n, a, role in rr} == want and len(rr) == len(want)
    for n, a, role in rr:
        assert a[2:5] == (d, B, d) and a[-2] == state, (n, a)     # seed_dev: the device step counter
        if n == "mmda_rrelu_forward":
            assert a[0] == a[1]                                      # in place
    # the linear in front of each RReLU site runs without an epilogue, and the RReLU backward takes
    # the place of the activation backward; everything else is the LeakyReLU step's list, launch
    # for launch
    act_of = {ACTIVATIONS["leakyrelu"], ACTIVATIONS["rrelu"]}
    strip = [("mmda_act_backward" if n == "mmda_rrelu_backward" else n, role)
             for n, a, role in got if n != "mmda_rrelu_forward"]
    assert strip == [(n, role) for n, a, role in ref]
    assert sum(n == "mmda_act_backward" and a[-1] == ACTIVATIONS["leakyrelu"]
               for n, a, role in ref) == len(want) // 2
    assert not any(n == "mmda_sgemm" and a[15] in act_of for n, a, role in got)
    n_act = sum(n == "mmda_sgemm" and a[15] == ACTIVATIONS["leakyrelu"] for n, a, role in ref)
    assert n_act == (3 if use_cmd_sim else 6)
    assert not any(n.startswith("mmda_rrelu_") for n, a, role in ref)


def test_rrelu_in_eval_mode_is_a_fused_epilogue(launches):
    got, _, _ = _fused_step(launches, train=False, activation="rrelu")
    assert not any(n.startswith("mmda_rrelu_") for n, a, role in got)
    assert sum(n == "mmda_sgemm" and a[15] == ACTIVATIONS["rrelu"] for n, a, role in got) == 3
    assert sum(n == "mmda_act_backward" and a[-1] == ACTIVATIONS["rrelu"] for n, a, role in got) == 3
