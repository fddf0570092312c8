"""CPU-side checks: the C-ABI library loads and exports every symbol include/mmda_b200.h declares
(no compute calls without a GPU), and the host logic around it (config mapping, synthetic data,
arena/bucket plan, kernel sequencing of the engine with a stubbed library)."""
import collections
import ctypes
import os

import pytest
import torch

from mmda_b200 import MISA, MisaConfig, mosei_config
from mmda_b200._lib import LIB, LIB_PATH, MmdaError, parse_header


def test_library_exports_every_declared_symbol():
    assert os.path.exists(LIB_PATH), "build with `python -m mmda_b200.build` / __graft_entry__.build()"
    dll = ctypes.CDLL(LIB_PATH)
    protos = parse_header()
    assert len(protos) >= 30
    for name in protos:
        assert hasattr(dll, name), f"{name} declared in include/mmda_b200.h but not exported"
    assert LIB.load().mmda_abi_version() == 2
    assert LIB.load().mmda_last_error() is not None


def test_pack_weights_refuses_misaligned_outputs():
    """A pack mode (0 / 1 / 2) in out_a's place, or any output that is no float array, is an
    argument error before anything is launched (no GPU needed to see it)."""
    pack = LIB.raw("mmda_lstm_pack_weights")
    p = 1 << 40                                    # 16-byte aligned stand-in, never dereferenced
    for out_a, out_b, bias in ((1, p, p), (2, p, p), (p, p + 2, p), (p, p, p + 1)):
        rc = pack(p, p, p, p, p, p, 37, 23, out_a, out_b, 29, bias, None)
        assert rc == -2, (out_a, out_b, bias, rc)    # MMDA_ERR_ARG
        assert b"aligned" in LIB.load().mmda_last_error()


def test_header_cites_reference_sites():
    text = open(os.path.join(os.path.dirname(LIB_PATH), "..", "include", "mmda_b200.h")).read()
    for site in ("src/models.py:164", "src/models.py:48-55", "src/solver.py:185-186",
                 "src/utils/functions.py:112-115", "src/solver.py:163-181"):
        assert site in text, site


def test_config_activation_mapping_and_errors():
    import torch.nn as nn
    from mmda_b200.config import activation_name
    assert activation_name(nn.LeakyReLU) == "leakyrelu"
    assert activation_name(nn.ReLU()) == "relu"
    assert activation_name("Tanh") == "tanh"
    with pytest.raises(ValueError):
        activation_name(nn.PReLU)
    gru = MISA(MisaConfig(vocab_size=10, rnncell="gru", embedding_size=8)).state_dict()
    assert gru["trnn2.weight_ih_l0_reverse"].shape == (24, 16) and gru["trnn1.bias_hh_l0"].shape == (24,)
    adv = MISA(MisaConfig(vocab_size=10, use_cmd_sim=False))
    assert "discriminator.discriminator_layer_2.weight" in adv.state_dict()


def test_product_path_refuses_cpu():
    """No CPU fallback: a model left on the CPU must fail loudly, not compute in eager PyTorch."""
    from mmda_b200._lib import MmdaError
    from mmda_b200.synthetic import batch_for
    cfg = MisaConfig(embedding_size=8, visual_size=4, acoustic_size=4, hidden_size=8, vocab_size=30)
    model = MISA(cfg)
    b = batch_for(cfg, seed=0, lengths="ragged", batch=3, seq_len=4)
    with pytest.raises(MmdaError):
        model(*b.model_args())


def test_state_dict_keys_and_same_seed_init_match_oracle():
    from oracle.misa_oracle import OracleMISA
    cfg = mosei_config(vocab_size=50)
    torch.manual_seed(7); a = MISA(cfg)
    torch.manual_seed(7); b = OracleMISA(cfg)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb)
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert [n for n, _ in a.named_parameters()] == [n for n, _ in b.named_parameters()]
    assert a.param_names_without_grad() == [n for n in sa if n.startswith(("sp_discriminator.", "confidence."))]


def test_synthetic_batch_contract():
    from mmda_b200.synthetic import PAD_ID, batch_for
    cfg = mosei_config(vocab_size=100)
    for mode in ("full", "ragged", "shuffled"):
        b = batch_for(cfg, seed=3, lengths=mode, batch=17, seq_len=11)
        T = int(b.lengths.max())
        assert b.sentences.shape == (T, 17) and b.sentences.dtype == torch.int64
        assert b.visual.shape == (T, 17, 35) and b.acoustic.shape == (T, 17, 74)
        assert not b.lengths.is_cuda and T == 11
        for j in range(17):
            L = int(b.lengths[j])
            assert bool((b.sentences[L:, j] == PAD_ID).all()) and bool((b.sentences[:L, j] >= 2).all())
            assert float(b.visual[L:, j].abs().sum()) == 0 and float(b.acoustic[L:, j].abs().sum()) == 0
        assert bool((b.labels.sum(0) > 0).all())
        if mode == "ragged":
            assert bool((b.lengths[:-1] >= b.lengths[1:]).all())


def test_arena_plan_buckets_are_contiguous_and_ordered():
    from mmda_b200.trainer import ALIGN, bucket_of, plan_arena
    m = MISA(mosei_config(vocab_size=64))
    shapes = [(n, tuple(p.shape)) for n, p in m.named_parameters()]
    for confid in (False, True):
        layout, ranges, n_active, n_total = plan_arena(shapes, confid)
        assert len(ranges) == 7 and ranges[0][0] == 0 and ranges[-1][1] == n_active <= n_total
        for (lo, hi), (lo2, _hi2) in zip(ranges, ranges[1:]):
            assert hi == lo2 and lo <= hi
        for n, (off, sz) in layout.items():
            assert off % ALIGN == 0
            inactive = n.startswith("sp_discriminator.") or (n.startswith("confidence.") and not confid)
            if inactive:
                assert off >= n_active
            else:
                b = bucket_of(n)
                assert ranges[b][0] <= off and off + sz <= ranges[b][1], n
        spans = sorted(layout.values())
        for (o1, s1), (o2, _s2) in zip(spans, spans[1:]):
            assert o1 + s1 <= o2


class _StubLib:
    """Records the C-ABI call sequence (names; arguments in `args`, the stream last); lets the
    engine's host orchestration run on CPU."""
    def __init__(self):
        self.calls, self.args = [], []
    def __call__(self, name, *args):
        self.calls.append(name)
        self.args.append(args)
        return 0


@pytest.fixture
def dryrun(monkeypatch):
    import mmda_b200.engine as E
    stub = _StubLib()
    monkeypatch.setattr(E, "_DRYRUN", True)
    monkeypatch.setattr(LIB, "call", stub)
    monkeypatch.setattr(LIB, "raw", lambda name: (lambda *a: 4096))
    return stub


def test_engine_kernel_sequence_level1_and_level2_early_loss(dryrun):
    """Level-1 gradient contract, then the C-ABI order of a fused step as the GPU runs it: the
    token-only loss chain forked behind the heads, the rest of the losses before the backward."""
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=80, batch_size=12, use_confidNet=True)
    torch.manual_seed(0)
    model = MISA(cfg).train()
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=7)
    scores, labels = model(*b.model_args())
    assert scores.shape == (12, 6) and labels.shape == (12, 6) and not labels.requires_grad
    for attr in model.OUTPUT_ATTRS:
        assert getattr(model, attr).requires_grad, attr
    (scores.sum() + model.utt_shared_t.sum()).backward()
    none = [n for n, p in model.named_parameters() if p.grad is None]
    assert none == [n for n, _ in model.named_parameters() if n.startswith(("sp_discriminator.", "confidence."))]
    fwd = collections.Counter(dryrun.calls)
    assert fwd["mmda_lstm_forward"] == 6 and fwd["mmda_lstm_backward"] == 6
    # every encoder's hoisted GEMMs run on tcgen05: 2 fwd + 4 dW_ih + 4 dW_hh each, + dX of both
    # text layers (the embedding needs it) / of layer 2 only (visual, acoustic): 12 + 11 + 11
    assert fwd["mmda_gemm_tc"] == 34
    dryrun.calls.clear()
    dryrun.args.clear()
    tr = FusedTrainer(model)
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels)
    seq = dryrun.calls
    assert seq[-1] == "mmda_adam_clip_step"
    mode = lambda name: [a[-2] for n, a in zip(seq, dryrun.args) if n == name]    # last arg: stream
    assert mode("mmda_loss_phase1") == [1, 2] and mode("mmda_loss_finalize") == [1, 2]
    # the token-only part of the losses (DiffLoss / CMD) is enqueued right behind the heads (the
    # last one ends with utt = private + shared and the recon linear), before the fusion layer
    i1 = seq.index("mmda_loss_phase1")
    assert seq[i1 - 2:i1] == ["mmda_add2d", "mmda_sgemm"]
    assert seq[i1:i1 + 9] == ["mmda_loss_phase1", "mmda_loss_phase2", "mmda_loss_gram",
                              "mmda_loss_finalize", "mmda_loss_dxn", "mmda_loss_phase4a",
                              "mmda_loss_phase4b", "mmda_sgemm", "mmda_attention_forward"]
    late = lambda name: len(seq) - 1 - seq[::-1].index(name)       # last call of that name
    order = [seq.index("mmda_embedding_forward"), seq.index("mmda_lstm_forward"),
             seq.index("mmda_attention_forward"), late("mmda_loss_phase1"),
             late("mmda_loss_finalize"), seq.index("mmda_loss_grad_misc"),
             seq.index("mmda_attention_backward"), seq.index("mmda_lstm_backward"),
             seq.index("mmda_embedding_backward"), seq.index("mmda_adam_clip_step")]
    assert order == sorted(order)
    c2 = collections.Counter(seq)
    assert c2["mmda_loss_phase1"] == 2 and c2["mmda_loss_phase2"] == c2["mmda_loss_phase4a"] == 1
    # parameters alias the arena; untouched-by-contract params sit past the active range
    for n, p in model.named_parameters():
        off, sz = tr.layout[n]
        assert p.data_ptr() == tr.p_arena[off:].data_ptr()


def test_metrics_from_stats_matches_reference_definitions():
    """Host-side finalisation of the device metric counters vs the reference's formulas
    (src/utils/eval.py:14-65: get_accuracy loop restated, sklearn precision/recall/F1)."""
    import numpy as np
    from sklearn import metrics as M
    from mmda_b200.evaluate import metrics_from_stats
    rng = np.random.default_rng(0)
    y = (rng.random((300, 6)) < 0.3).astype(np.float32)
    p = (rng.random((300, 6)) < 0.35).astype(np.float32)
    y[:, 5] = 0                      # a class with no positives: zero-division paths
    NC = 6
    both, anyv = (y * p).sum(1), np.maximum(((y + p) > 0).sum(1), 1)
    stats = [float((both / anyv).sum()), 300.0, 12.5, 5.0]
    stats += [float(((y > 0) & (p > 0))[:, c].sum()) for c in range(NC)]
    stats += [float(((y == 0) & (p > 0))[:, c].sum()) for c in range(NC)]
    stats += [float(((y > 0) & (p == 0))[:, c].sum()) for c in range(NC)]
    got = metrics_from_stats(stats, NC)
    # reference get_accuracy
    count = 0.0
    for i in range(300):
        t = sum(1 for j in range(6) if y[i][j] > 0 and p[i][j] > 0)
        a = sum(1 for j in range(6) if y[i][j] > 0 or p[i][j] > 0) or 1
        count += t / a
    assert got["acc"] == round(count / 300, 4)
    assert got["loss"] == 2.5
    for avg, pre in (("macro", ""), ("micro", "micro_"), ("weighted", "weighted_")):
        assert abs(got[pre + "f1"] - M.f1_score(y, p, average=avg, zero_division=0)) < 1e-9
        assert abs(got[pre + "precision"] - M.precision_score(y, p, average=avg, zero_division=0)) < 1e-9
        assert abs(got[pre + "recall"] - M.recall_score(y, p, average=avg, zero_division=0)) < 1e-9


def test_bert_branch_kernel_sequence_and_freeze_contract(dryrun):
    """use_bert=True on the stubbed library: the hand-written BERT encoder issues 6 dense GEMMs per
    layer forward, 6 data-gradient GEMMs per layer backward, and weight-gradient GEMMs only for
    the layers the Solver leaves trainable (solver.py:66-73 freezes encoder layers 0-8)."""
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=50, batch_size=4, use_bert=True)
    torch.manual_seed(0)
    model = MISA(cfg).train()
    for n, p in model.named_parameters():
        if "bertmodel.encoder.layer" in n and int(n.split("encoder.layer.")[-1].split(".")[0]) <= 8:
            p.requires_grad = False
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=5)
    tr = FusedTrainer(model)
    # frozen tensors and the never-used pooler / tlayer_norm sit past the optimizer's range
    for n, _ in model.named_parameters():
        off, sz = tr.layout[n]
        frozen = ("encoder.layer." in n and int(n.split("encoder.layer.")[-1].split(".")[0]) <= 8) \
            or n.startswith(("bertmodel.pooler.", "tlayer_norm.", "sp_discriminator.", "confidence."))
        assert (off >= tr.n_active) == frozen, n
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels, b.bert_sent, b.bert_sent_type,
            b.bert_sent_mask)
    c = collections.Counter(dryrun.calls)
    assert c["mmda_bert_attention_forward"] == 12 and c["mmda_bert_attention_backward"] == 12
    assert c["mmda_gelu_forward"] == 12 and c["mmda_gelu_backward"] == 12
    # BERT: fwd + dgrad + wgrad(layers 9-11); + the visual / acoustic LSTM encoders' hoisted GEMMs
    assert c["mmda_gemm_tc"] == 12 * 6 + 12 * 6 + 3 * 6 + 2 * 11
    assert c["mmda_bert_embed_forward"] == c["mmda_bert_embed_backward"] == 1
    assert c["mmda_lstm_forward"] == 4                          # visual + acoustic only
    seq = dryrun.calls
    assert seq.index("mmda_bert_embed_forward") < seq.index("mmda_masked_mean_forward") \
        < seq.index("mmda_loss_phase1") < seq.index("mmda_masked_mean_backward") \
        < seq.index("mmda_bert_embed_backward") < seq.index("mmda_adam_clip_step")
    with pytest.raises(MmdaError):
        tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels)     # bert inputs missing


def test_padded_row_buckets():
    """Row count a captured step is launched with (FusedTrainer.step): never below the real count,
    at most one granule above it, capped at B*T, and equal to it for full-length batches."""
    from mmda_b200.trainer import padded_rows, ROW_GRANULE
    assert ROW_GRANULE == 512
    assert padded_rows(12800, 256, 50) == 12800                  # full lengths: exact
    assert padded_rows(6500, 256, 50) == 6656
    assert padded_rows(6656, 256, 50) == 6656
    assert padded_rows(12799, 256, 50) == 12800                  # cap
    assert padded_rows(90, 8, 12) == 96                          # small batches: one bucket = the cap
    assert padded_rows(1, 8, 12, granule=4) == 4
    import random
    rnd = random.Random(0)
    for _ in range(200):
        B, T = rnd.randint(1, 300), rnd.randint(1, 60)
        n = rnd.randint(B, B * T)
        p = padded_rows(n, B, T)
        assert n <= p <= B * T and p - n < ROW_GRANULE
        assert p == B * T or p % ROW_GRANULE == 0


def test_optimizer_state_dict_round_trips_with_torch_adam(dryrun):
    """S1 boundary (src/solver.py:97-99, :219-220): the fused step's Adam state is written / read in
    torch.optim.Adam's own state_dict layout, in both directions."""
    from mmda_b200.trainer import FusedTrainer
    from mmda_b200._lib import MmdaError
    cfg = mosei_config(vocab_size=60, batch_size=4)
    torch.manual_seed(0)
    model = MISA(cfg)
    tr = FusedTrainer(model, lr=3e-4)
    skip = set(model.param_names_without_grad())
    # (1) reference -> fused: a torch Adam that took two steps over the same parameter list
    ref_params = [torch.nn.Parameter(p.detach().clone()) for p in model.parameters() if p.requires_grad]
    names = [n for n, p in model.named_parameters() if p.requires_grad]
    opt = torch.optim.Adam(ref_params, lr=5e-5)
    g = torch.Generator().manual_seed(1)
    for _ in range(2):
        for n, p in zip(names, ref_params):
            p.grad = None if n in skip else torch.randn(p.shape, generator=g)
        opt.step()
    sd = opt.state_dict()
    assert set(sd["state"]) == {i for i, n in enumerate(names) if n not in skip}
    tr.load_optimizer_state_dict(sd)
    assert tr.step_count == 2 and tr.lr == 5e-5
    assert dryrun.calls[-1] == "mmda_step_state_init"
    for i, n in enumerate(names):
        off, sz = tr.layout[n]
        if n in skip:
            assert off >= tr.n_active
            continue
        assert torch.equal(tr.m[off:off + sz].view(ref_params[i].shape), sd["state"][i]["exp_avg"])
        assert torch.equal(tr.v[off:off + sz].view(ref_params[i].shape), sd["state"][i]["exp_avg_sq"])
    # (2) fused -> reference: torch accepts it and sees the same tensors
    out = tr.optimizer_state_dict()
    assert set(out["state"]) == set(sd["state"]) and out["param_groups"][0]["lr"] == 5e-5
    opt2 = torch.optim.Adam([torch.nn.Parameter(p.detach().clone()) for p in ref_params], lr=1.0)
    opt2.load_state_dict(out)
    sd2 = opt2.state_dict()
    assert sd2["param_groups"][0]["lr"] == 5e-5
    for i in sd["state"]:
        assert float(sd2["state"][i]["step"]) == 2.0
        assert torch.equal(sd2["state"][i]["exp_avg"], sd["state"][i]["exp_avg"])
        assert torch.equal(sd2["state"][i]["exp_avg_sq"], sd["state"][i]["exp_avg_sq"])
    # (3) a fresh trainer has no per-parameter state, like a fresh torch optimizer
    tr0 = FusedTrainer(MISA(cfg))
    assert tr0.optimizer_state_dict()["state"] == {}
    # (4) anything but the reference's Adam settings is refused
    bad = opt.state_dict()
    bad["param_groups"][0]["weight_decay"] = 0.01
    with pytest.raises(MmdaError):
        tr.load_optimizer_state_dict(bad)


def test_bench_roofline_block_is_derived_from_the_live_plan():
    """bench.py's roofline object (SURVEY.md M2/M3): every figure follows from the batch, the live
    recurrence plan (mmda_lstm_tc_plan, a host-side query) and the measured launch time -- no
    literals tied to one shape (VERDICT r1 weak #9)."""
    import argparse
    import importlib.util
    import os
    from mmda_b200.synthetic import batch_for
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for B, T in ((256, 50), (512, 120)):
        cfg = mosei_config(vocab_size=100, batch_size=B)
        b = batch_for(cfg, seed=3, lengths="full", seq_len=T)
        args = argparse.Namespace(batch=B, lengths="full")
        ntok, H = B * T, 300
        ms = 0.60 * ntok / 12800          # a launch time in proportion to the C2 one
        kdur = {"mmda_lstm_tc_forward": ms / 2, "mmda_lstm_tc_backward": ms, "mmda_lstm_forward": 0.0}
        r = bench.roofline_block(cfg, b, kdur, {"sm_mhz": 1965.0}, args)
        assert r["kernel"].startswith("mmda_lstm_tc_backward")
        assert r["algorithmic_bytes"] == 2 * 10 * H * 4 * ntok              # M3: 10H words / token / direction
        assert r["algorithmic_flops"] == 2 * 2 * 4 * H * H * ntok
        assert r["binding_roofline"] == "fp32_fma" and r["bound"] == "fp32_fma"
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
        assert abs(r["frac"] - r["frac_of_binding_roofline"]) < 1e-9
        assert abs(r["peak"] - 148 * 128 * 2 * 1965.0e6 / 1e12) < 1e-9
        assert abs(r["achieved"] - r["algorithmic_flops"] / (ms * 1e-3) / 1e12) < 1e-9
        plan = r["plan"]
        assert plan["ctas"] == 2 * plan["slices"] * plan["groups"] <= 148
        assert plan["groups"] * plan["batch_tile"] >= B or plan["tiles"] * plan["batch_tile"] >= B
        assert r["hbm"]["frac"] < r["frac"] < 1.0
    assert bench.roofline_block(cfg, b, {"mmda_lstm_tc_backward": 0.0}, None, args) is None


def test_bench_clock_sampler_covers_short_runs(tmp_path, monkeypatch):
    """bench.py's nvidia-smi sampler: waits for the tool's (slow) start-up before the timed region,
    reports only samples taken after mark(), and still yields one for a region shorter than the
    sampling period; a box without nvidia-smi is reported, not fatal."""
    import importlib.util
    import os
    import stat
    import time
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nsleep 0.3\ni=0\nwhile true; do\n"
                    "if [ $i -lt 1 ]; then echo '0, 345, 1965, 150.0, Not Active, Not Active, Not Active, Not Active';\n"
                    "else echo '0, 1950, 1965, 600.0, Not Active, Not Active, Not Active, Active'; fi\n"
                    "i=$((i+1)); sleep 0.05\ndone\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod2", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setenv("PATH", f"{tmp_path}:{os.environ['PATH']}")
    c = bench.ClockSampler(0)
    c.start(); c.wait_first()
    assert len(c.rows) >= 1                      # the idle-clock sample before the region
    c.mark()
    time.sleep(0.25)
    out = c.stop()
    assert out["samples"] >= 2 and out["sm_mhz"] == 1950.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"]
    c = bench.ClockSampler(0)
    c.start(); c.wait_first(); c.mark()
    out = c.stop()                               # empty region: the next sample is taken
    assert out["samples"] >= 1 and out["sm_mhz"] == 1950.0
    monkeypatch.setenv("PATH", str(tmp_path / "nowhere"))
    c = bench.ClockSampler(0)
    c.start(); c.wait_first(); c.mark()
    assert c.stop()["reasons"] == ["nvidia-smi unavailable"]


def test_bench_dump_outputs(dryrun, tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy files of the step's losses and of the parameters and
    gradients in named_parameters() order; above DUMP_SAMPLE elements both are sampled at the same
    positions, and every run picks the same ones."""
    import importlib.util
    import numpy as np
    from mmda_b200.trainer import FusedTrainer
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod3", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    torch.manual_seed(0)
    model = MISA(mosei_config(vocab_size=60, batch_size=4))
    tr = FusedTrainer(model)
    tr.g_arena.copy_(2 * tr.p_arena + 1)
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).numpy()
    losses = torch.arange(8, dtype=torch.float32)

    def dump(name):
        bench.dump_outputs(str(tmp_path / name), tr, losses)
        return {k: np.load(tmp_path / name / (k + ".npy")) for k in ("losses", "params", "grads")}

    monkeypatch.setattr(bench, "DUMP_SAMPLE", flat.size)
    full = dump("full")
    assert all(v.dtype == np.float32 for v in full.values())
    assert np.array_equal(full["losses"], losses.numpy())
    assert np.array_equal(full["params"], flat) and np.array_equal(full["grads"], 2 * flat + 1)
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    a, b = dump("a"), dump("b")
    assert a["params"].shape == a["grads"].shape == (1000,)
    assert np.array_equal(a["grads"], 2 * a["params"] + 1)
    assert np.isin(a["params"], flat).all()
    assert all(np.array_equal(a[k], b[k]) for k in a)


@pytest.mark.parametrize("variant", [dict(rnncell="gru"), dict(use_cmd_sim=False),
                                     dict(rnncell="gru", use_cmd_sim=False, use_confidNet=True)])
def test_variant_kernel_sequences(dryrun, variant):
    """Host orchestration of the non-default variants (SURVEY.md row N4: GRU cells,
    src/models.py:39; adversarial branch, src/models.py:219-227 + src/solver.py:388-407) on the
    stubbed library: the right entry points are reached, level 1 and level 2."""
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=50, batch_size=6, **variant)
    torch.manual_seed(0)
    model = MISA(cfg).train()
    b = batch_for(cfg, seed=2, lengths="ragged", seq_len=5)
    scores, _ = model(*b.model_args())
    extra = model.domain_label_t.sum() if not cfg.use_cmd_sim else 0.0
    (scores.sum() + extra).backward()
    c1 = collections.Counter(dryrun.calls)
    gru = variant.get("rnncell") == "gru"
    assert c1["mmda_gru_forward" if gru else "mmda_lstm_forward"] == 6
    assert c1["mmda_gru_backward" if gru else "mmda_lstm_backward"] == 6
    assert (c1["mmda_gru_expand_weights"] > 0) == gru and (c1["mmda_gru_fold_grads"] > 0) == gru
    dryrun.calls.clear()
    tr = FusedTrainer(model)
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels)
    c2 = collections.Counter(dryrun.calls)
    assert (c2["mmda_loss_domain"] == 1) == (not cfg.use_cmd_sim)
    assert dryrun.calls[-1] == "mmda_adam_clip_step"
    # the discriminator exists (src/models.py:122-127) and trains only in the adversarial variant
    name = "discriminator.discriminator_layer_1.weight"
    assert (name in tr.layout) == (not cfg.use_cmd_sim)
    if name in tr.layout:
        assert tr.layout[name][0] < tr.n_active
