"""CPU-side checks of the optimizer choice (``config.optimizer``: Adam or RMSprop, reference
src/config.py:24-27, src/solver.py:97-99) and of the device-resident learning rate: config mapping,
refusals, torch.optim.RMSprop checkpoint interop, the restated RMSprop step (tests/optim_ref.py) against torch, and the
C-ABI calls of the fused step on a stubbed library."""
import numpy as np
import pytest
import torch

from mmda_b200 import MISA, mosei_config
from mmda_b200._lib import LIB, MmdaError


class _StubLib:
    """Records the C-ABI calls (name and arguments); lets the host orchestration run on CPU."""
    def __init__(self):
        self.calls = []

    def __call__(self, name, *args):
        self.calls.append((name, args))
        return 0

    def names(self):
        return [n for n, _ in self.calls]


@pytest.fixture
def dryrun(monkeypatch):
    import mmda_b200.engine as E
    stub = _StubLib()
    monkeypatch.setattr(E, "_DRYRUN", True)
    monkeypatch.setattr(LIB, "call", stub)
    monkeypatch.setattr(LIB, "raw", lambda name: (lambda *a: 4096))
    return stub


def test_config_optimizer_mapping():
    from mmda_b200.config import MisaConfig, optimizer_name
    assert MisaConfig().optimizer == "Adam"
    p = [torch.nn.Parameter(torch.zeros(2))]
    assert optimizer_name(torch.optim.Adam) == "Adam"
    assert optimizer_name(torch.optim.RMSprop) == "RMSprop"
    assert optimizer_name(torch.optim.Adam(p, lr=3e-4)) == "Adam"
    assert optimizer_name(torch.optim.RMSprop(p, lr=3e-4)) == "RMSprop"
    for s, want in (("Adam", "Adam"), ("RMSprop", "RMSprop"), ("rmsprop", "RMSprop"), ("adam", "Adam")):
        assert optimizer_name(s) == want
    for bad in (torch.optim.SGD, torch.optim.AdamW, "SGD", torch.optim.SGD(p, lr=0.1)):
        with pytest.raises(ValueError, match="supported: \\['Adam', 'RMSprop'\\]"):
            optimizer_name(bad)
    # an instance built with settings the fused step does not implement
    for bad in (torch.optim.RMSprop(p, momentum=0.9), torch.optim.RMSprop(p, centered=True),
                torch.optim.RMSprop(p, alpha=0.9), torch.optim.Adam(p, betas=(0.8, 0.999)),
                torch.optim.Adam(p, weight_decay=1e-2)):
        with pytest.raises(ValueError):
            optimizer_name(bad)


def test_trainer_refuses_unsupported_optimizer(dryrun):
    from mmda_b200.trainer import FusedTrainer
    for opt in (torch.optim.SGD, "Adagrad"):
        cfg = mosei_config(vocab_size=40, batch_size=4, optimizer=opt)
        with pytest.raises(MmdaError, match="Adam.*RMSprop"):
            FusedTrainer(MISA(cfg))
    for opt, want in ((torch.optim.RMSprop, "RMSprop"), ("RMSprop", "RMSprop"), (torch.optim.Adam, "Adam")):
        assert FusedTrainer(MISA(mosei_config(vocab_size=40, optimizer=opt))).optimizer == want

    class Bare:          # a reference-style config object without the field: Adam, as before
        pass
    cfg = mosei_config(vocab_size=40)
    bare = Bare()
    bare.__dict__.update(cfg.__dict__)
    del bare.__dict__["optimizer"]
    model = MISA(cfg)
    model.config = bare
    assert FusedTrainer(model).optimizer == "Adam"


def test_rmsprop_step_uses_rmsprop_kernel_and_device_lr(dryrun):
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=60, batch_size=6, optimizer="RMSprop")
    torch.manual_seed(0)
    tr = FusedTrainer(MISA(cfg).train())
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=5)
    tr.step(b.sentences, b.visual, b.acoustic, b.lengths, b.labels)
    names = dryrun.names()
    assert names[-1] == "mmda_rmsprop_clip_step" and "mmda_adam_clip_step" not in names
    assert names.index("mmda_step_state_set_lr") < names.index("mmda_step_state_advance_device_lr")
    assert "mmda_step_state_advance" not in names
    args = dryrun.calls[-1][1]
    # params, grads, square_avg (= the v arena), n, lr, clip, alpha, eps, grad_scale, state
    assert args[2] == tr.v.data_ptr() and args[3] == tr.n_active
    assert args[5:9] == (cfg.clip, 0.99, 1e-8, 1.0) and args[9] == tr.state.data_ptr()
    assert tr.state.numel() * tr.state.element_size() == 40


def test_learning_rate_written_to_the_device_only_when_it_changes(dryrun):
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=60, batch_size=6)
    torch.manual_seed(0)
    tr = FusedTrainer(MISA(cfg).train(), lr=1e-3)
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=5)
    args = (b.sentences, b.visual, b.acoustic, b.lengths, b.labels)
    schedule = [1e-3, 1e-3, 2e-3, 2e-3, 2e-3, 3e-3, 1e-3]
    written = []
    for lr in schedule:
        tr.lr = lr
        dryrun.calls.clear()
        tr.step(*args)
        sets = [a for n, a in dryrun.calls if n == "mmda_step_state_set_lr"]
        assert len(sets) <= 1
        written.append(sets[0][1] if sets else None)
        assert sets[0][0] == tr.state.data_ptr() if sets else True
    assert written == [1e-3, None, 2e-3, None, None, 3e-3, 1e-3]
    # forward_backward + optimizer_step (no step()) writes it too, once
    tr.lr = 5e-4
    dryrun.calls.clear()
    tr.forward_backward(*args)
    tr.optimizer_step()
    tr.forward_backward(*args)
    assert [a[1] for n, a in dryrun.calls if n == "mmda_step_state_set_lr"] == [5e-4]
    # a loaded checkpoint re-initialises the step state but keeps the device rate: the restored
    # rate is written before the next step, only if it differs
    sd = tr.optimizer_state_dict()
    sd["param_groups"][0]["lr"] = 7e-4
    tr.load_optimizer_state_dict(sd)
    assert dryrun.names()[-1] == "mmda_step_state_init"
    dryrun.calls.clear()
    tr.step(*args)
    assert [a[1] for n, a in dryrun.calls if n == "mmda_step_state_set_lr"] == [7e-4]


def _trained_rmsprop(model, lr, steps=2, seed=1):
    skip = set(model.param_names_without_grad())
    names = [n for n, p in model.named_parameters() if p.requires_grad]
    ref = [torch.nn.Parameter(p.detach().clone()) for p in model.parameters() if p.requires_grad]
    opt = torch.optim.RMSprop(ref, lr=lr)
    g = torch.Generator().manual_seed(seed)
    for _ in range(steps):
        for n, p in zip(names, ref):
            p.grad = None if n in skip else torch.randn(p.shape, generator=g)
        opt.step()
    return opt, names, ref, skip


def test_rmsprop_state_dict_round_trips_with_torch(dryrun):
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=60, batch_size=4, optimizer=torch.optim.RMSprop)
    torch.manual_seed(0)
    model = MISA(cfg)
    tr = FusedTrainer(model, lr=3e-4)
    assert tr.optimizer_state_dict()["state"] == {}
    # (1) torch -> fused
    opt, names, ref, skip = _trained_rmsprop(model, 5e-5)
    sd = opt.state_dict()
    assert set(sd["state"]) == {i for i, n in enumerate(names) if n not in skip}
    tr.m.fill_(3.0)
    tr.load_optimizer_state_dict(sd)
    assert tr.step_count == 2 and tr.lr == 5e-5
    assert dryrun.names()[-1] == "mmda_step_state_init"
    assert float(tr.m.abs().max()) == 0.0                  # RMSprop leaves the m arena unused
    for i, n in enumerate(names):
        off, sz = tr.layout[n]
        if n in skip:
            assert off >= tr.n_active
            continue
        assert torch.equal(tr.v[off:off + sz].view(ref[i].shape), sd["state"][i]["square_avg"])
    # (2) fused -> torch: same keys as torch writes them, and torch loads it
    out = tr.optimizer_state_dict()
    assert list(out["param_groups"][0]) == list(sd["param_groups"][0])
    assert {k: v for k, v in out["param_groups"][0].items() if k != "params"} == \
        {k: v for k, v in sd["param_groups"][0].items() if k != "params"}
    assert set(out["state"]) == set(sd["state"])
    for i in sd["state"]:
        assert list(out["state"][i]) == list(sd["state"][i]) == ["step", "square_avg"]
    opt2 = torch.optim.RMSprop([torch.nn.Parameter(p.detach().clone()) for p in ref], lr=1.0)
    opt2.load_state_dict(out)
    sd2 = opt2.state_dict()
    assert sd2["param_groups"][0]["lr"] == 5e-5
    for i in sd["state"]:
        assert float(sd2["state"][i]["step"]) == 2.0
        assert torch.equal(sd2["state"][i]["square_avg"], sd["state"][i]["square_avg"])
    # (3) settings the fused step does not implement are refused
    for key, val in (("alpha", 0.9), ("eps", 1e-6), ("momentum", 0.9), ("centered", True),
                     ("weight_decay", 0.01)):
        bad = opt.state_dict()
        bad["param_groups"][0][key] = val
        with pytest.raises(MmdaError, match="RMSprop"):
            tr.load_optimizer_state_dict(bad)


def test_cross_loading_adam_and_rmsprop_states_is_refused(dryrun):
    from mmda_b200.trainer import FusedTrainer
    torch.manual_seed(0)
    model = MISA(mosei_config(vocab_size=60, batch_size=4))
    rms_opt, names, ref, skip = _trained_rmsprop(model, 1e-4)
    adam = torch.optim.Adam(ref, lr=1e-4)
    for n, p in zip(names, ref):
        p.grad = None if n in skip else torch.ones_like(p)
    adam.step()
    for opt_name, foreign in (("Adam", rms_opt.state_dict()), ("RMSprop", adam.state_dict())):
        tr = FusedTrainer(MISA(mosei_config(vocab_size=60, batch_size=4, optimizer=opt_name)))
        with pytest.raises(MmdaError, match=f"config.optimizer is {opt_name}"):
            tr.load_optimizer_state_dict(foreign)
        assert tr.step_count == 0
        # a fresh foreign optimizer (no per-parameter state yet) is refused by its group keys
        fresh = (torch.optim.RMSprop if opt_name == "Adam" else torch.optim.Adam)(ref, lr=1e-4)
        with pytest.raises(MmdaError, match="config.optimizer"):
            tr.load_optimizer_state_dict(fresh.state_dict())
        # and its own optimizer's state still loads
        own = (adam if opt_name == "Adam" else rms_opt).state_dict()
        tr.load_optimizer_state_dict(own)
        assert tr.step_count == (1 if opt_name == "Adam" else 2)


def test_rmsprop_clip_step_matches_torch():
    """optim_ref.rmsprop_clip_step (the fp64 restatement the GPU tests use) against
    clip_grad_value_ + torch.optim.RMSprop, with gradients past the clip bound and exact zeros."""
    import optim_ref as E
    g0 = torch.Generator().manual_seed(3)
    n = 4099
    p0 = torch.randn(n, generator=g0, dtype=torch.float64)
    pt = p0.clone().requires_grad_(True)
    opt = torch.optim.RMSprop([pt], lr=1e-2)
    pn, v = p0.numpy().copy(), np.zeros(n)
    for step in range(6):
        gr = torch.randn(n, generator=g0, dtype=torch.float64) * 2
        gr[step::7] = 0.0
        pt.grad = gr.clone()
        torch.nn.utils.clip_grad_value_([pt], 1.0)
        opt.step()
        pn, v = E.rmsprop_clip_step(pn, gr.numpy(), v, 1e-2, 1.0)
        np.testing.assert_allclose(v, opt.state[pt]["square_avg"].numpy(), rtol=1e-13, atol=1e-300)
        np.testing.assert_allclose(pn, pt.detach().numpy(), rtol=1e-13, atol=1e-15)
    # grad_scale multiplies before the clip
    g = np.array([3.0, -0.4, 0.0, 1.5])
    p1, v1 = E.rmsprop_clip_step(np.zeros(4), g, np.zeros(4), 1.0, 1.0, grad_scale=0.5)
    gc = np.array([1.0, -0.2, 0.0, 0.75])
    np.testing.assert_allclose(v1, 0.01 * gc * gc)
    np.testing.assert_allclose(p1, -gc / (np.sqrt(0.01 * gc * gc) + 1e-8))


def test_reference_optimizer_follows_config():
    """optim_ref.reference_optimizer: what solver.py:97-99 builds from config.optimizer."""
    from optim_ref import reference_optimizer
    model = torch.nn.Linear(3, 2)
    model.bias.requires_grad = False
    for opt, cls in ((None, torch.optim.Adam), ("Adam", torch.optim.Adam), ("RMSprop", torch.optim.RMSprop),
                     (torch.optim.RMSprop, torch.optim.RMSprop)):
        cfg = mosei_config(vocab_size=10) if opt is None else mosei_config(vocab_size=10, optimizer=opt)
        o = reference_optimizer(model, cfg)
        assert type(o) is cls and o.param_groups[0]["lr"] == cfg.learning_rate
        assert o.param_groups[0]["params"] == [model.weight]
