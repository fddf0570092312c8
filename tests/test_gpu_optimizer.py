"""The optimizer step on the device: the fused clip + RMSprop kernel against fp64, the whole fused
step with ``config.optimizer = RMSprop`` against torch.optim.RMSprop, and learning-rate schedules
under CUDA-graph replay (the rate lives in the device step state).  Run with ``-m gpu`` on a B200.

Bounds are scale-relative (max |a-b| / max |ref|).  Every check is written to
test_reports/optimizer.txt with its error."""
import os

import numpy as np
import pytest
import torch

from helpers import ROOT, load_small, max_rel, small_batch, small_cfg, state_from_npz

pytestmark = pytest.mark.gpu

ROWS = []          # (test, check, err, bound, ok)


def _check(test, name, err, bound, ok=None):
    ok = err <= bound if ok is None else ok
    ROWS.append((test, name, err, bound, ok))
    out = os.path.join(ROOT, "test_reports")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "optimizer.txt"), "w") as f:
        for t, n, e, b, k in ROWS:
            f.write(f"{'ok  ' if k else 'FAIL'} {t:28s} {n:64s} err={e:.3e} bound={b:.1e}\n")
    return ok


def _finish(test):
    rows = [r for r in ROWS if r[0] == test]
    worst = max(rows, key=lambda r: r[2] / r[3] if r[3] else (0.0 if r[4] else float("inf")))
    bad = [r for r in rows if not r[4]]
    assert not bad, "\n".join(f"{n}: err={e:.3e} > {b:.1e}" for _, n, e, b, _ in bad[:30])
    return worst


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return torch.device("cuda:0")


def _state(k, lr=None):
    from mmda_b200.engine import _ptr
    st = torch.zeros(5, dtype=torch.float64, device="cuda")
    k._c("mmda_step_state_init", _ptr(st), 0, 0.9, 0.999)
    if lr is not None:
        k._c("mmda_step_state_set_lr", _ptr(st), lr)
    return st


# ------------------------------------------------------------------------------------------
# the kernel
# ------------------------------------------------------------------------------------------
BIG = 148 * 8 * 256 * 4 + 4099        # past one grid-stride sweep of the capped grid, n % 4 == 3


def test_rmsprop_kernel_matches_fp64(dev):
    """mmda_rmsprop_clip_step over 10 consecutive steps against the fp64 restatement in
    tests/optim_ref.py: gradients past +-clip and exact zeros, grad_scale 1 and 0.5, the float4 body,
    the scalar tail and the grid-stride loop.  The learning rate read from the device step state
    gives the same bits as the one passed by argument, and nothing past n is written."""
    from mmda_b200.engine import Kernels, _ptr
    from optim_ref import rmsprop_clip_step
    k = Kernels(); k.bind_stream()
    gen = torch.Generator().manual_seed(4)
    lr, clip, alpha, eps = 1e-2, 1.0, 0.99, 1e-8
    T = "rmsprop kernel"
    for n in (1, 3, 4, 5, 1023, BIG):
        for gs in (1.0, 0.5):
            p0 = torch.randn(n, generator=gen) * 0.1
            bufs = {}
            for path in ("host", "device"):
                p = torch.full((n + 8,), 7.0, device=dev); p[:n] = p0.to(dev)
                v = torch.full((n + 8,), 7.0, device=dev); v[:n] = 0.0
                bufs[path] = (p, v)
            st = _state(k, lr)
            p64, v64 = p0.double().numpy(), np.zeros(n)
            for step in range(10):
                gr = torch.randn(n, generator=gen) * 1.5
                gr[step % 7::7] = 0.0
                g = torch.full((n + 8,), 5.0, device=dev); g[:n] = gr.to(dev)
                for path, (p, v) in bufs.items():
                    if path == "host":
                        k._c("mmda_rmsprop_clip_step", _ptr(p), _ptr(g), _ptr(v), n, lr, clip, alpha,
                             eps, gs, None)
                    else:       # a wrong host lr: the device one must win
                        k._c("mmda_rmsprop_clip_step", _ptr(p), _ptr(g), _ptr(v), n, 123.0, clip,
                             alpha, eps, gs, _ptr(st))
                p64, v64 = rmsprop_clip_step(p64, gr.double().numpy(), v64, lr, clip, alpha, eps, gs)
                (ph, vh), (pd, vd) = bufs["host"], bufs["device"]
                assert torch.equal(ph, pd) and torch.equal(vh, vd), (n, gs, step)
            p, v = bufs["host"]
            pc, vc = p.cpu().double(), v.cpu().double()
            tag = f"n={n} grad_scale={gs}"
            _check(T, f"{tag} square_avg after 10 steps", max_rel(vc[:n], torch.from_numpy(v64)), 1e-5)
            _check(T, f"{tag} accumulated update p - p0", max_rel(pc[:n] - p0.double(),
                                                               torch.from_numpy(p64) - p0.double()), 1e-5)
            _check(T, f"{tag} nothing written past n", 0.0, 0.0,
                   bool((pc[n:] == 7.0).all() and (vc[n:] == 7.0).all()))
    worst = _finish(T)
    print("worst row:", worst)


def test_constant_lr_adam_is_bit_identical_to_host_lr_path(dev):
    """At a constant learning rate the device-lr advance gives Adam the same step sizes as the
    host-lr advance, bit for bit: parameters, moments and the whole step state agree exactly."""
    from mmda_b200.engine import Kernels, _ptr
    k = Kernels(); k.bind_stream()
    gen = torch.Generator().manual_seed(6)
    n = 100003
    for lr in (1e-4, 3e-3, 0.1):
        st_h, st_d = _state(k), _state(k, lr)
        p0 = torch.randn(n, generator=gen)
        arenas = {s: [p0.to(dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)] for s in ("h", "d")}
        for step in range(1, 8):
            g = (torch.randn(n, generator=gen) * 2).to(dev)
            k._c("mmda_step_state_advance", _ptr(st_h), lr, 0.9, 0.999)
            k._c("mmda_step_state_advance_device_lr", _ptr(st_d), 0.9, 0.999)
            for s, st in (("h", st_h), ("d", st_d)):
                p, m, v = arenas[s]
                k._c("mmda_adam_clip_step", _ptr(p), _ptr(g), _ptr(m), _ptr(v), n, step, lr, 1.0,
                     0.9, 0.999, 1e-8, 1.0, _ptr(st))
            assert torch.equal(st_h[:4], st_d[:4]), (lr, step)
            for a, b in zip(arenas["h"], arenas["d"]):
                assert torch.equal(a, b), (lr, step)
    # and the trainer: its step state after five steps at a constant rate (two eager, one
    # captured, two replayed) equals five host-lr advances of a fresh state
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=300, batch_size=32)
    b = batch_for(cfg, seed=3, lengths="full", seq_len=10)
    torch.manual_seed(3)
    tr = FusedTrainer(MISA(cfg).to(dev).train(), lr=3e-4)
    ref = _state(k)
    for _ in range(5):
        tr.step(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths, b.labels.to(dev))
        k.bind_stream()
        k._c("mmda_step_state_advance", _ptr(ref), 3e-4, 0.9, 0.999)
    torch.cuda.synchronize()
    assert tr._graph is not None
    assert torch.equal(tr.state[:4], ref[:4])
    tr.close()


# ------------------------------------------------------------------------------------------
# the whole fused step
# ------------------------------------------------------------------------------------------
def test_whole_step_rmsprop_matches_torch(dev):
    """config.optimizer = RMSprop, eval mode, three steps against the oracle driving
    torch.optim.RMSprop in fp64: the losses of every step, and the clip + RMSprop update on every
    element from the device gradients (RMSprop's first step, like Adam's, turns a rounding-level
    gradient into a +-10*lr update, so the post-step parameters are compared against the update of
    the device's own gradients; the gradients themselves are pinned by test_gpu_parity)."""
    from mmda_b200 import MISA
    from mmda_b200.synthetic import Batch
    from mmda_b200.trainer import FusedTrainer, LOSS_NAMES
    from optim_ref import reference_optimizer, rmsprop_clip_step
    from oracle.misa_oracle import OracleMISA, oracle_step
    T = "whole step rmsprop"
    z, meta = load_small("small_ragged")
    cfg = small_cfg(meta, optimizer="RMSprop")
    state, batch = state_from_npz(z), small_batch(z)
    ref = OracleMISA(cfg)
    ref.load_state_dict(state)
    ref = ref.double().eval()
    opt = reference_optimizer(ref, cfg)
    assert isinstance(opt, torch.optim.RMSprop)
    b64 = Batch(batch.sentences, batch.visual.double(), batch.acoustic.double(), batch.labels.double(),
                batch.lengths, batch.bert_sent, batch.bert_sent_type, batch.bert_sent_mask)
    model = MISA(cfg)
    model.load_state_dict(state)
    model = model.to(dev).eval()
    tr = FusedTrainer(model, use_graph=False)
    assert tr.optimizer == "RMSprop"
    na = tr.n_active
    args = (batch.sentences.to(dev), batch.visual.to(dev), batch.acoustic.to(dev), batch.lengths,
            batch.labels.to(dev))
    for step in range(1, 4):
        _, L, _ = oracle_step(ref, b64, cfg, opt)
        losses = tr.forward_backward(*args)[:6].cpu()
        for i, kk in enumerate(LOSS_NAMES):
            _check(T, f"step {step} loss {kk}", max_rel(losses[i], torch.as_tensor(L[kk]).detach()), 1e-5)
        g = tr.g_arena[:na].cpu().double().numpy()
        p0 = tr.p_arena[:na].cpu().double().numpy()
        v0 = tr.v[:na].cpu().double().numpy()
        tr.optimizer_step()
        p_exp, v_exp = rmsprop_clip_step(p0, g, v0, cfg.learning_rate, cfg.clip)
        _check(T, f"step {step} params after clip + RMSprop (every element)",
               max_rel(tr.p_arena[:na].cpu(), torch.from_numpy(p_exp)), 2e-6)
        _check(T, f"step {step} square_avg (every element)",
               max_rel(tr.v[:na].cpu(), torch.from_numpy(v_exp)), 1e-5)
    _check(T, "Adam moments untouched", 0.0, 0.0, float(tr.m.abs().max()) == 0.0)
    assert tr.step_count == 3
    _finish(T)


def _warmup_lr(i, base):
    return base * min(1.0, (i + 1) / 8.0)          # linear warm-up over 8 steps


@pytest.mark.parametrize("optimizer", ["Adam", "RMSprop"])
def test_lr_schedule_replays_one_graph(dev, optimizer, monkeypatch):
    """A C2-shaped step (MOSEI shapes, batch 256, seq 50, full lengths, train mode) with a learning
    rate that changes every step: one capture, every later step a replay, and the same trajectory
    as eager launches of the same schedule.  The device step state (step counter, Adam bias
    corrections, learning rate) is bit-identical to the eager run's after every step; losses and
    parameters agree up to the rounding noise of the atomic reductions (see
    test_cuda_graph_replay_equals_eager).  On one replayed step the update must be the one of
    that step's learning rate, and clearly not the previous step's."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200 import trainer as TR
    from mmda_b200.synthetic import batch_for
    from optim_ref import rmsprop_clip_step
    from oracle.explicit import adam_clip_step
    T = f"lr schedule {optimizer}"
    cfg = mosei_config(vocab_size=2000, batch_size=256, optimizer=optimizer)
    base = cfg.learning_rate           # the warm-up ends at the reference's default rate
    batches = [batch_for(cfg, seed=60 + i, lengths="full", seq_len=50) for i in range(3)]
    dbat = [(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths, b.labels.to(dev))
            for b in batches]
    captures = []
    real_graph = torch.cuda.graph

    def counting_graph(*a, **kw):
        captures.append(1)
        return real_graph(*a, **kw)
    monkeypatch.setattr(torch.cuda, "graph", counting_graph)
    steps, probe = 10, 5
    res = {}
    for mode in (False, True):
        captures.clear()
        torch.manual_seed(5)
        model = MISA(cfg)
        for n, p in model.named_parameters():
            if "weight_hh" in n:
                torch.nn.init.orthogonal_(p)
        tr = TR.FusedTrainer(model.to(dev).train(), use_graph=mode)
        eager = []
        orig = tr._eager_step
        tr._eager_step = lambda *a, **kw: (eager.append(1), orig(*a, **kw))[1]
        Ls, states = [], []
        for i in range(steps):
            tr.lr = _warmup_lr(i, base)
            if mode and i == probe:
                before = [t[:tr.n_active].cpu().double().numpy() for t in (tr.p_arena, tr.m, tr.v)]
            Ls.append(tr.step(*dbat[i % 3])[:6].clone())
            states.append(tr.state.clone())
            if mode and i == probe:
                g = tr.g_arena[:tr.n_active].cpu().double().numpy()
                after = tr.p_arena[:tr.n_active].cpu().double().numpy()
        torch.cuda.synchronize()
        if mode:
            _check(T, "captures (exactly one)", float(len(captures)), 1.0, len(captures) == 1)
            # two eager warm-up steps, the step traced by the capture, then replays only
            _check(T, f"eager steps {len(eager)} = 2 warm-up + 1 captured, {steps - 3} later replays",
                   0.0, 0.0, len(eager) == 3 and len(tr._graphs) == 1)
        else:
            assert len(eager) == steps and not captures
        res[mode] = (torch.stack(Ls).cpu(), tr.p_arena[:tr.n_active].cpu(), torch.stack(states).cpu(),
                     tr.step_count)
        tr.close()
    assert res[True][3] == res[False][3] == steps
    _check(T, "device step state after every step (bit-identical)", 0.0, 0.0,
           torch.equal(res[True][2], res[False][2]))
    _check(T, "losses over the schedule vs eager", max_rel(res[True][0], res[False][0]), 1e-5)
    # atomics make rounding-level gradient elements differ run to run, and Adam / RMSprop turn one
    # into a full-size update of noise sign: up to lr (Adam) or 10*lr (RMSprop) per step
    per_step = (1.0 if optimizer == "Adam" else 10.0) * base
    dp = float((res[True][1] - res[False][1]).abs().max())
    _check(T, "parameters after the schedule vs eager: max |delta| <= 2*noise floor*steps",
           dp, 2 * per_step * steps)
    # the replayed step used ITS learning rate
    p0, m0, v0 = before
    lr_i, lr_prev = _warmup_lr(probe, base), _warmup_lr(probe - 1, base)

    def upd(lr):
        if optimizer == "Adam":
            return adam_clip_step(p0, g, m0, v0, probe + 1, lr, cfg.clip)[0] - p0
        return rmsprop_clip_step(p0, g, v0, lr, cfg.clip)[0] - p0
    got = torch.from_numpy(after - p0)
    _check(T, f"replayed step {probe + 1}: update of lr={lr_i:.3e}", max_rel(got, torch.from_numpy(upd(lr_i))), 1e-2)
    e_prev = max_rel(got, torch.from_numpy(upd(lr_prev)))
    _check(T, f"replayed step {probe + 1}: NOT the update of lr={lr_prev:.3e}", e_prev, 0.1, e_prev > 0.1)
    _finish(T)


def test_rmsprop_checkpoint_resume_matches_uninterrupted_run(dev):
    """test_checkpoint_resume_matches_uninterrupted_run with config.optimizer = RMSprop: model +
    optimizer state saved after step 3 (passed through torch.optim.RMSprop.load_state_dict, as the
    reference's checkpoint files hold it), loaded into a fresh model / trainer and resumed: steps
    4..6 in train mode match the uninterrupted run."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    T = "rmsprop checkpoint resume"
    cfg = mosei_config(vocab_size=300, batch_size=32, use_confidNet=True, optimizer=torch.optim.RMSprop)
    batches = [batch_for(cfg, seed=90 + i, lengths="ragged", seq_len=10) for i in range(6)]

    def step(tr, b):
        return tr.step(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths,
                       b.labels.to(dev))[:6].clone().cpu()

    torch.manual_seed(11)
    model = MISA(cfg).to(dev).train()
    tr = FusedTrainer(model, use_graph=False)
    for b in batches[:3]:
        step(tr, b)
    ckpt_model = {k: v.detach().clone().cpu() for k, v in model.state_dict().items()}
    ckpt_optim = tr.optimizer_state_dict()
    rms = torch.optim.RMSprop([p for p in model.parameters() if p.requires_grad], lr=1.0)
    rms.load_state_dict(ckpt_optim)
    ckpt_optim = rms.state_dict()
    assert all(set(s) == {"step", "square_avg"} for s in ckpt_optim["state"].values())
    ref = [step(tr, b) for b in batches[3:]]
    ref_params = tr.p_arena[:tr.n_active].clone().cpu()

    torch.manual_seed(12)
    model2 = MISA(cfg).to(dev).train()
    model2.load_state_dict(ckpt_model)
    tr2 = FusedTrainer(model2, use_graph=False)
    tr2.load_optimizer_state_dict(ckpt_optim)
    assert tr2.step_count == 3 and tr2.lr == cfg.learning_rate
    got = [step(tr2, b) for b in batches[3:]]
    _check(T, "losses of steps 4..6", max_rel(torch.stack(got), torch.stack(ref)), 1e-5)
    dp = float((tr2.p_arena[:tr2.n_active].cpu() - ref_params).abs().max())
    # noise floor of three RMSprop steps on rounding-level gradient elements: 2 * 10*lr * steps
    _check(T, "parameters after step 6: max |delta| <= 2*10*lr*steps", dp, 2 * 10 * cfg.learning_rate * 3)
    _finish(T)
