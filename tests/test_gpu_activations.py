"""ELU / Hardshrink / Hardtanh / RReLU on the B200 (run with ``-m gpu``): the epilogue and backward
primitives against fp64 torch, the training-mode RReLU kernels (slope distribution, redraw in the
backward, device step counter), and the whole model at level 1 and level 2 against the fp64
oracle, RReLU's random slopes included.

Branch alignment: each new activation has a kink or a jump (0 for ELU / RReLU, +-0.5 for
Hardshrink, +-1 for Hardtanh).  A pre-activation within fp32 rounding of it may land on either side
on the device and in the fp64 oracle; where the two disagree and the oracle's pre-activation is
within 1e-5 of the threshold, the oracle's is moved onto the device's side (read from the stored
activation output A) and the count is reported, as the ReLU kink rule of test_gpu_parity.py does.
"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from helpers import GOLDEN, load_small, small_batch, small_cfg, state_from_npz
from test_gpu_parity import ADV_ATTRS, ATTR_CHECK, Checks, _run_level1, _to

pytestmark = pytest.mark.gpu
NEW = ("elu", "hardshrink", "hardtanh", "rrelu")
TORCH = {"elu": nn.ELU, "hardshrink": nn.Hardshrink, "hardtanh": nn.Hardtanh, "rrelu": nn.RReLU}
R_LO, R_HI = np.float32(1 / 8), np.float32(1 / 3)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return torch.device("cuda:0")


def _ref(name, x):
    """torch's eval-mode function (fp64 in, fp64 out)"""
    return TORCH[name]().eval()(x)


def _kernels():
    from mmda_b200.engine import Kernels
    k = Kernels()
    k.bind_stream()
    return k


def _slopes(k, rows, cols, seed, sid, seed_dev=None, dev="cuda"):
    """the slopes mmda_rrelu_forward draws: its output on a tensor of -1s, negated"""
    x = -torch.ones(rows, cols, device=dev)
    k.rrelu(x, seed, sid, seed_dev)
    return -x


# ------------------------------------------------------------------------------------------
# primitives
# ------------------------------------------------------------------------------------------
def _edge_values():
    e = [0.0, -0.0, 0.5, -0.5, 1.0, -1.0, -10.0, 10.0, 1e-30, -1e-30]
    for t in (0.5, -0.5, 1.0, -1.0, 0.0):
        t32 = torch.tensor(t, dtype=torch.float32)
        e += [float(torch.nextafter(t32, torch.tensor(9.0))), float(torch.nextafter(t32, torch.tensor(-9.0)))]
    grid = torch.linspace(-10, 10, 4001, dtype=torch.float32).tolist()
    return torch.tensor(e + grid, dtype=torch.float32)


@pytest.mark.parametrize("name", NEW)
def test_epilogue_and_backward_against_fp64(dev, name):
    from mmda_b200.config import ACTIVATIONS
    act = ACTIVATIONS[name]
    k = _kernels()
    g = torch.Generator().manual_seed(11)
    C = Checks(f"act_{name}")
    # exact edge points through mmda_act_forward / mmda_act_backward (-0.0 kept)
    x = _edge_values()
    y = x.clone().view(1, -1).to(dev)
    k.act(y, act)
    dy = torch.randn(1, x.numel(), generator=g).to(dev)
    dx = dy.clone()
    k.act_bwd(dx, y, act)
    xd = x.double().view(1, -1).requires_grad_(True)
    yr = _ref(name, xd)
    yr.backward(dy.double().cpu())
    C.add("act_forward edges", y, yr, 1e-6)
    C.add("act_backward edges", dx, xd.grad, 1e-6)
    # the derivative at the kinks is torch's (0 / 1 / the slope, not a neighbouring piece's)
    ratio = (dx.double() / dy.double()).cpu()[0]
    ref_ratio = (xd.grad / dy.double().cpu())[0]
    for i in range(10):
        C.flag(f"derivative at {x[i].item()!r}: {ratio[i].item():.8f} vs torch {ref_ratio[i].item():.8f}",
               abs(float(ratio[i] - ref_ratio[i])) < 1e-6)
    # the same edge points through mmda_sgemm's epilogue: K = 1, x * 1 + no bias is exact
    M = x.numel()
    A = x.view(M, 1).to(dev)
    Bm = torch.ones(1, 64, device=dev)
    out = torch.empty(M, 64, device=dev)
    k.gemm(A, Bm, out, act=act)
    ref = _ref(name, x.double().view(M, 1).expand(M, 64).clone())
    nz = x != 0           # x * 1 + 0 turns -0.0 into +0.0
    C.add("sgemm epilogue, edge points", out[nz.to(dev)], ref[nz], 1e-6)
    # a real product: the epilogue against torch on the same fp32 pre-activation (same launch
    # without the epilogue), and both against the fp64 product
    for (M, N, K) in [(256, 128, 64), (300, 128, 500), (37, 129, 33)]:
        Am = (torch.randn(M, K, generator=g) * 3 / K ** 0.5).to(dev)
        W = torch.randn(N, K, generator=g).to(dev)
        b = torch.randn(N, generator=g).to(dev)
        z = torch.empty(M, N, device=dev)
        o = torch.empty(M, N, device=dev)
        k.linear(Am, W, b, z)
        k.linear(Am, W, b, o, act=act)
        C.add(f"sgemm epilogue {M}x{N}x{K}", o, _ref(name, z.double().cpu()), 1e-6)
        C.add(f"sgemm pre-activation {M}x{N}x{K}", z, Am.double() @ W.double().t() + b.double(), 1e-5)
        d = torch.randn(M, N, generator=g).to(dev)
        dd = d.clone()
        k.act_bwd(dd, o, act)
        zd = z.double().cpu().requires_grad_(True)
        _ref(name, zd).backward(d.double().cpu())
        C.add(f"act_backward {M}x{N}", dd, zd.grad, 1e-6)
    C.finish()


def test_rrelu_training_kernel(dev):
    from scipy import stats
    k = _kernels()
    seed, sid = 0x1234_5678_9ABC, 9
    # 10^6 slopes: all in [1/8, 1/3], uniform (KS)
    r = _slopes(k, 1000, 1000, seed, sid)
    rc = r.cpu().numpy().ravel()
    assert rc.min() >= R_LO and rc.max() <= R_HI, (rc.min(), rc.max())
    ks = stats.kstest(rc.astype(np.float64), "uniform", args=(1 / 8, 1 / 3 - 1 / 8))
    assert ks.pvalue > 1e-3, ks
    # the backward with dy = 1 returns the forward's r bit for bit, at x = -1, at 0 and at -0.0
    for fill in (-1.0, 0.0, -0.0):
        x = torch.full((1000, 1000), fill, device=dev)
        k.rrelu(x, seed, sid)
        g1 = torch.ones_like(x)
        k.rrelu_bwd(g1, x, seed, sid)
        assert torch.equal(g1, r), fill
    # y = x * r to fp32 rounding (one multiplication), x > 0 passes through
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1000, 1000, generator=g).to(dev)
    y = x.clone()
    k.rrelu(y, seed, sid)
    assert torch.equal(y, torch.where(x > 0, x, x * r))
    # a pitched view draws index row * cols + col, like the contiguous tensor, and leaves the rest
    wide = torch.full((1000, 1500), -1.0, device=dev)
    k.rrelu(wide[:, :1000], seed, sid)
    assert torch.equal(-wide[:, :1000], r) and bool((wide[:, 1000:] == -1).all())
    # same (seed, stream, step): the same bits; the next step or another stream id: other slopes
    assert torch.equal(_slopes(k, 1000, 1000, seed, sid), r)
    step = torch.tensor([41, 0], dtype=torch.int64, device=dev)
    r41 = _slopes(k, 1000, 1000, seed, sid, step)
    step[0] = 42
    r42 = _slopes(k, 1000, 1000, seed, sid, step)
    assert float((r41 != r42).float().mean()) > 0.99
    assert float((_slopes(k, 1000, 1000, seed, sid + 1) != r).float().mean()) > 0.99
    # the device counter path equals the host seed that folds the same counter in
    host = (seed + 42 * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    assert torch.equal(_slopes(k, 1000, 1000, host, sid), r42)
    # the backward with the device counter redraws the forward's slopes
    x = torch.full((1000, 1000), -1.0, device=dev)
    k.rrelu(x, seed, sid, step)
    g1 = torch.ones_like(x)
    k.rrelu_bwd(g1, x, seed, sid, step)
    assert torch.equal(g1, r42)


# ------------------------------------------------------------------------------------------
# whole model
# ------------------------------------------------------------------------------------------
def _align(z, dev_out, kind, info, key):
    """move oracle pre-activations within 1e-5 of the threshold onto the device's side"""
    if kind == "hardshrink":
        mine, theirs, thr = dev_out != 0, z.abs() > 0.5, 0.5
    elif kind == "hardtanh":
        mine, theirs, thr = dev_out.abs() == 1, z.abs() >= 1, 1.0
    else:
        mine, theirs, thr = dev_out > 0, z > 0, 0.0
    flips = mine != theirs
    info[f"{key} flips"] = int(flips.sum())
    if not bool(flips.any()):
        return z
    info[f"{key} max|z-thr| at flips"] = float((z.abs() - thr).abs()[flips].max().detach()) if thr else \
        float(z[flips].abs().max().detach())
    ok = flips & ((z.abs() - thr).abs() < 1e-5 if thr else z.abs() < 1e-5)
    s = torch.where(z < 0, -torch.ones_like(z), torch.ones_like(z))
    if kind == "hardshrink":
        tgt = torch.where(mine, s * (0.5 + 1e-12), s * 0.5)
    elif kind == "hardtanh":
        tgt = torch.where(mine, s * 1.0, s * (1.0 - 1e-12))
    else:
        tgt = torch.where(mine, torch.full_like(z, 1e-12), torch.full_like(z, -1e-12))
    return z + (torch.where(ok, tgt, z) - z).detach()


class _Site(nn.Module):
    """one activation site of the fp64 oracle: branch alignment against the device's output, then
    torch's function, or (training-mode RReLU) a multiply by the device's slopes"""

    def __init__(self, name, dev_out, info, key, slopes=None):
        super().__init__()
        self.name, self.dev_out, self.info, self.key, self.slopes = name, dev_out, info, key, slopes

    def forward(self, z):
        kind = self.name if self.name in ("hardshrink", "hardtanh") else "sign"
        z = _align(z, self.dev_out, kind, self.info, self.key)
        if self.slopes is not None:
            return torch.where(z > 0, z, z * self.slopes)
        return _ref(self.name, z)


def _oracle64(cfg, name, state, batch, eng, slopes=None):
    """fp64 oracle step with every activation site replaced by a _Site aligned to the engine's
    last forward (A, DHpre, and the fusion FFN ReLU as test_gpu_parity.py aligns it)"""
    from mmda_b200.synthetic import Batch
    from oracle.misa_oracle import OracleMISA, oracle_step
    B, d = batch.lengths.numel(), cfg.hidden_size
    info = {}
    m = OracleMISA(cfg)
    m.load_state_dict(state)
    m = m.double().eval()
    A = eng.ws["A"][:3 * B * d].view(3, B, d).cpu()
    for i, mod in enumerate("tva"):
        setattr(getattr(m, f"project_{mod}"), f"project_{mod}_activation",
                _Site(name, A[i], info, f"proj[{mod}]", None if slopes is None else slopes["proj"][i]))
    if not cfg.use_cmd_sim:
        DH = eng.ws["DHpre"][:3 * B * d].view(3, B, d).cpu()
        sites = [_Site(name, DH[i], info, f"disc[{mod}]", None if slopes is None else slopes["disc"][i])
                 for i, mod in enumerate("tva")]
        cnt = [0]

        def disc_act(z):
            site = sites[cnt[0] % 3]
            cnt[0] += 1
            return site(z)
        m.discriminator.discriminator_layer_1_activation = _Lambda(disc_act)
    ffn = (eng.ws["F1"][:B * 6 * 2048].view(B, 6, 2048).permute(1, 0, 2) > 0).cpu()
    h = m.transformer_encoder.layers[0].linear1.register_forward_hook(
        lambda mod, i, o: _align(o, ffn.double(), "sign", info, "ffn-relu"))
    b = Batch(batch.sentences, batch.visual.double(), batch.acoustic.double(), batch.labels.double(),
              batch.lengths, batch.bert_sent, batch.bert_sent_type, batch.bert_sent_mask)
    out, L, grads = oracle_step(m, b, cfg, None)
    h.remove()
    return out, L, grads, info


class _Lambda(nn.Module):
    def __init__(self, fn):
        super().__init__()
        self.fn = fn

    def forward(self, z):
        return self.fn(z)


def _engine_slopes(eng, cfg, B, seed_dev=None):
    """the slopes the engine's last training-mode forward drew at each RReLU site"""
    from mmda_b200.engine import SID_RRELU_DISC, SID_RRELU_PROJECT
    k = eng.k
    k.bind_stream()
    d = cfg.hidden_size
    s = {"proj": [_slopes(k, B, d, eng.cur_seed, SID_RRELU_PROJECT + i, seed_dev).double().cpu()
                  for i in range(3)]}
    if not cfg.use_cmd_sim:
        s["disc"] = [_slopes(k, B, d, eng.cur_seed, SID_RRELU_DISC + i, seed_dev).double().cpu()
                     for i in range(3)]
    return s


def _activation_checks(tag, cfg, state, batch, dev, name, train=False):
    """level 1 (drop-in + autograd) and level 2 (fused losses + backward) against the fp64 oracle:
    all outputs, the six losses, every gradient.  ``train``: training-mode RReLU with the oracle
    multiplying by the slopes the device drew (dropout must be off: cfg.dropout = 0 and the
    fusion layer's ATT_P patched to 0 by the caller)."""
    from mmda_b200 import MISA
    from mmda_b200.trainer import FusedTrainer, LOSS_NAMES
    C = Checks(tag)
    B = batch.lengths.numel()
    # ---- level 1 ----
    model = MISA(cfg)
    model.load_state_dict(state)
    model = model.to(dev).train(train)
    out, L = _run_level1(model, batch, cfg, dev)
    eng = model.engine
    assert eng.rrelu_train == (train and name == "rrelu")
    # both pieces of the activation are exercised at every site
    sites = [("proj", eng.ws["A"][:3 * B * cfg.hidden_size].view(3, B, -1))]
    if not cfg.use_cmd_sim:
        sites.append(("disc", eng.ws["DHpre"][:3 * B * cfg.hidden_size].view(3, B, -1)))
    for site, Y in sites:
        for i in range(3):
            y = Y[i]
            on = {"hardshrink": y != 0, "hardtanh": y.abs() < 1}.get(name, y > 0)
            n_on, n = int(on.sum()), y.numel()
            C.flag(f"L1 {site}[{i}] elements on each piece: {n_on} / {n - n_on}", 0 < n_on < n)
    slopes = _engine_slopes(eng, cfg, B) if eng.rrelu_train else None
    o64, L64, g64, info = _oracle64(cfg, name, state, batch, eng, slopes)
    for kk, vv in info.items():
        C.rows.append((f"L1 branch alignment: {kk} = {vv}", 0.0, 0.0, True))
    C.add("L1 scores", out["scores"], o64["scores"])
    C.flag("L1 labels", torch.equal(out["labels"].cpu(), o64["labels"].float()) or
           float((o64["scores"] - cfg.threshold).abs().min()) < 1e-5)
    if not cfg.use_cmd_sim:
        out.update({a: getattr(model, a) for a in ADV_ATTRS})
    for a in ATTR_CHECK + (() if cfg.use_cmd_sim else ADV_ATTRS):
        C.add("L1 " + a, out[a], o64[a])
    for kk in ("cls", "diff", "recon", "sim", "conf", "total"):
        C.add("L1 loss " + kk, L[kk], L64[kk])
    none = set(model.param_names_without_grad())
    for n, p in model.named_parameters():
        if g64[n] is None:
            C.flag(f"L1 grad None {n}", p.grad is None and n in none)
        elif p.grad is None:
            C.flag(f"L1 grad present {n}", False)
        else:
            C.add("L1 grad " + n, p.grad, g64[n])
    # ---- level 2 ----
    model2 = MISA(cfg)
    model2.load_state_dict(state)
    model2 = model2.to(dev).train(train)
    tr = FusedTrainer(model2)
    s, v, a, ln = _to(batch, dev)
    losses = tr.forward_backward(s, v, a, ln, batch.labels.to(dev))
    lv = dict(zip(LOSS_NAMES, losses[:6].tolist()))
    eng2 = model2.engine
    if eng2.rrelu_train:      # the fused step draws from the device step counter: other slopes
        slopes2 = _engine_slopes(eng2, cfg, B, tr.state)
        assert not torch.equal(slopes2["proj"][0], slopes["proj"][0])
        o64, L64, g64, info = _oracle64(cfg, name, state, batch, eng2, slopes2)
        for kk, vv in info.items():
            C.rows.append((f"L2 branch alignment: {kk} = {vv}", 0.0, 0.0, True))
    for kk in LOSS_NAMES:
        C.add("L2 loss " + kk, torch.tensor(lv[kk]), L64[kk])
    for n, p in model2.named_parameters():
        if g64[n] is not None:
            C.add("L2 grad " + n, tr.G[n], g64[n])
    tr.close()
    C.finish()


def _widened(state):
    """At the reference's initialisation every pre-activation of project_m stays inside +-0.5 on
    these inputs: Hardshrink would zero the whole projection (every later output is then the same
    for all samples and modalities, the CMD terms sit at sqrt(0) and the oracle's gradient is NaN),
    and neither Hardshrink's nor Hardtanh's other piece would be reached.  Scaling project_m and
    discriminator_layer_1 by 4 puts pre-activations on both sides of every threshold."""
    return {k: v * 4 if k.split(".")[1] in ("project_t", "project_v", "project_a", "discriminator_layer_1")
            else v for k, v in state.items()}


# the configs carry the torch class, as the reference's config does: MISA maps it like the name,
# and the oracle builds it
def _c1(name, **kw):
    from mmda_b200.config import mosi_config
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build
    rec = json.load(open(os.path.join(GOLDEN, "c1_mosi_b64.json")))
    cfg = mosi_config(vocab_size=2000, activation=TORCH[name], **kw)
    state = {k: v.clone() for k, v in oracle_build(cfg, rec["seed"]).state_dict().items()}
    return cfg, _widened(state), batch_for(cfg, seed=rec["batch_seed"], lengths="ragged")


def _adversarial(name, **kw):
    z, meta = load_small("small_adversarial")
    return small_cfg(meta, activation=TORCH[name], **kw), _widened(state_from_npz(z)), small_batch(z)


@pytest.mark.parametrize("name", NEW)
def test_c1_mosi_b64_ragged(dev, name):
    _activation_checks(f"c1_{name}", *_c1(name), dev, name)


@pytest.mark.parametrize("name", NEW)
def test_small_adversarial(dev, name):
    _activation_checks(f"adversarial_{name}", *_adversarial(name), dev, name)


@pytest.mark.parametrize("fixture", ["c1", "small_adversarial"])
def test_rrelu_train_mode_with_the_device_slopes(dev, monkeypatch, fixture):
    import mmda_b200.engine as E
    monkeypatch.setattr(E, "ATT_P", 0.0)        # fusion-layer dropout off: only the slopes are random
    make = _c1 if fixture == "c1" else _adversarial
    _activation_checks(f"rrelu_train_{fixture}", *make("rrelu", dropout=0.0), dev, "rrelu", train=True)


def test_rrelu_graph_replay_draws_new_slopes_each_step(dev):
    """One capture of the fused step with training-mode RReLU (adversarial variant: both sites),
    then replays: per step the losses equal an eager trainer's with the same step state, and two
    consecutive replays draw different slopes -- the ones the device step counter selects."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.engine import SID_RRELU_PROJECT
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=300, batch_size=48, use_confidNet=True, activation="rrelu",
                       use_cmd_sim=False)
    b = batch_for(cfg, seed=40, lengths="full", seq_len=12)
    args = (b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths, b.labels.to(dev))
    B, d = 48, cfg.hidden_size
    res = {}
    for mode in (False, True):
        torch.manual_seed(5)
        model = MISA(cfg).to(dev).train()
        # learning rate 0: the parameters stay put, so from step to step only the random draws
        # (slopes, dropout masks) change what the step computes
        tr = FusedTrainer(model, lr=0.0, use_graph=mode)
        eng = model.engine
        Ls, As, counters = [], [], []
        for it in range(7):
            if mode and it == 3:
                launches = eng.k.launches          # after the capture: replays launch nothing
            L = tr.step(*args)
            torch.cuda.synchronize()
            Ls.append(L[:6].clone())
            As.append(eng.ws["A"][:3 * B * d].view(3, B, d).clone())
            counters.append(int(tr.state[:1].view(torch.int64).item()))
        if mode:
            assert len(tr._graphs) == 1 and eng.k.launches == launches
            res["slopes"] = [_slopes(eng.k, B, d, eng.seed, SID_RRELU_PROJECT, torch.tensor(
                [c, 0], dtype=torch.int64, device=dev)) for c in counters]
        res[mode] = (torch.stack(Ls).cpu(), As, counters)
        tr.close()
    C = Checks("rrelu_graph")
    C.add("losses per step, graph replay vs eager", res[True][0], res[False][0], 1e-5)
    counters = res[True][2]
    assert counters == res[False][2] and all(b - a == 1 for a, b in zip(counters, counters[1:])), counters
    C.flag("consecutive steps differ", all(not torch.equal(res[True][0][i], res[True][0][i + 1])
                                            for i in range(6)))
    # project_t: A = z where z > 0, z * r(step) elsewhere, z fixed: consecutive replays (steps 4..7)
    # scale the negative entries by the ratio of the slopes the counter selects
    As, r = res[True][1], res["slopes"]
    for i in range(3, 6):
        a0, a1 = As[i][0], As[i + 1][0]
        neg = a0 <= 0
        C.flag(f"replay {i + 1}->{i + 2}: positive part unchanged", torch.equal(a0[~neg], a1[~neg]))
        C.flag(f"replay {i + 1}->{i + 2}: new slopes", float((r[i] != r[i + 1]).float().mean()) > 0.99)
        z = a0.double() / r[i].double()
        C.add(f"replay {i + 1}->{i + 2}: A = z * r(counter)", torch.where(neg, a1, a0),
              torch.where(neg, z * r[i + 1].double(), a0.double()), 1e-6)
    C.finish()
