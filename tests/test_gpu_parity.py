"""Parity of the CUDA path (through the C ABI) against the oracle.  Run with ``-m gpu`` on a B200.

Tolerances (BASELINE.json north_star): logits, losses and gradients within 1e-5 relative in fp32
mode; packing indices bit-exact.  "Relative" is scale-relative (max |a-b| / max |ref|) against
an fp64 run of the oracle.  The bound is a hard 1e-5 (no allowance for the fp32 oracle's own
distance from fp64).
"""
import json
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, load_small, max_rel, small_batch, small_cfg, state_from_npz

pytestmark = pytest.mark.gpu
TOL = 1e-5


class Checks:
    def __init__(self, tag):
        self.tag, self.rows = tag, []

    def add(self, name, got, ref, tol=TOL, ref32=None):
        err = max_rel(got.detach().cpu() if torch.is_tensor(got) else got,
                      ref.detach().cpu() if torch.is_tensor(ref) else ref)
        bound = tol        # hard bound; ref32 (the fp32 oracle) is accepted for the call sites' sake only
        self.rows.append((name, err, bound, err <= bound))

    def flag(self, name, ok):
        self.rows.append((name, 0.0 if ok else float("inf"), 0.0, bool(ok)))

    def finish(self):
        out = os.path.join(os.path.dirname(GOLDEN), "..", "gpurun_out")
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, f"parity_{self.tag}.txt"), "w") as f:
            for n, e, b, ok in self.rows:
                f.write(f"{'ok  ' if ok else 'FAIL'} {n:60s} err={e:.3e} bound={b:.1e}\n")
        bad = [(n, e, b) for n, e, b, ok in self.rows if not ok]
        assert not bad, "\n".join(f"{n}: err={e:.3e} > {b:.1e}" for n, e, b in bad[:40])


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return torch.device("cuda:0")


def _to(batch, dev):
    return (batch.sentences.to(dev), batch.visual.to(dev), batch.acoustic.to(dev), batch.lengths)


# ------------------------------------------------------------------------------------------
# primitives
# ------------------------------------------------------------------------------------------
def test_sgemm_layouts(dev):
    from mmda_b200.engine import Kernels
    k = Kernels(); k.bind_stream()
    g = torch.Generator(device="cpu").manual_seed(0)
    C = Checks("sgemm")
    for (M, N, K) in [(5, 7, 3), (64, 64, 64), (256, 128, 140), (1536, 2048, 128), (300, 1200, 1000),
                      (1200, 300, 5000), (37, 129, 4099)]:
        for ta in (False, True):
            for tb in (False, True):
                A = torch.randn((K, M) if ta else (M, K), generator=g).to(dev)
                B = torch.randn((N, K) if tb else (K, N), generator=g).to(dev)
                bias = torch.randn(N, generator=g).to(dev)
                out = torch.full((M, N), 7.0, device=dev)
                k.gemm(A, B, out, ta=ta, tb=tb, bias=bias)
                ref = (A.double().t() if ta else A.double()) @ (B.double().t() if tb else B.double()) + bias.double()
                C.add(f"gemm {M}x{N}x{K} ta={ta} tb={tb}", out, ref, 1e-5)
                # deterministic in-CTA split-K: same answer, bit-identical run to run, beta / act
                o1 = torch.full((M, N), 0.5, device=dev); o2 = o1.clone()
                k.gemm(A, B, o1, ta=ta, tb=tb, bias=bias, beta=1.0, split_k=-1)
                k.gemm(A, B, o2, ta=ta, tb=tb, bias=bias, beta=1.0, split_k=-1)
                C.add(f"gemm in-CTA split-K {M}x{N}x{K} ta={ta} tb={tb}", o1, ref + 0.5, 1e-5)
                assert torch.equal(o1, o2)
                if K <= 64:     # fused activation (absolute check: sigmoid outputs are O(1))
                    k.gemm(A, B, o2, ta=ta, tb=tb, bias=bias, act=2, split_k=-1)
                    C.add(f"gemm in-CTA split-K sigmoid {M}x{N}x{K} ta={ta} tb={tb}", o2, torch.sigmoid(ref), 2e-6)
        # split-K accumulate
        A = torch.randn(K, M, generator=g).to(dev); B = torch.randn(K, N, generator=g).to(dev)
        acc = torch.randn(M, N, generator=g).to(dev); ref = acc.double() + A.double().t() @ B.double()
        k.gemm(A, B, acc, ta=True, beta=1.0, split_k=0)
        C.add(f"gemm splitk auto {M}x{N}x{K}", acc, ref, 1e-5)
    # strided C / A views and fused activation
    X = torch.randn(256, 128, generator=g).to(dev); W = torch.randn(128, 128, generator=g).to(dev)
    b = torch.randn(128, generator=g).to(dev)
    tok = torch.zeros(256, 6, 128, device=dev)
    k.linear(X, W, b, tok.view(256, 768)[:, 256:384], act=2)
    C.add("linear sigmoid strided", tok[:, 2, :], torch.sigmoid(X.double() @ W.double().t() + b.double()), 2e-6)
    assert float(tok[:, 1].abs().max()) == 0 and float(tok[:, 3].abs().max()) == 0
    C.finish()


def test_layernorm_attention_colsum(dev):
    from mmda_b200.engine import Kernels, _ptr
    k = Kernels(); k.bind_stream()
    g = torch.Generator().manual_seed(1)
    C = Checks("rowwise")
    for rows, width in [(37, 70), (1536, 128), (999, 600), (8, 148), (300, 768), (65, 1024)]:
        x = torch.randn(rows, width, generator=g).to(dev); r = torch.randn(rows, width, generator=g).to(dev)
        gam = (torch.rand(width, generator=g) + 0.5).to(dev); bet = torch.randn(width, generator=g).to(dev)
        dy = torch.randn(rows, width, generator=g).to(dev)
        for res in (None, r):
            y = torch.empty_like(x); mu = torch.empty(rows, device=dev); rs = torch.empty(rows, device=dev)
            k.layernorm(x, res, gam, bet, y, mu, rs)
            xd = (x if res is None else x + res).double().requires_grad_(True)
            gd, bd = gam.double().requires_grad_(True), bet.double().requires_grad_(True)
            yr = torch.nn.functional.layer_norm(xd, (width,), gd, bd, 1e-5)
            yr.backward(dy.double())
            C.add(f"ln fwd {rows}x{width} res={res is not None}", y, yr, 2e-6)
            dx = torch.empty_like(x); dg = torch.zeros(width, device=dev); db = torch.zeros(width, device=dev)
            k.layernorm_bwd(dy, x, res, gam, mu, rs, dx, dg, db)
            C.add(f"ln dx {rows}x{width}", dx, xd.grad, 5e-6)
            C.add(f"ln dgamma {rows}x{width}", dg, gd.grad, 5e-6)
            C.add(f"ln dbeta {rows}x{width}", db, bd.grad, 5e-6)
        cs = torch.zeros(width, device=dev); cs2 = torch.ones(width, device=dev)
        k.colsum(x, cs, cs2)
        C.add(f"colsum {rows}x{width}", cs, x.double().sum(0), 5e-6)
        C.add(f"colsum2 {rows}x{width}", cs2, x.double().sum(0) + 1, 5e-6)
    # attention core vs torch MHA math (eval: no dropout)
    for B, d in [(3, 16), (256, 128), (17, 64)]:
        hd = d // 2
        qkv = torch.randn(B * 6, 3 * d, generator=g).to(dev)
        ctx = torch.empty(B * 6, d, device=dev); pr = torch.empty(B, 2, 6, 6, device=dev)
        k._c("mmda_attention_forward", _ptr(qkv), _ptr(ctx), _ptr(pr), B, 6, 2, hd, 0.0, 1, None, 1)
        q3 = qkv.double().view(B, 6, 3, 2, hd).requires_grad_(True)
        q, kk, v = q3[:, :, 0], q3[:, :, 1], q3[:, :, 2]              # (B,6,2,hd)
        s = torch.einsum("bihd,bjhd->bhij", q, kk) / hd ** 0.5
        p = torch.softmax(s, -1)
        o = torch.einsum("bhij,bjhd->bihd", p, v).reshape(B * 6, d)
        C.add(f"attn fwd B={B} d={d}", ctx, o, 2e-6)
        C.add(f"attn probs B={B} d={d}", pr, p, 2e-6)
        do = torch.randn(B * 6, d, generator=g).to(dev)
        o.backward(do.double())
        dqkv = torch.empty_like(qkv)
        k._c("mmda_attention_backward", _ptr(qkv), _ptr(pr), _ptr(do), _ptr(dqkv), B, 6, 2, hd, 0.0, 1, None, 1)
        C.add(f"attn bwd B={B} d={d}", dqkv, q3.grad.reshape(B * 6, 3 * d), 5e-6)
    C.finish()


def test_pack_indices_bit_exact(dev):
    from mmda_b200 import MISA, MisaConfig
    from mmda_b200.engine import MisaEngine
    cfg = MisaConfig(embedding_size=8, visual_size=4, acoustic_size=4, hidden_size=8, vocab_size=30)
    eng = MISA(cfg).to(dev).engine
    eng.params(); eng.k.bind_stream()
    g = torch.Generator().manual_seed(5)
    for B, T in [(1, 1), (7, 9), (40, 50), (256, 50), (300, 17)]:
        for trial in range(3):
            ln = torch.randint(1, T + 1, (B,), generator=g)
            x = torch.randn(int(ln.max()), B, 3, generator=g)
            ref = torch.nn.utils.rnn.pack_padded_sequence(x, ln, enforce_sorted=False)
            pk = eng._pack(ln)
            assert torch.equal(pk["bs"].cpu().long(), ref.batch_sizes)
            assert torch.equal(pk["sidx"].cpu().long(), ref.sorted_indices)
            off = torch.zeros(len(ref.batch_sizes) + 1, dtype=torch.long)
            off[1:] = torch.cumsum(ref.batch_sizes, 0)
            assert torch.equal(pk["off"].cpu().long(), off)
            # the gather itself: packed rows == PackedSequence.data bit for bit
            X = torch.empty(pk["N"], 3, device=dev)
            from mmda_b200.engine import _ptr
            eng.k._c("mmda_gather_rows", _ptr(x.to(dev)), _ptr(X), 3, _ptr(pk["row_t"]), _ptr(pk["row_j"]),
                     _ptr(pk["sidx"]), pk["N"], B, 3)
            assert torch.equal(X.cpu(), ref.data)


def test_adam_clip_matches_torch(dev):
    from mmda_b200.engine import Kernels, _ptr
    k = Kernels(); k.bind_stream()
    g = torch.Generator().manual_seed(2)
    n = 100003
    p0 = torch.randn(n + 1, generator=g)[:n]
    pt = p0.clone().double().requires_grad_(True)
    opt = torch.optim.Adam([pt], lr=1e-3)
    p = torch.zeros(n + 1, device=dev)[:n]; p.copy_(p0)
    m = torch.zeros(n + 1, device=dev)[:n]; v = torch.zeros(n + 1, device=dev)[:n]
    C = Checks("adam")
    for step in range(1, 5):
        gr = torch.randn(n, generator=g) * 2
        pt.grad = gr.double().clone()
        torch.nn.utils.clip_grad_value_([pt], 1.0)
        opt.step()
        gd = gr.to(dev)
        k._c("mmda_adam_clip_step", _ptr(p), _ptr(gd), _ptr(m), _ptr(v), n, step, 1e-3, 1.0, 0.9, 0.999, 1e-8, 1.0, None)
        C.add(f"adam step {step}", p, pt.detach(), 2e-6)
    C.finish()


# ------------------------------------------------------------------------------------------
# whole model
# ------------------------------------------------------------------------------------------
def _oracle_pair(cfg, state, batch, masks=None, frozen=None):
    """fp32 and fp64 oracle runs (CPU) of one step: outputs, losses, grads-before-clip.

    ``masks`` (from the device run) aligns the piecewise-linear activations: the FFN ReLU
    (393k-3.1M units) and the projection activation have a kink at 0, and a pre-activation within
    fp32 rounding of 0 may fall on either side.  Such a flip changes a gradient row by O(1e-4)
    relative although both runs are "correct".  Where the device mask and the oracle mask
    disagree AND the oracle's pre-activation is within 1e-5 of zero, the oracle's pre-activation
    is nudged across zero (by < 1e-5 absolute) so both differentiate the same linear piece.  The
    number of aligned units and their largest |z| are recorded in the parity report."""
    from oracle.misa_oracle import OracleMISA, oracle_step
    res, info = {}, {}
    for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
        m = OracleMISA(cfg)
        m.load_state_dict(state)
        m = m.to(dt).eval()
        if frozen is not None:
            for n, p in m.named_parameters():
                p.requires_grad = not frozen(n)
        handles = []
        if masks is not None:
            def align(z, mine, key):
                flips = (z > 0) != mine
                n = int(flips.sum())
                info[f"{tag} {key} flips"] = n
                if n == 0:
                    return z
                info[f"{tag} {key} max|z| at flips"] = float(z[flips].abs().max())
                ok = flips & (z.abs() < 1e-5)
                tgt = torch.where(mine, torch.full_like(z, 1e-12), torch.full_like(z, -1e-12))
                return z + (torch.where(ok, tgt, z) - z).detach()
            lin1 = m.transformer_encoder.layers[0].linear1
            handles.append(lin1.register_forward_hook(
                lambda mod, i, o: align(o, masks["ffn"], "ffn-relu")))
            cnt = [0]
            def pre(mod, inp):
                if cnt[0] >= 3:      # the same activation instance also serves the discriminator
                    return None
                i = cnt[0] % 3
                cnt[0] += 1
                return (align(inp[0], masks["proj"][i], f"proj-act[{i}]"),)
            handles.append(m.project_t[1].register_forward_pre_hook(pre))
        b = batch
        if dt == torch.float64:
            from mmda_b200.synthetic import Batch
            b = Batch(batch.sentences, batch.visual.double(), batch.acoustic.double(),
                      batch.labels.double(), batch.lengths, batch.bert_sent, batch.bert_sent_type,
                      batch.bert_sent_mask)
        out, L, grads = oracle_step(m, b, cfg, None)
        for h in handles:
            h.remove()
        res[tag] = (out, L, grads)
    res["info"] = info
    return res


def _run_level1(model, batch, cfg, dev):
    """The reference's own loss code shape (oracle_losses mirrors solver.get_*_loss) on the
    drop-in model's autograd-connected attributes."""
    from oracle.misa_oracle import oracle_losses
    model.zero_grad()
    bert = (batch.bert_sent.to(dev), batch.bert_sent_type.to(dev), batch.bert_sent_mask.to(dev)) \
        if cfg.use_bert else (None, None, None)
    scores, labels = model(*_to(batch, dev), *bert)
    out = {k: getattr(model, k) for k in model.OUTPUT_ATTRS}
    if not cfg.use_cmd_sim:
        out.update({a: getattr(model, a) for a in ("domain_label_t", "domain_label_v", "domain_label_a")})
    out["scores"], out["labels"] = scores, labels
    L = oracle_losses(out, batch.labels.to(dev), cfg)
    L["total"].backward()
    return out, L


ADV_ATTRS = ("domain_label_t", "domain_label_v", "domain_label_a")
ATTR_CHECK = ("utt_t_orig", "utt_v_orig", "utt_a_orig", "utt_private_t", "utt_private_v",
              "utt_private_a", "utt_shared_t", "utt_shared_v", "utt_shared_a", "utt_t_recon",
              "utt_v_recon", "utt_a_recon", "tcp", "shared_or_private_p_t", "shared_or_private_s")


def _model_checks(tag, cfg, state, batch, dev, golden=None, frozen=None):
    from mmda_b200 import MISA
    from mmda_b200.trainer import FusedTrainer, LOSS_NAMES
    C = Checks(tag)
    is_frozen = frozen or (lambda n: False)
    # exactly 0 in exact arithmetic (softmax shift invariance): pure rounding noise
    noise = lambda n: n.startswith("bertmodel.") and n.endswith("attention.self.key.bias")
    # ---- level 1: drop-in forward + autograd bridge ----
    model = MISA(cfg)
    model.load_state_dict(state)
    for n, p in model.named_parameters():
        p.requires_grad = not is_frozen(n)
    model = model.to(dev).eval()
    out, L = _run_level1(model, batch, cfg, dev)
    eng, B, d = model.engine, batch.lengths.numel(), cfg.hidden_size
    masks = {"ffn": (eng.ws["F1"][:B * 6 * 2048].view(B, 6, 2048).permute(1, 0, 2) > 0).cpu(),
             "proj": (eng.ws["A"][:3 * B * d].view(3, B, d) > 0).cpu()}
    orc = _oracle_pair(cfg, state, batch, masks, frozen)
    o32, L32, g32 = orc["f32"]
    o64, L64, g64 = orc["f64"]
    for kk, vv in orc["info"].items():
        C.rows.append((f"kink alignment: {kk} = {vv}", 0.0, 0.0, True))
    C.add("L1 scores", out["scores"], o64["scores"], ref32=o32["scores"])
    C.flag("L1 labels", torch.equal(out["labels"].cpu(), o32["labels"]) or
           float((o64["scores"] - cfg.threshold).abs().min()) < 1e-5)
    if not cfg.use_cmd_sim:
        out.update({a: getattr(model, a) for a in ADV_ATTRS})
    for a in ATTR_CHECK + (() if cfg.use_cmd_sim else ADV_ATTRS):
        C.add("L1 " + a, out[a], o64[a], ref32=o32[a])
    for kk in ("cls", "diff", "recon", "sim", "conf", "total"):
        C.add("L1 loss " + kk, L[kk], L64[kk], ref32=L32[kk])
    none = set(model.param_names_without_grad())
    for n, p in model.named_parameters():
        if g64[n] is None:
            C.flag(f"L1 grad None {n}", p.grad is None and (n in none or is_frozen(n)))
        elif noise(n):
            continue
        elif p.grad is None:
            C.flag(f"L1 grad present {n}", False)
        else:
            C.add("L1 grad " + n, p.grad, g64[n], ref32=g32[n])
    # ---- level 2: fused losses + backward + clip + Adam ----
    model2 = MISA(cfg)
    model2.load_state_dict(state)
    for n, p in model2.named_parameters():
        p.requires_grad = not is_frozen(n)
    model2 = model2.to(dev).eval()
    tr = FusedTrainer(model2)
    s, v, a, ln = _to(batch, dev)
    bert = (batch.bert_sent.to(dev), batch.bert_sent_type.to(dev), batch.bert_sent_mask.to(dev)) \
        if cfg.use_bert else None
    losses = tr.forward_backward(s, v, a, ln, batch.labels.to(dev), bert)
    lv = dict(zip(LOSS_NAMES, losses[:6].tolist()))
    for kk in LOSS_NAMES:
        C.add("L2 loss " + kk, torch.tensor(lv[kk]), L64[kk], ref32=L32[kk])
    for n, p in model2.named_parameters():
        if g64[n] is not None and not noise(n):
            C.add("L2 grad " + n, tr.G[n], g64[n], ref32=g32[n])
    # ---- clip + Adam: the update applied to the device gradients must equal the restated
    # optimiser (oracle/explicit.py::adam_clip_step, checked against torch.optim.Adam on CPU)
    # applied to the SAME gradients.  Comparing against the oracle's post-step parameters
    # directly is ill-conditioned: Adam's first update is lr*g/(|g|+1e-8), so gradient elements
    # at rounding-noise level (e.g. the attention key bias, exactly 0 in exact arithmetic) get a
    # +-lr update whose sign is noise in any fp32 implementation.  Gradient parity is asserted
    # above; together the two imply step parity wherever the step is well-conditioned.
    from oracle.explicit import adam_clip_step
    g_dev = {n: tr.G[n].detach().cpu().double().numpy().copy() for n in state}
    tr.optimizer_step()
    for n, p in model2.named_parameters():
        if g64[n] is not None:
            p0 = state[n].double().numpy()
            exp, _, _ = adam_clip_step(p0, g_dev[n], np.zeros_like(p0), np.zeros_like(p0), 1,
                                       cfg.learning_rate, cfg.clip)
            C.add("L2 param-after-step " + n, p.data, torch.from_numpy(exp), 2e-6)
        else:
            C.flag(f"L2 untouched {n}", torch.equal(p.data.cpu(), state[n]))
    if golden is not None:
        for kk, vv in golden["losses"].items():
            C.add("golden loss " + kk, torch.tensor(lv[kk]), torch.tensor(vv), 2e-5)
        C.add("golden scores", out["scores"], torch.tensor(golden["scores"]), 2e-5)
    C.finish()


@pytest.mark.parametrize("name", ["small_ragged", "small_shuffled_confid", "small_adversarial", "small_gru"])
def test_small_fixture(dev, name):
    z, meta = load_small(name)
    cfg = small_cfg(meta)
    golden = {"losses": {k: float(z["loss/" + k]) for k in ("cls", "diff", "recon", "sim", "conf", "total")},
              "scores": z["out/scores"].tolist()}
    _model_checks(name, cfg, state_from_npz(z), small_batch(z), dev, golden)


def _full(cfgname, recname, lengths, dev, **kw):
    from mmda_b200 import config as Cfg
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build
    rec = json.load(open(os.path.join(GOLDEN, recname + ".json")))
    cfg = getattr(Cfg, cfgname + "_config")(vocab_size=2000, **kw)
    state = {k: v.clone() for k, v in oracle_build(cfg, rec["seed"]).state_dict().items()}
    batch = batch_for(cfg, seed=rec["batch_seed"], lengths=lengths)
    _model_checks(recname, cfg, state, batch, dev, rec["steps"][0])


def test_c1_mosi_b64_ragged(dev):
    _full("mosi", "c1_mosi_b64", "ragged", dev)


def test_c2_mosei_b256_full(dev):
    _full("mosei", "c2_mosei_b256", "full", dev)


def test_c3_mosei_confid_ragged(dev):
    _full("mosei", "c3_mosei_confid_b256", "ragged", dev, use_confidNet=True)


def test_train_mode_dropout_statistics(dev):
    """Train-mode dropout is checked statistically (SURVEY.md hard part 5): keep rate and the
    0.5 score of dropped classifier logits (dropout sits before the sigmoid, models.py:150-153)."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    cfg = mosei_config(vocab_size=500, dropout=0.5)
    torch.manual_seed(0)
    model = MISA(cfg).to(dev).train()
    batch = batch_for(cfg, seed=3, lengths="ragged", seq_len=12)
    with torch.no_grad():
        scores, _ = model(*_to(batch, dev), None, None, None)
    frac = float((scores == 0.5).float().mean())
    assert 0.42 < frac < 0.58, frac
    model.eval()
    with torch.no_grad():
        s1, _ = model(*_to(batch, dev), None, None, None)
        s2, _ = model(*_to(batch, dev), None, None, None)
    assert torch.equal(s1, s2) and float((s1 == 0.5).float().mean()) < 0.01


def test_missing_library_fails_loudly(dev, monkeypatch):
    import mmda_b200._lib as L
    fresh = L._Lib()
    monkeypatch.setattr(L, "LIB_PATH", "/nonexistent/libmmda_b200.so")
    with pytest.raises(L.MmdaError):
        fresh.load()


def test_gemm_tc_tf32x3_and_bf16(dev):
    """tcgen05/TMA GEMM: 3xTF32 must be fp32-accurate (<= 1e-5), bf16 within 2e-2; all operand
    majors (K-major / MN-major), ragged tiles, bias, accumulate and split-K."""
    from mmda_b200.engine import Kernels, _ptr
    k = Kernels(); k.bind_stream()
    g = torch.Generator().manual_seed(7)
    C = Checks("gemm_tc")

    def split(x):
        hi, lo = torch.empty_like(x), torch.empty_like(x)
        k._c("mmda_split_tf32", _ptr(x), x.stride(0), x.shape[0], x.shape[1], _ptr(hi), _ptr(lo), hi.stride(0))
        return hi, lo

    shapes = [(128, 128, 32), (256, 128, 64), (1000, 300, 300), (12800, 2400, 300), (1200, 300, 12800),
              (300, 1200, 1000), (77, 52, 36)]
    for (M, N, K) in shapes:
        for a_mn in (0, 1):
            for b_mn in (0, 1):
                A = torch.randn((K, M) if a_mn else (M, K), generator=g).to(dev)
                B = torch.randn((K, N) if b_mn else (N, K), generator=g).to(dev)
                if (A.stride(0) * 4) % 16 or (B.stride(0) * 4) % 16:
                    continue
                bias = torch.randn(N, generator=g).to(dev)
                ref = (A.double().t() if a_mn else A.double()) @ (B.double() if b_mn else B.double().t())
                Ah, Al = split(A); Bh, Bl = split(B)
                out = torch.full((M, N), 3.0, device=dev)
                k._c("mmda_gemm_tc", 0, a_mn, b_mn, M, N, K, _ptr(Ah), _ptr(Al), A.stride(0), _ptr(Bh),
                     _ptr(Bl), B.stride(0), 1.0, _ptr(out), N, _ptr(bias), None, 0, 1, 0)
                # one accumulation chain over K=12800 drifts to ~1e-5 (tensor-core fp32 adds truncate);
                # the library's own callers use the auto split-K for such shapes (checked below)
                C.add(f"tf32x3 {M}x{N}x{K} a_mn={a_mn} b_mn={b_mn}", out, ref + bias.double(),
                      1e-5 if K <= 4096 else 3e-5)
                # kind 2: the same contraction from the plain fp32 operands (hi/lo split inside
                # the kernel's shared-memory pipeline) must give the same bits
                out2 = torch.full((M, N), 5.0, device=dev)
                k._c("mmda_gemm_tc", 2, a_mn, b_mn, M, N, K, _ptr(A), None, A.stride(0), _ptr(B),
                     None, B.stride(0), 1.0, _ptr(out2), N, _ptr(bias), None, 0, 1, 0)
                C.flag(f"tf32x3 raw == pre-split {M}x{N}x{K} a_mn={a_mn} b_mn={b_mn}",
                       torch.equal(out, out2))
                # mixed: A plain fp32, B pre-split (how weights are fed)
                out3 = torch.full((M, N), 6.0, device=dev)
                k._c("mmda_gemm_tc", 2, a_mn, b_mn, M, N, K, _ptr(A), None, A.stride(0), _ptr(Bh),
                     _ptr(Bl), B.stride(0), 1.0, _ptr(out3), N, _ptr(bias), None, 0, 1, 0)
                C.flag(f"tf32x3 raw-A/split-B == pre-split {M}x{N}x{K} a_mn={a_mn} b_mn={b_mn}",
                       torch.equal(out, out3))
                if K >= 1000:
                    acc = torch.randn(M, N, generator=g).to(dev)
                    ref2 = acc.double() + 0.5 * ref
                    k._c("mmda_gemm_tc", 0, a_mn, b_mn, M, N, K, _ptr(Ah), _ptr(Al), A.stride(0), _ptr(Bh),
                         _ptr(Bl), B.stride(0), 0.5, _ptr(acc), N, None, None, 1, 0, 0)
                    C.add(f"tf32x3 splitK {M}x{N}x{K} a_mn={a_mn} b_mn={b_mn}", acc, ref2, 1e-5)
    # bf16 (pitches padded to 8 elements)
    for (M, N, K) in [(256, 128, 64), (1000, 304, 304), (1200, 304, 4096)]:
        for a_mn in (0, 1):
            for b_mn in (0, 1):
                A = torch.randn((K, M) if a_mn else (M, K), generator=g).to(dev)
                B = torch.randn((K, N) if b_mn else (N, K), generator=g).to(dev)
                Ab = torch.empty(A.shape, dtype=torch.bfloat16, device=dev)
                Bb = torch.empty(B.shape, dtype=torch.bfloat16, device=dev)
                k._c("mmda_cast_bf16", _ptr(A), A.stride(0), A.shape[0], A.shape[1], _ptr(Ab), Ab.stride(0))
                k._c("mmda_cast_bf16", _ptr(B), B.stride(0), B.shape[0], B.shape[1], _ptr(Bb), Bb.stride(0))
                assert torch.equal(Ab, A.bfloat16())
                out = torch.empty(M, N, device=dev)
                k._c("mmda_gemm_tc", 1, a_mn, b_mn, M, N, K, _ptr(Ab), None, Ab.stride(0), _ptr(Bb), None,
                     Bb.stride(0), 1.0, _ptr(out), N, None, None, 0, 1, 0)
                Ad, Bd = Ab.double(), Bb.double()
                ref = (Ad.t() if a_mn else Ad) @ (Bd if b_mn else Bd.t())
                C.add(f"bf16 {M}x{N}x{K} a_mn={a_mn} b_mn={b_mn}", out, ref, 1e-5)
    C.finish()


def test_c3_precision_flag_packs_the_lstm_weights_fp32(dev):
    """BASELINE configs[2] (ConfidNet branch, "bf16 input-projection GEMMs").  Round 1 measured that
    a bf16 input projection moves this model's text-encoder gradients by 5-15 % -- far outside the
    2e-2 bar against the reference -- and gains no time, so the LSTM encoders now run fp32-accurate
    (3xTF32 GEMMs, fp32-accurate tensor-core recurrence) whatever ``precision`` says; the flag only
    selects bf16 operands for the BERT encoder (C4).  With precision="bf16" the whole C3 check
    list (outputs, losses, every gradient, level 1 and 2) must hold at the fp32 bar of 1e-5."""
    from mmda_b200 import MISA, config as Cfg
    from mmda_b200.synthetic import batch_for
    cfg = Cfg.mosei_config(vocab_size=50, use_confidNet=True, precision="bf16")
    probe = MISA(cfg).to(dev).eval()
    assert probe.engine.tc_kind == 1
    b = batch_for(cfg, seed=3, batch=8, seq_len=5)
    with torch.no_grad():
        probe(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths)
    # the LSTM input projections packed their weights as 3xTF32 hi / lo pairs, none as bf16
    ws = probe.engine.ws
    assert all(f"tcW_{r}_lo" in ws for r in ("trnn1", "trnn2", "vrnn1", "vrnn2", "arnn1", "arnn2"))
    assert not any(n.startswith(("tcW_", "tcX_")) and n.endswith("_bf") for n in ws)
    _full("mosei", "c3_mosei_confid_b256", "ragged", dev, use_confidNet=True, precision="bf16")


@pytest.mark.parametrize("rnncell", ["lstm", "gru"])
def test_cuda_graph_replay_equals_eager(dev, rnncell):
    """The captured CUDA graph of the fused step (multi-stream forks, device-resident step state)
    must produce the same training trajectory as eager launches, including train-mode dropout
    (same device seed counter) and varying inputs."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=300, batch_size=48, use_confidNet=True, rnncell=rnncell)
    batches = [batch_for(cfg, seed=40 + i, lengths="full", seq_len=12) for i in range(3)]
    res = {}
    for mode in (False, True):
        torch.manual_seed(5)
        model = MISA(cfg).to(dev).train()
        tr = FusedTrainer(model, use_graph=mode)
        Ls = []
        for it in range(7):
            b = batches[it % 3]
            L = tr.step(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths, b.labels.to(dev))
            Ls.append(L[:6].clone())
        assert (tr._graph is not None) == mode
        res[mode] = (torch.stack(Ls).cpu(), tr.p_arena[:tr.n_active].clone().cpu(), tr.step_count)
    assert res[True][2] == res[False][2] == 7
    C = Checks("graph_" + rnncell)
    C.add("losses over 7 steps", res[True][0], res[False][0], 1e-5)
    # parameters: atomics (split-K, RED epilogues) make rounding-level gradient elements differ
    # between two runs, and Adam turns such an element into a +-lr update whose sign is noise:
    # the bound is Adam's noise floor 2*lr*steps, the trajectory check above is the tight one
    dp = float((res[True][1] - res[False][1]).abs().max())
    C.rows.append((f"parameters after 7 steps: max |delta| = {dp:.3e} <= 2*lr*steps", dp,
                   2 * cfg.learning_rate * 7, dp <= 2 * cfg.learning_rate * 7))
    C.finish()


def test_graph_step_follows_the_model_to_another_gpu(dev):
    """The step's side streams belong to a device: after ``model.to('cuda:1')`` a trainer that
    replayed a graph on cuda:0 steps on cuda:1 (eager warm-up, new capture, replays) and trains
    exactly as a trainer built there with the same parameters and optimizer state."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=300, batch_size=48, use_confidNet=True)
    b = batch_for(cfg, seed=7, lengths="full", seq_len=12)
    d1 = torch.device("cuda:1")

    def run(tr, d, n):
        return torch.stack([tr.step(b.sentences.to(d), b.visual.to(d), b.acoustic.to(d), b.lengths,
                                    b.labels.to(d))[:6].clone() for _ in range(n)]).cpu()
    torch.manual_seed(5)
    model = MISA(cfg).to(dev).eval()
    tr = FusedTrainer(model)
    run(tr, dev, 4)
    assert tr._graph is not None
    with torch.cuda.device(1):
        model.to(d1)
        ref = MISA(cfg)
        ref.load_state_dict(model.state_dict())
        fresh = FusedTrainer(ref.to(d1).eval())
        tr._check_alias()                  # the moved trainer's optimizer state, on cuda:1
        fresh.load_optimizer_state_dict(tr.optimizer_state_dict())
        got, want = run(tr, d1, 5), run(fresh, d1, 5)
        assert tr._graph is not None and tr.p_arena.device == d1
        torch.cuda.synchronize()
    err = float(((got - want).abs() / want.abs().clamp_min(1e-6)).max())
    assert err < 1e-5, err


def test_graph_replay_after_other_forwards(dev):
    """A captured step reads the packing buffers by pointer.  evaluate(), a level-1 forward or an
    eager step with other lengths overwrite them between two replays; the next replay must still
    be the step of ITS lengths (ADVICE r1: stale pack buffers)."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=300, batch_size=48)
    b1 = batch_for(cfg, seed=5, lengths="ragged", seq_len=14)
    b2 = batch_for(cfg, seed=6, lengths="shuffled", seq_len=14)     # same shapes, other lengths

    def make():
        torch.manual_seed(11)
        m = MISA(cfg)
        for n, p in m.named_parameters():
            if "weight_hh" in n:
                torch.nn.init.orthogonal_(p)
        return m.to(dev).eval()

    def args(b):
        return (b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths, b.labels.to(dev))

    seq = [b1, b1, b1, b1, b2, b1, "fwd", b1, b1]
    outs = {}
    for mode in (True, False):
        tr = FusedTrainer(make(), use_graph=mode)
        L = []
        for item in seq:
            if item == "fwd":          # a level-1 forward on the same engine with other lengths
                with torch.no_grad():
                    tr.model(*args(b2)[:4])
                continue
            L.append(tr.step(*args(item))[:6].clone())
        if mode:
            # one graph for both length patterns: the key carries the padded row count only
            assert len(tr._graphs) == 1 and tr._graph["key"][3] in (512, 48 * 14)
        outs[mode] = (torch.stack(L), tr.p_arena[:tr.n_active].clone())
        tr.close()
    lerr = float(((outs[True][0] - outs[False][0]).abs() / outs[False][0].abs().clamp_min(1e-6)).max())
    assert lerr < 2e-5, lerr
    assert float((outs[True][1] - outs[False][1]).abs().max()) <= 2 * 1e-4 * len(seq) + 1e-6


@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_one_step_graph_serves_a_ragged_stream(dev, cell):
    """VERDICT r1 #3: the captured step must not be keyed by the lengths.  Ten batches with ten
    different length patterns run through at most two graphs (packed rows rounded to the row
    granule); losses and parameters match the exact-row eager steps of the same stream."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200 import trainer as T
    from mmda_b200.synthetic import batch_for
    cfg = mosei_config(vocab_size=300, batch_size=64, rnncell=cell)
    stream = [batch_for(cfg, seed=40 + i, lengths="ragged" if i % 3 else "shuffled", seq_len=20)
              for i in range(10)]
    assert len({tuple(b.lengths.tolist()) for b in stream}) == 10

    def make():
        torch.manual_seed(12)
        m = MISA(cfg)
        for n, p in m.named_parameters():
            if "weight_hh" in n:
                torch.nn.init.orthogonal_(p)
        return m.to(dev).eval()

    outs, old = {}, T.ROW_GRANULE
    T.ROW_GRANULE = 256
    try:
        for mode in (True, False):
            tr = T.FusedTrainer(make(), use_graph=mode)
            L = [tr.step(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths,
                         b.labels.to(dev))[:6].clone() for b in stream + stream]
            if mode:
                keys = list(tr._graphs)
                assert 1 <= len(keys) <= 3, keys
                assert all(k[3] % 256 == 0 or k[3] == 64 * 20 for k in keys), keys
            outs[mode] = (torch.stack(L), tr.p_arena[:tr.n_active].clone())
            tr.close()
    finally:
        T.ROW_GRANULE = old
    lerr = float(((outs[True][0] - outs[False][0]).abs() / outs[False][0].abs().clamp_min(1e-6)).max())
    # 20 optimisation steps: padded and exact launches differ in summation order (split-K over Np
    # vs N rows), and Adam amplifies 1e-7 gradient differences; single-step gradients are compared
    # tightly in test_padded_rows_gradients_match_exact_rows
    assert lerr < 1e-4, lerr
    assert float((outs[True][1] - outs[False][1]).abs().max()) <= 2 * 1e-4 * 20 + 1e-6


def test_step_batch_loss_future(dev):
    """step_batch(fetch=True): the LossFuture of step i, read after step i+1 was enqueued, holds
    step i's losses (the bench's e2e loop), for graph-replayed steps too."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=300, batch_size=32)
    host = [batch_for(cfg, seed=70 + i, lengths="full", seq_len=12) for i in range(3)]

    def make():
        torch.manual_seed(14)
        return MISA(cfg).to(dev).eval()

    ref_tr = FusedTrainer(make())
    ref = [ref_tr.step_batch(host[i % 3]).tolist() for i in range(8)]
    ref_tr.close()
    tr = FusedTrainer(make())
    got, pending = [], None
    for i in range(8):
        fut = tr.step_batch(host[i % 3], prefetch=host[(i + 1) % 3], fetch=True)
        if pending is not None:
            got.append(pending.result())
        pending = fut
    got.append(pending.result())
    tr.close()
    assert len(got) == 8
    for a, b in zip(got, ref):
        assert max(abs(x - y) / max(abs(y), 1e-6) for x, y in zip(a[:6], b[:6])) < 2e-5, (a, b)


@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_padded_rows_gradients_match_exact_rows(dev, cell):
    """The padded launch (Np > N rows, T_pad > Tmax) must give the exact launch's gradients: same
    batch, engine.pad set by hand, every parameter gradient compared."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=300, batch_size=32, rnncell=cell)
    b = batch_for(cfg, seed=9, lengths="ragged", seq_len=16)
    b.lengths = b.lengths.clamp(max=11)            # Tmax < T of the tensors
    torch.manual_seed(13)
    model = MISA(cfg).to(dev).eval()
    tr = FusedTrainer(model, use_graph=False)
    a = (b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths, b.labels.to(dev))
    res = {}
    for pad in (None, (16, 32 * 16), (16, int(b.lengths.sum()) + 5)):
        tr.eng.pad = pad
        tr.g_arena.zero_()
        losses = tr.forward_backward(*a)
        res[pad] = (losses[:6].clone(), tr.g_arena[:tr.n_active].clone())
    tr.eng.pad = None
    for pad in list(res)[1:]:
        dl = float((res[pad][0] - res[None][0]).abs().max())
        g0 = res[None][1]
        dg = float((res[pad][1] - g0).abs().max() / g0.abs().max())
        assert dl < 1e-6 and dg < 2e-6, (pad, dl, dg)
    tr.close()


def test_long_ragged_sequences_t130(dev):
    """Sequence-length sweep (BASELINE configs[4]): T=130, ragged + shuffled lengths."""
    from mmda_b200 import config as Cfg
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build
    cfg = Cfg.mosi_config(vocab_size=500, batch_size=24)
    state = {k: v.clone() for k, v in oracle_build(cfg, 77).state_dict().items()}
    batch = batch_for(cfg, seed=78, lengths="shuffled", seq_len=130)
    _model_checks("t130_shuffled", cfg, state, batch, dev, None)


def test_eval_pass_metrics_on_device(dev):
    """Solver.eval (src/solver.py:311-370) on the device: forward-only, cls loss, metrics."""
    import numpy as np
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.evaluate import evaluate
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import OracleMISA, oracle_losses
    cfg = mosei_config(vocab_size=400, batch_size=40, threshold=0.5)
    torch.manual_seed(11)
    model = MISA(cfg)
    state = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.to(dev)
    batches = [batch_for(cfg, seed=60 + i, lengths="ragged", seq_len=15) for i in range(3)]
    got = evaluate(model, batches)
    ref = OracleMISA(cfg); ref.load_state_dict(state); ref.eval()
    ys, ps, losses = [], [], []
    with torch.no_grad():
        for b in batches:
            out = ref(*b.model_args())
            losses.append(float(oracle_losses(out, b.labels, cfg)["cls"]))
            ys.append(b.labels.numpy()); ps.append(out["labels"].numpy())
    y, p = np.concatenate(ys), np.concatenate(ps)
    from sklearn import metrics as M
    jac = np.mean((y * p).sum(1) / np.maximum(((y + p) > 0).sum(1), 1))
    assert abs(got["loss"] - np.mean(losses)) < 1e-5 * np.mean(losses)
    assert abs(got["acc"] - round(float(jac), 4)) <= 1e-4
    assert abs(got["f1"] - M.f1_score(y, p, average="macro", zero_division=0)) < 1e-6
    assert abs(got["micro_precision"] - M.precision_score(y, p, average="micro", zero_division=0)) < 1e-6
    assert abs(got["weighted_recall"] - M.recall_score(y, p, average="weighted", zero_division=0)) < 1e-6


def test_bert_text_branch_level1(dev):
    """use_bert=True (BASELINE configs[3] / SURVEY 8f N1): random-init bert-base on the
    hand-written kernels (mmda_b200/bert.py) vs the oracle's HF BertModel; level-1 contract incl.
    the reference's layer freezing (solver.py:69-73): frozen tensors keep grad None, every
    trainable BERT tensor (layers 9-11 + embeddings) is compared."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build, oracle_step
    cfg = mosei_config(vocab_size=100, batch_size=6, use_bert=True)
    ref = oracle_build(cfg, 21).eval()
    state = {k: v.clone() for k, v in ref.state_dict().items()}
    batch = batch_for(cfg, seed=22, lengths="ragged", seq_len=9)
    out_r, L_r, g_r = oracle_step(ref, batch, cfg, None)
    model = MISA(cfg)
    model.load_state_dict(state)
    for n, p in model.named_parameters():
        if "bertmodel.encoder.layer" in n and int(n.split("encoder.layer.")[-1].split(".")[0]) <= 8:
            p.requires_grad = False
    model = model.to(dev).eval()
    from oracle.misa_oracle import oracle_losses
    scores, labels = model(batch.sentences.to(dev), batch.visual.to(dev), batch.acoustic.to(dev),
                           batch.lengths, batch.bert_sent.to(dev), batch.bert_sent_type.to(dev),
                           batch.bert_sent_mask.to(dev))
    out = {k: getattr(model, k) for k in model.OUTPUT_ATTRS}
    out["scores"], out["labels"] = scores, labels
    L = oracle_losses(out, batch.labels.to(dev), cfg)
    L["total"].backward()
    C = Checks("bert_l1")
    C.add("scores", scores, out_r["scores"].detach(), 2e-5)
    for a in ("utt_t_orig", "utt_shared_t", "utt_private_a", "utt_t_recon", "tcp"):
        C.add(a, out[a], out_r[a].detach(), 2e-5)
    for kk in ("cls", "diff", "recon", "sim", "conf", "total"):
        C.add("loss " + kk, L[kk], L_r[kk].detach(), 2e-5)
    for n, p in model.named_parameters():
        if g_r[n] is None:
            C.flag("grad None " + n, p.grad is None)
        elif n.startswith("bertmodel.") and not p.requires_grad:
            C.flag("frozen grad None " + n, p.grad is None)
        elif "key.bias" in n:    # exactly 0 in exact arithmetic (softmax shift invariance): pure noise
            continue
        else:
            C.add("grad " + n, p.grad, g_r[n], 1e-4)
    C.finish()


def test_bert_fused_step_level2(dev):
    """use_bert=True through both levels with the full parity harness (fp64 oracle incl. an fp64
    HF BertModel, kink alignment, None-gradient contract, clip+Adam): the fused level-2 step runs
    the hand-written BERT encoder forward and backward; frozen layers 0-8 (solver.py:69-73) get
    no gradient and stay bit-identical after the step."""
    from mmda_b200 import mosei_config
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build
    cfg = mosei_config(vocab_size=100, batch_size=8, use_bert=True, use_confidNet=True)
    state = {k: v.clone() for k, v in oracle_build(cfg, 31).state_dict().items()}
    batch = batch_for(cfg, seed=32, lengths="shuffled", seq_len=11)
    frozen = lambda n: "bertmodel.encoder.layer" in n and \
        int(n.split("encoder.layer.")[-1].split(".")[0]) <= 8
    _model_checks("bert_l2", cfg, state, batch, dev, None, frozen=frozen)


def test_bert_c4_sequence_length(dev):
    """The C4 sequence shape (BASELINE configs[3]: seq 50 + [CLS]/[SEP] = 52 BERT positions, the
    attention kernels' S = 52 tile) through both levels with the full parity harness against the
    fp64 HF oracle; batch 16 keeps the CPU oracle to seconds (C4's batch 512 only adds rows)."""
    from mmda_b200 import mosei_config
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build
    cfg = mosei_config(vocab_size=100, batch_size=16, use_bert=True, use_confidNet=True)
    state = {k: v.clone() for k, v in oracle_build(cfg, 41).state_dict().items()}
    batch = batch_for(cfg, seed=42, lengths="ragged", seq_len=50)
    assert batch.bert_sent.shape[1] == 52
    frozen = lambda n: "bertmodel.encoder.layer" in n and \
        int(n.split("encoder.layer.")[-1].split(".")[0]) <= 8
    _model_checks("bert_c4_s52", cfg, state, batch, dev, None, frozen=frozen)


@pytest.mark.parametrize("sizes,B,T", [((160, 128, 200), 9, 6), ((96, 33, 260), 41, 5), ((300, 1, 2), 2, 3)])
def test_other_recurrence_plans(dev, sizes, B, T):
    """Hidden sizes that exercise the other cluster plans of the recurrence kernels (cluster of
    2 / 4 CTAs, 8- and 32-row tiles, tcgen05 and SIMT GEMM routing, tiny batch; B=1 is degenerate in the reference itself: CMD of a single sample differentiates sqrt at 0)."""
    from mmda_b200.config import MisaConfig
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build
    cfg = MisaConfig(embedding_size=sizes[0], visual_size=sizes[1], acoustic_size=sizes[2],
                     hidden_size=32, vocab_size=60, batch_size=B, use_confidNet=True)
    state = {k: v.clone() for k, v in oracle_build(cfg, 5).state_dict().items()}
    batch = batch_for(cfg, seed=6, lengths="shuffled", seq_len=T)
    _model_checks(f"plans_{sizes[0]}_{sizes[1]}_{sizes[2]}", cfg, state, batch, dev, None)


@pytest.mark.parametrize("sizes,B,T", [((300, 35, 74), 64, 20), ((96, 33, 160), 41, 5)])
def test_gru_cells(dev, sizes, B, T):
    """rnncell='gru' (reference models.py:39,168-169,177-178; SURVEY.md 8f N4) at MOSEI widths
    (cluster of 8, tcgen05 GEMMs) and at sizes that take the smaller cluster plans."""
    from mmda_b200.config import MisaConfig
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build
    cfg = MisaConfig(embedding_size=sizes[0], visual_size=sizes[1], acoustic_size=sizes[2],
                     hidden_size=32 if sizes[0] < 300 else 128, vocab_size=200, batch_size=B,
                     use_confidNet=True, rnncell="gru")
    state = {k: v.clone() for k, v in oracle_build(cfg, 7).state_dict().items()}
    batch = batch_for(cfg, seed=8, lengths="shuffled", seq_len=T)
    _model_checks(f"gru_{sizes[0]}_{B}", cfg, state, batch, dev, None)


def test_fused_dropout_layernorm_kernels(dev):
    """BERT residual blocks: the fused dropout+LayerNorm forward and LayerNorm-backward+dropout
    kernels against the stand-alone dropout / LayerNorm kernels on the same dropout stream
    (identical masks), including the bf16 operand copies they emit."""
    from mmda_b200.engine import Kernels, _ptr
    k = Kernels(); k.bind_stream()
    g = torch.Generator().manual_seed(8)
    C = Checks("fused_ln")
    for rows, width, p in [(300, 768, 0.1), (65, 1024, 0.3), (41, 128, 0.1), (500, 600, 0.0)]:
        x = torch.randn(rows, width, generator=g).to(dev); res = torch.randn(rows, width, generator=g).to(dev)
        gam = (torch.rand(width, generator=g) + 0.5).to(dev); bet = torch.randn(width, generator=g).to(dev)
        dy = torch.randn(rows, width, generator=g).to(dev)
        # reference: separate kernels
        xd = x.clone()
        if p > 0:
            k.dropout(xd, xd, p, 77, 9, None)
        y0 = torch.empty_like(x); mu0 = torch.empty(rows, device=dev); rs0 = torch.empty(rows, device=dev)
        k.layernorm(xd, res, gam, bet, y0, mu0, rs0)
        dx0 = torch.empty_like(x); dg0 = torch.zeros(width, device=dev); db0 = torch.zeros(width, device=dev)
        k.layernorm_bwd(dy, xd, res, gam, mu0, rs0, dx0, dg0, db0)
        dd0 = dx0.clone()
        if p > 0:
            k.dropout(dx0, dd0, p, 77, 9, None)
        # fused
        x1 = x.clone(); y1 = torch.empty_like(x); yb = torch.empty(rows, width, device=dev, dtype=torch.bfloat16)
        mu1 = torch.empty(rows, device=dev); rs1 = torch.empty(rows, device=dev)
        k._c("mmda_dropout_layernorm_forward", _ptr(x1), width, _ptr(res), width, _ptr(gam), _ptr(bet),
             _ptr(y1), width, _ptr(yb), _ptr(mu1), _ptr(rs1), rows, width, 1e-5, p, 77, None, 9)
        assert torch.equal(x1, xd), "dropout mask / scaling differs from the stand-alone kernel"
        C.add(f"fused ln fwd {rows}x{width}", y1, y0, 2e-6)
        assert torch.equal(yb, y1.to(torch.bfloat16))
        dx1 = torch.empty_like(x); dg1 = torch.zeros(width, device=dev); db1 = torch.zeros(width, device=dev)
        dd1 = torch.empty_like(x); ddb = torch.empty(rows, width, device=dev, dtype=torch.bfloat16)
        k._c("mmda_layernorm_backward_dropout", _ptr(dy), width, _ptr(x1), width, _ptr(res), width, _ptr(gam),
             _ptr(mu1), _ptr(rs1), _ptr(dx1), width, _ptr(dg1), _ptr(db1), rows, width, _ptr(dd1), _ptr(ddb),
             p, 77, None, 9)
        C.add(f"fused ln dx {rows}x{width}", dx1, dx0, 5e-6)
        C.add(f"fused ln dropped dx {rows}x{width}", dd1, dd0, 5e-6)
        assert torch.equal((dd1 == 0), (dd0 == 0)) or p == 0
        assert torch.equal(ddb, dd1.to(torch.bfloat16))
        C.add(f"fused ln dgamma {rows}x{width}", dg1, dg0, 5e-6)
        C.add(f"fused ln dbeta {rows}x{width}", db1, db0, 5e-6)
    C.finish()


def test_bert_attention_tensor_core_kernels(dev):
    """bf16-mode attention core (mma.sync) vs fp64 math built from the bf16-rounded operands'
    fp32 originals: forward context / probabilities and the three input gradients within the
    2e-2 bf16 bar (relative to the tensor's max); with dropout on, against the fp32 SIMT kernels
    of the same dropout stream."""
    from mmda_b200.engine import Kernels, _ptr
    k = Kernels(); k.bind_stream()
    g = torch.Generator().manual_seed(3)
    C = Checks("bert_attn_mma")
    for B, S, nh in [(3, 52, 12), (2, 64, 12), (5, 11, 12), (4, 17, 2)]:
        Hd = nh * 64
        qkv = (torch.randn(B * S, 3 * Hd, generator=g) * 1.5).to(dev)
        mask = torch.ones(B, S, dtype=torch.int64)
        for bi in range(B):
            mask[bi, S - (bi * 3) % S:] = 0 if bi else 1          # right-padded samples
        mask = mask.to(dev)
        do = torch.randn(B * S, Hd, generator=g).to(dev)
        ctx = torch.empty(B * S, Hd, device=dev); pr = torch.empty(B, nh, S, S, device=dev)
        ctx_bf = torch.empty(B * S, Hd, device=dev, dtype=torch.bfloat16)
        k._c("mmda_bert_attention_forward_mma", _ptr(qkv), _ptr(mask), _ptr(ctx), _ptr(ctx_bf), _ptr(pr),
             B, S, nh, 64, 0.0, 1, None, 7)
        assert torch.equal(ctx_bf, ctx.to(torch.bfloat16))
        q3 = qkv.double().view(B, S, 3, nh, 64).requires_grad_(True)
        q, kk, v = q3[:, :, 0], q3[:, :, 1], q3[:, :, 2]
        s = torch.einsum("bihd,bjhd->bhij", q, kk) / 8.0
        s = s.masked_fill(mask[:, None, None, :] == 0, float("-inf"))
        p = torch.softmax(s, -1)
        o = torch.einsum("bhij,bjhd->bihd", p, v).reshape(B * S, Hd)
        o.backward(do.double())
        C.add(f"ctx B={B} S={S} nh={nh}", ctx, o, 2e-2)
        C.add(f"probs B={B} S={S} nh={nh}", pr, p, 2e-2)
        dqkv = torch.full_like(qkv, float("nan"))
        dq_bf = torch.empty(B * S, 3 * Hd, device=dev, dtype=torch.bfloat16)
        k._c("mmda_bert_attention_backward_mma", _ptr(qkv), _ptr(pr), _ptr(do), _ptr(dqkv), _ptr(dq_bf),
             B, S, nh, 64, 0.0, 1, None, 7)
        assert torch.equal(dq_bf, dqkv.to(torch.bfloat16))
        gq = q3.grad.reshape(B * S, 3, Hd)
        for j, nm in enumerate(("dQ", "dK", "dV")):
            C.add(f"{nm} B={B} S={S} nh={nh}", dqkv.view(B * S, 3, Hd)[:, j], gq[:, j], 2e-2)
        # dropout on: same stream -> same mask as the fp32 kernels
        ctx1 = torch.empty_like(ctx); pr1 = torch.empty_like(pr); d1 = torch.empty_like(qkv)
        ctx2 = torch.empty_like(ctx); pr2 = torch.empty_like(pr); d2 = torch.empty_like(qkv)
        for sfx, (c_, p_, d_) in (("", (ctx1, pr1, d1)), ("_mma", (ctx2, pr2, d2))):
            k._c("mmda_bert_attention_forward" + sfx, _ptr(qkv), _ptr(mask), _ptr(c_),
                 *((None,) if sfx else ()), _ptr(p_), B, S, nh, 64, 0.1, 99, None, 5)
            k._c("mmda_bert_attention_backward" + sfx, _ptr(qkv), _ptr(p_), _ptr(do), _ptr(d_),
                 *((None,) if sfx else ()), B, S, nh, 64, 0.1, 99, None, 5)
        C.add(f"dropout ctx B={B} S={S}", ctx2, ctx1, 2e-2)
        C.add(f"dropout dqkv B={B} S={S}", d2, d1, 2e-2)
    C.finish()


def test_bert_bf16_mode_within_2e2(dev):
    """precision='bf16' on the BERT branch (BASELINE configs[3]): every dense layer of the encoder
    runs forward and backward with bf16 operands / fp32 accumulation.  Outputs and losses within
    the 2e-2 bf16 bar of the fp32 oracle; gradients are checked for direction (cosine) because
    bf16 operand rounding makes their element-wise error ill-conditioned (see the C3 test)."""
    from mmda_b200 import MISA, FusedTrainer, mosei_config
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build, oracle_step
    cfg = mosei_config(vocab_size=100, batch_size=8, use_bert=True, precision="bf16")
    ref = oracle_build(cfg, 51).eval()
    state = {k: v.clone() for k, v in ref.state_dict().items()}
    batch = batch_for(cfg, seed=52, lengths="shuffled", seq_len=11)
    out_r, L_r, g_r = oracle_step(ref, batch, cfg, None)
    model = MISA(cfg)
    model.load_state_dict(state)
    model = model.to(dev).eval()
    tr = FusedTrainer(model)
    L = tr.forward_backward(batch.sentences.to(dev), batch.visual.to(dev), batch.acoustic.to(dev),
                            batch.lengths, batch.labels.to(dev),
                            (batch.bert_sent.to(dev), batch.bert_sent_type.to(dev),
                             batch.bert_sent_mask.to(dev))).cpu()
    C = Checks("bert_bf16")
    for i, kk in enumerate(("cls", "diff", "sim", "recon", "total")):
        idx = {"cls": 0, "diff": 1, "sim": 2, "recon": 3, "total": 5}[kk]
        C.add("loss " + kk, L[idx], L_r[kk].detach(), 2e-2)
    C.add("utterance_text (BERT masked mean)", tr.eng.ws["bert_utt"][:8 * 768].view(8, 768),
          out_r["utterance_t"].detach(), 2e-2)
    for n in ("project_t.project_t.weight", "bertmodel.encoder.layer.11.output.dense.weight",
              "bertmodel.encoder.layer.9.intermediate.dense.weight",
              "bertmodel.embeddings.position_embeddings.weight"):
        a, b = tr.G[n].detach().cpu().double().flatten(), g_r[n].double().flatten()
        cos = float((a @ b) / (a.norm() * b.norm() + 1e-30))
        C.flag(f"grad direction {n} cos={cos:.5f}", cos > 0.99)
    C.finish()


def test_checkpoint_resume_matches_uninterrupted_run(dev):
    """src/solver.py:219-220: model + optimizer state_dict saved after step 3, loaded into a fresh
    model / trainer (through torch.optim.Adam's own layout, as the reference's checkpoint files hold
    it) and resumed: steps 4..6 -- train mode, so the dropout stream is part of the state -- match
    the uninterrupted run."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=300, batch_size=32, use_confidNet=True)
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
    # the optimizer checkpoint is a genuine torch.optim.Adam state: pass it through one
    adam = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1.0)
    adam.load_state_dict(ckpt_optim)
    ckpt_optim = adam.state_dict()
    ref = [step(tr, b) for b in batches[3:]]
    ref_params = tr.p_arena[:tr.n_active].clone().cpu()

    torch.manual_seed(12)                                  # different init: everything comes from the files
    model2 = MISA(cfg).to(dev).train()
    model2.load_state_dict(ckpt_model)
    tr2 = FusedTrainer(model2, use_graph=False)
    tr2.load_optimizer_state_dict(ckpt_optim)
    assert tr2.step_count == 3 and tr2.lr == cfg.learning_rate
    got = [step(tr2, b) for b in batches[3:]]
    C = Checks("checkpoint_resume")
    C.add("losses of steps 4..6", torch.stack(got), torch.stack(ref), 1e-5)
    dp = float((tr2.p_arena[:tr2.n_active].cpu() - ref_params).abs().max())
    C.rows.append((f"parameters after step 6: max |delta| = {dp:.3e} <= 2*lr*steps", dp,
                   2 * cfg.learning_rate * 3, dp <= 2 * cfg.learning_rate * 3))
    C.finish()
