"""BERT text branch beyond the shared-memory resident attention kernels (S > 84 in training, S > 116
in eval), up to bert-base's 512 positions.  The tiled attention kernels (csrc/bert.cu,
mmda_bert_attention_{forward,backward}_tiled[_mma]) are checked through the C ABI against fp64
math that applies the exact dropout mask (the generator of csrc/common.cuh, restated below), against
the resident kernels on the same dropout stream, and for run-to-run determinism; then the whole
model trains and evaluates at long sequences against the fp64 HF oracle."""
import numpy as np
import pytest
import torch

from test_gpu_parity import Checks, _model_checks

pytestmark = pytest.mark.gpu

SEED = 0x1234_5678_9ABC_DEF1
M32 = np.uint64(0xFFFFFFFF)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return torch.device("cuda:0")


# ---- the dropout generator of csrc/common.cuh (mix32 / rng_uniform), uint32 arithmetic ----
def mix32(x):
    x = x & M32
    x ^= x >> np.uint64(16); x = (x * np.uint64(0x7FEB352D)) & M32
    x ^= x >> np.uint64(15); x = (x * np.uint64(0x846CA68B)) & M32
    x ^= x >> np.uint64(16)
    return x


def rng_uniform(seed, stream, idx):
    h = mix32(np.uint64(seed & 0xFFFFFFFF) ^ mix32(idx + np.uint64((0x9E3779B9 * (stream + 1)) & 0xFFFFFFFF)))
    h = mix32(h ^ np.uint64(seed >> 32) ^ np.uint64((stream * 0x85EBCA6B) & 0xFFFFFFFF))
    return (h >> np.uint64(8)).astype(np.float64) / 16777216.0


def drop_factor(B, nh, S, p, seed, stream):
    """[B][nh][S][S] float64: 0 where element (b, h, i, j) is dropped, else 1 / (1 - p) in fp32"""
    idx = np.arange(B * nh * S * S, dtype=np.uint64)       # (b*nh + h)*S*S + i*S + j
    keep = rng_uniform(seed, stream, idx) >= float(np.float32(p))
    inv = float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))
    return torch.from_numpy(np.where(keep, inv, 0.0).reshape(B, nh, S, S))


def test_dropout_restatement_matches_the_device_generator(dev):
    """mmda_dropout draws element e at rng_uniform(seed, stream, e): its mask is the restatement's"""
    from mmda_b200.engine import Kernels
    k = Kernels(); k.bind_stream()
    x = torch.ones(3000, device=dev)
    y = torch.empty_like(x)
    k.dropout(x, y, 0.3, SEED, 17, None)
    keep = rng_uniform(SEED, 17, np.arange(3000, dtype=np.uint64)) >= float(np.float32(0.3))
    assert torch.equal((y.cpu() != 0), torch.from_numpy(keep))


def _masks(B, S, case):
    """right-padded samples; one with only [CLS] valid; one whose valid keys all sit in the first
    64-key tile; one whose valid keys all sit beyond it (the first tile a row sees is masked)"""
    g = torch.Generator().manual_seed(1000 + case)
    mask = torch.ones(B, S, dtype=torch.int64)
    for b in range(B):
        kind = (b + case) % 5
        if kind == 1:
            mask[b, 1:] = 0
        elif kind == 2:
            mask[b, min(S, 37):] = 0
        elif kind == 3 and S > 64:
            mask[b, :64] = 0
            mask[b, S - 5:] = 0
        elif kind == 4:
            mask[b, int(torch.randint(1, S + 1, (1,), generator=g)):] = 0
    return mask


def _inputs(B, S, nh, case, dev):
    g = torch.Generator().manual_seed(7 * case + S)
    qkv = (torch.randn(B * S, 3 * nh * 64, generator=g) * 1.5).to(dev)
    do = torch.randn(B * S, nh * 64, generator=g).to(dev)
    return qkv, _masks(B, S, case).to(dev), do


def _reference(qkv, mask, do, nh, p, stream):
    """fp64 attention from the same fp32 inputs: ctx, lse, d(qkv)"""
    B, S = mask.shape
    q3 = qkv.double().view(B, S, 3, nh, 64).requires_grad_(True)
    q, kk, v = q3[:, :, 0], q3[:, :, 1], q3[:, :, 2]
    s = torch.einsum("bihd,bjhd->bhij", q, kk) / 8.0
    s = s.masked_fill(mask[:, None, None, :] == 0, float("-inf"))
    lse = torch.logsumexp(s, -1)
    pr = torch.softmax(s, -1)
    if p > 0:
        pr = pr * drop_factor(B, nh, S, p, SEED, stream).to(qkv.device)
    o = torch.einsum("bhij,bjhd->bihd", pr, v).reshape(B * S, nh * 64)
    o.backward(do.double())
    return o.detach(), lse.detach(), q3.grad.reshape(B * S, 3 * nh * 64)


def _tiled(k, qkv, mask, do, nh, p, stream, mma):
    from mmda_b200.engine import _ptr
    B, S = mask.shape
    dev = qkv.device
    nan = float("nan")
    ctx = torch.full((B * S, nh * 64), nan, device=dev)
    lse = torch.full((B, nh, S), nan, device=dev)
    delta = torch.full((B, nh, S), nan, device=dev)
    dqkv = torch.full_like(qkv, nan)
    out = dict(ctx=ctx, lse=lse, dqkv=dqkv)
    if mma:
        ctx_bf = torch.full((B * S, nh * 64), nan, device=dev, dtype=torch.bfloat16)
        dq_bf = torch.full((B * S, 3 * nh * 64), nan, device=dev, dtype=torch.bfloat16)
        k._c("mmda_bert_attention_forward_tiled_mma", _ptr(qkv), _ptr(mask), _ptr(ctx), _ptr(ctx_bf),
             _ptr(lse), B, S, nh, 64, p, SEED, None, stream)
        k._c("mmda_bert_attention_backward_tiled_mma", _ptr(qkv), _ptr(mask), _ptr(ctx), _ptr(lse),
             _ptr(do), _ptr(delta), _ptr(dqkv), _ptr(dq_bf), B, S, nh, 64, p, SEED, None, stream)
        out.update(ctx_bf=ctx_bf, dq_bf=dq_bf)
    else:
        k._c("mmda_bert_attention_forward_tiled", _ptr(qkv), _ptr(mask), _ptr(ctx), _ptr(lse),
             B, S, nh, 64, p, SEED, None, stream)
        k._c("mmda_bert_attention_backward_tiled", _ptr(qkv), _ptr(mask), _ptr(ctx), _ptr(lse),
             _ptr(do), _ptr(delta), _ptr(dqkv), B, S, nh, 64, p, SEED, None, stream)
    torch.cuda.synchronize()
    return out


SHAPES = [(2, 85, 12), (3, 130, 12), (2, 257, 2), (4, 200, 12), (1, 512, 12)]


@pytest.mark.parametrize("mma", [False, True], ids=["fp32", "bf16"])
@pytest.mark.parametrize("p", [0.0, 0.1])
def test_tiled_kernels_vs_fp64(dev, mma, p):
    from mmda_b200.engine import Kernels
    k = Kernels(); k.bind_stream()
    tol = 2e-2 if mma else 1e-5
    C = Checks(f"bert_tiled_{'bf16' if mma else 'fp32'}_p{p}")
    for case, (B, S, nh) in enumerate(SHAPES):
        qkv, mask, do = _inputs(B, S, nh, case, dev)
        stream = 201 + 4 * case
        o, lse, dq = _reference(qkv, mask, do, nh, p, stream)
        got = _tiled(k, qkv, mask, do, nh, p, stream, mma)
        tag = f"B={B} S={S} nh={nh}"
        C.add(f"ctx {tag}", got["ctx"], o, tol)
        C.add(f"lse {tag}", got["lse"], lse, tol)
        H = nh * 64
        for j, nm in enumerate(("dQ", "dK", "dV")):
            C.add(f"{nm} {tag}", got["dqkv"][:, j * H:(j + 1) * H], dq[:, j * H:(j + 1) * H], tol)
        if mma:
            C.flag(f"ctx bf16 copy {tag}", torch.equal(got["ctx_bf"], got["ctx"].to(torch.bfloat16)))
            C.flag(f"dqkv bf16 copy {tag}", torch.equal(got["dq_bf"], got["dqkv"].to(torch.bfloat16)))
    for n, e, b, ok in C.rows:
        print(f"{'ok  ' if ok else 'FAIL'} {n:40s} err={e:.3e} bound={b:.1e}")
    C.finish()


def _resident(k, qkv, mask, do, nh, p, stream, mma):
    from mmda_b200.engine import _ptr
    B, S = mask.shape
    sfx = "_mma" if mma else ""
    ctx = torch.empty(B * S, nh * 64, device=qkv.device)
    probs = torch.empty(B, nh, S, S, device=qkv.device)
    dqkv = torch.empty_like(qkv)
    k._c("mmda_bert_attention_forward" + sfx, _ptr(qkv), _ptr(mask), _ptr(ctx),
         *((None,) if mma else ()), _ptr(probs), B, S, nh, 64, p, SEED, None, stream)
    k._c("mmda_bert_attention_backward" + sfx, _ptr(qkv), _ptr(probs), _ptr(do), _ptr(dqkv),
         *((None,) if mma else ()), B, S, nh, 64, p, SEED, None, stream)
    torch.cuda.synchronize()
    return ctx, dqkv


@pytest.mark.parametrize("S,mma", [(17, False), (52, False), (84, False), (52, True), (64, True)])
def test_same_dropout_stream_as_resident_kernels(dev, S, mma):
    from mmda_b200.engine import Kernels
    k = Kernels(); k.bind_stream()
    tol = 2e-2 if mma else 1e-5
    C = Checks(f"bert_tiled_vs_resident_S{S}_{'bf16' if mma else 'fp32'}")
    B, nh = 3, 12
    qkv, mask, do = _inputs(B, S, nh, 2, dev)
    c0, d0 = _resident(k, qkv, mask, do, nh, 0.1, 205, mma)
    got = _tiled(k, qkv, mask, do, nh, 0.1, 205, mma)
    C.add(f"ctx S={S}", got["ctx"], c0, tol)
    C.add(f"dqkv S={S}", got["dqkv"], d0, tol)
    for n, e, b, ok in C.rows:
        print(f"{'ok  ' if ok else 'FAIL'} {n:40s} err={e:.3e} bound={b:.1e}")
    C.finish()


@pytest.mark.parametrize("mma", [False, True], ids=["fp32", "bf16"])
def test_tiled_kernels_are_deterministic(dev, mma):
    from mmda_b200.engine import Kernels
    k = Kernels(); k.bind_stream()
    qkv, mask, do = _inputs(2, 512, 12, 4, dev)
    a = _tiled(k, qkv, mask, do, 12, 0.1, 9, mma)
    b = _tiled(k, qkv, mask, do, 12, 0.1, 9, mma)
    for n in a:
        assert torch.equal(a[n], b[n]), n
        assert not torch.isnan(a[n]).any(), n


def _frozen(n):
    return "bertmodel.encoder.layer" in n and int(n.split("encoder.layer.")[-1].split(".")[0]) <= 8


@pytest.mark.parametrize("seq_len,B", [(128, 4), (510, 2)])
def test_whole_model_fp32_long_sequences(dev, seq_len, B):
    """The full 1e-5 harness (both levels, fp64 HF oracle, freeze contract) with the BERT branch on
    the tiled attention kernels; 'ragged' lengths keep one full-length sample."""
    from mmda_b200 import mosei_config
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build
    cfg = mosei_config(vocab_size=100, batch_size=B, use_bert=True, use_confidNet=True)
    state = {k: v.clone() for k, v in oracle_build(cfg, 61).state_dict().items()}
    batch = batch_for(cfg, seed=62, lengths="ragged", seq_len=seq_len)
    assert batch.bert_sent.shape[1] == seq_len + 2
    assert int(batch.bert_sent_mask.sum(1).max()) == seq_len + 2
    _model_checks(f"bert_long_s{seq_len + 2}", cfg, state, batch, dev, None, frozen=_frozen)


def test_whole_model_bf16_s200(dev):
    """precision='bf16' at S = 200 (the _tiled_mma pair): the checks of the S = 13 bf16 test."""
    from mmda_b200 import MISA, FusedTrainer, mosei_config
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build, oracle_step
    cfg = mosei_config(vocab_size=100, batch_size=8, use_bert=True, precision="bf16")
    ref = oracle_build(cfg, 51).eval()
    state = {k: v.clone() for k, v in ref.state_dict().items()}
    batch = batch_for(cfg, seed=52, lengths="shuffled", seq_len=198)
    out_r, L_r, g_r = oracle_step(ref, batch, cfg, None)
    model = MISA(cfg)
    model.load_state_dict(state)
    model = model.to(dev).eval()
    tr = FusedTrainer(model)
    L = tr.forward_backward(batch.sentences.to(dev), batch.visual.to(dev), batch.acoustic.to(dev),
                            batch.lengths, batch.labels.to(dev),
                            (batch.bert_sent.to(dev), batch.bert_sent_type.to(dev),
                             batch.bert_sent_mask.to(dev))).cpu()
    assert "bert_lse_0" in tr.eng.ws and not [n for n in tr.eng.ws if n.startswith("bert_probs_")]
    C = Checks("bert_bf16_s200")
    for kk in ("cls", "diff", "sim", "recon", "total"):
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


@pytest.mark.parametrize("seq_len", [128, 298])
def test_eval_pass_long_sequences(dev, seq_len):
    """evaluate() with the BERT branch at S = 130 / 300 (tiled forward, no lse) against the
    oracle's cls loss and metrics."""
    from sklearn import metrics as M
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.evaluate import evaluate
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import OracleMISA, oracle_losses
    cfg = mosei_config(vocab_size=100, batch_size=6, use_bert=True, threshold=0.5)
    torch.manual_seed(13)
    model = MISA(cfg)
    state = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.to(dev)
    batches = [batch_for(cfg, seed=70 + i, lengths="ragged", seq_len=seq_len) for i in range(2)]
    got = evaluate(model, batches)
    assert not [n for n in model.engine.ws if n.startswith(("bert_probs_", "bert_lse_"))]
    ref = OracleMISA(cfg); ref.load_state_dict(state); ref.eval()
    ys, ps, losses = [], [], []
    with torch.no_grad():
        for b in batches:
            out = ref(*b.model_args())
            losses.append(float(oracle_losses(out, b.labels, cfg)["cls"]))
            ys.append(b.labels.numpy()); ps.append(out["labels"].numpy())
    y, p = np.concatenate(ys), np.concatenate(ps)
    jac = np.mean((y * p).sum(1) / np.maximum(((y + p) > 0).sum(1), 1))
    assert abs(got["loss"] - np.mean(losses)) < 1e-5 * np.mean(losses)
    assert abs(got["acc"] - round(float(jac), 4)) <= 1e-4
    assert abs(got["f1"] - M.f1_score(y, p, average="macro", zero_division=0)) < 1e-6
    assert abs(got["micro_precision"] - M.precision_score(y, p, average="micro", zero_division=0)) < 1e-6
    assert abs(got["weighted_recall"] - M.recall_score(y, p, average="weighted", zero_division=0)) < 1e-6


def test_s513_raises_at_the_position_embeddings(dev):
    from mmda_b200 import MISA, mosei_config
    from mmda_b200._lib import MmdaError
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=100, batch_size=2, use_bert=True)
    torch.manual_seed(0)
    model = MISA(cfg).to(dev)
    b = batch_for(cfg, seed=1, lengths="ragged", seq_len=511)
    assert b.bert_sent.shape[1] == 513
    tr = FusedTrainer(model)
    with pytest.raises(MmdaError, match="position embeddings"):
        tr.forward_backward(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths,
                            b.labels.to(dev), (b.bert_sent.to(dev), b.bert_sent_type.to(dev),
                                               b.bert_sent_mask.to(dev)))
    torch.cuda.synchronize()
