"""Deterministic mode on the B200: the fixed-order reduction kernels against fp64 and bitwise over
repeated launches, and whole training steps / level-1 backward / evaluate bit-identical run to run
while torch.use_deterministic_algorithms(True) is on."""
import pytest
import torch

from mmda_b200._lib import LIB

pytestmark = pytest.mark.gpu


@pytest.fixture
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch.device("cuda")


@pytest.fixture
def det():
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(False)


def _p(t):
    return None if t is None else t.data_ptr()


def _ws(query, *args):
    """workspace filled with NaN: a kernel that reads scratch it did not write returns NaN"""
    n = int(LIB.raw(query)(*args))
    return torch.full((max(n // 4, 4),), float("nan"), dtype=torch.float32, device="cuda")


def _call(name, *args):
    LIB.call(name, *args, torch.cuda.current_stream().cuda_stream)


def _repeat_bitwise(run, n=3):
    """run() -> tensor; identical bits on every launch, and with other work on a second stream"""
    ref = run().clone()
    side = torch.cuda.Stream()
    big = torch.randn(4096, 4096, device="cuda")
    for i in range(n):
        with torch.cuda.stream(side):
            for _ in range(2):
                big = big @ big.t() * 1e-4
        out = run()
        assert torch.equal(out, ref), i
    torch.cuda.synchronize()
    return ref


def _pad_rows(x, extra):
    return torch.cat([x, torch.zeros(extra, *x.shape[1:], device=x.device, dtype=x.dtype)])


@pytest.mark.parametrize("rows,cols,ilv", [(1, 7, 0), (37, 130, 0), (12800, 1024, 256), (1536, 128, 0)])
def test_colsum_det(dev, rows, cols, ilv):
    g = torch.Generator(device="cpu").manual_seed(rows)
    x = torch.randn(rows, cols, generator=g).to(dev)
    base = torch.randn(cols, generator=g).to(dev)

    def launch(x):
        ws = _ws("mmda_colsum_det_workspace_bytes", x.shape[0], cols)
        out, out2 = base.clone(), base.clone()
        _call("mmda_colsum_det", _p(x), cols, x.shape[0], cols, _p(out), _p(out2), ilv, _p(ws))
        assert torch.equal(out, out2)
        return out
    out = _repeat_bitwise(lambda: launch(x))
    # zero rows appended (a padded launch) change no bit
    assert torch.equal(launch(_pad_rows(x, 300)), out)
    ref = x.double().sum(0)
    if ilv:
        c = torch.arange(cols, device=dev)
        ref = torch.zeros_like(ref).index_copy_(0, (c % 4) * ilv + c // 4, ref)
    ref = ref + base.double()
    assert (out.double() - ref).abs().max() <= 1e-5 * ref.abs().max() + 1e-5


def _ln_inputs(rows, width, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x, dy = torch.randn(rows, width, generator=g).cuda(), torch.randn(rows, width, generator=g).cuda()
    gamma = torch.randn(width, generator=g).cuda()
    mu = x.mean(1)
    rs = 1.0 / torch.sqrt(x.var(1, unbiased=False) + 1e-5)
    return x, dy, gamma, mu, rs


@pytest.mark.parametrize("rows,width", [(1, 128), (1536, 128), (12800, 256), (1000, 70), (600, 768)])
def test_layernorm_backward_det(dev, rows, width):
    x, dy, gamma, mu, rs = _ln_inputs(rows, width, width)

    def launch(x, dy, mu, rs):
        n = x.shape[0]
        ws = _ws("mmda_layernorm_backward_det_workspace_bytes", n, width)
        dx = torch.empty_like(x)
        dg, db = torch.ones(width, device=dev), torch.ones(width, device=dev)
        _call("mmda_layernorm_backward_det", _p(dy), width, _p(x), width, None, 0, _p(gamma), _p(mu),
              _p(rs), _p(dx), width, _p(dg), _p(db), n, width, _p(ws))
        return torch.cat([dg, db, dx[:rows].flatten()])
    out = _repeat_bitwise(lambda: launch(x, dy, mu, rs))
    # padded rows: zero gradient, finite activations
    e = 130
    assert torch.equal(launch(_pad_rows(x, e) + 0, _pad_rows(dy, e), torch.cat([mu, torch.zeros(e, device=dev)]),
                              torch.cat([rs, torch.ones(e, device=dev)])), out)
    xh = (x.double() - mu.double()[:, None]) * rs.double()[:, None]
    ref_g = (dy.double() * xh).sum(0) + 1
    ref_b = dy.double().sum(0) + 1
    assert (out[:width].double() - ref_g).abs().max() <= 1e-5 * ref_g.abs().max()
    assert (out[width:2 * width].double() - ref_b).abs().max() <= 1e-5 * ref_b.abs().max()


@pytest.mark.parametrize("rows,width,p", [(1664, 768, 0.1), (1040, 768, 0.0), (520, 256, 0.1)])
def test_layernorm_backward_dropout_det(dev, rows, width, p):
    """the BERT encoder's LayerNorm backward with dropout(dx): same dx / dropped dx as the atomic
    entry, dgamma / dbeta against fp64, bitwise repeats"""
    x, dy, gamma, mu, rs = _ln_inputs(rows, width, rows)
    outs = {}
    for det in (False, True):
        def launch():
            dx, dd = torch.empty_like(x), torch.empty_like(x)
            dbf = torch.empty(rows, width, dtype=torch.bfloat16, device=dev)
            dg, db = torch.zeros(width, device=dev), torch.zeros(width, device=dev)
            args = (_p(dy), width, _p(x), width, None, 0, _p(gamma), _p(mu), _p(rs), _p(dx), width,
                    _p(dg), _p(db), rows, width, _p(dd), _p(dbf), p, 77, None, 5)
            if det:
                ws = _ws("mmda_layernorm_backward_det_workspace_bytes", rows, width)
                _call("mmda_layernorm_backward_dropout_det", *args, _p(ws))
            else:
                _call("mmda_layernorm_backward_dropout", *args)
            return torch.cat([dg, db, dx.flatten(), dd.flatten(), dbf.float().flatten()])
        outs[det] = _repeat_bitwise(launch) if det else launch()
    n = 2 * width
    assert torch.equal(outs[True][n:], outs[False][n:])
    xh = (x.double() - mu.double()[:, None]) * rs.double()[:, None]
    ref = torch.cat([(dy.double() * xh).sum(0), dy.double().sum(0)])
    assert (outs[True][:n].double() - ref).abs().max() <= 1e-5 * ref.abs().max()


@pytest.mark.parametrize("M,N,K,ilv", [(1200, 300, 12800, 300), (512, 256, 4096, 0), (132, 36, 640, 0),
                                       (132, 36, 2048, 0), (1280, 1280, 9000, 0), (64, 64, 100, 0)])
def test_gemm_tc_det_split_k(dev, M, N, K, ilv):
    """dW += dG^T X over the token axis (both operands MN-major, the LSTM weight-gradient shape):
    1, 2, 4, 5 and 13 slices; K padded with zero rows gives the same bits"""
    g = torch.Generator(device="cpu").manual_seed(M + K)
    A = torch.randn(K, M, generator=g).to(dev)       # [K][M]
    B = torch.randn(K, N, generator=g).to(dev)       # [K][N]
    C0 = torch.randn(M, N, generator=g).to(dev)

    def launch(A, B):
        k = A.shape[0]
        ws = _ws("mmda_gemm_tc_det_workspace_bytes", 2, M, N, k, 1, 0)
        C = C0.clone()
        _call("mmda_gemm_tc_det", 2, 1, 1, M, N, k, _p(A), None, M, _p(B), None, N, 1.0, _p(C), N,
              None, None, 1, 0, ilv, _p(ws))
        return C
    out = _repeat_bitwise(lambda: launch(A, B))
    for extra in (7, 1100):
        assert torch.equal(launch(_pad_rows(A, extra), _pad_rows(B, extra)), out), extra
    ref = A.double().t() @ B.double()
    if ilv:
        r = torch.arange(M, device=dev)
        ref = torch.zeros_like(ref).index_copy_(0, (r % 4) * ilv + r // 4, ref)
    ref = ref + C0.double()
    assert (out.double() - ref).abs().max() <= 1e-5 * ref.abs().max()


def test_embedding_backward_det(dev):
    """repeated ids (one id in a third of the rows), absent ids, an out-of-range id; rows appended
    at the end with zero gradient (a padded launch) change no bit"""
    T, B, D, V = 40, 32, 300, 500
    g = torch.Generator(device="cpu").manual_seed(3)
    sent = torch.randint(0, V // 2, (T, B), generator=g)
    sent[::3] = 7
    sent[0, 0] = V + 5
    N = T * B
    dX = torch.randn(N, D, generator=g)
    base = torch.randn(V, D, generator=g)
    sent_d = sent.to(dev)

    def launch(n_rows, dX):
        row_t = (torch.arange(n_rows, dtype=torch.int32) // B).clamp_max(T - 1).to(dev)
        row_j = (torch.arange(n_rows, dtype=torch.int32) % B).to(dev)
        sidx = torch.arange(B, dtype=torch.int32, device=dev)
        ws = _ws("mmda_embedding_backward_det_workspace_bytes", n_rows, V)
        dE = base.to(dev)
        _call("mmda_embedding_backward_det", _p(dE), _p(sent_d), _p(dX), _p(row_t), _p(row_j),
              _p(sidx), n_rows, B, D, V, _p(ws))
        return dE
    dX_d = dX.to(dev)
    out = _repeat_bitwise(lambda: launch(N, dX_d))
    assert torch.equal(launch(N + 100, _pad_rows(dX_d, 100)), out)
    ids = sent.flatten()
    ok = ids < V
    ref = base.double().index_add(0, ids[ok], dX.double()[ok])
    assert (out.cpu().double() - ref).abs().max() <= 1e-5 * ref.abs().max()
    absent = torch.ones(V, dtype=torch.bool)
    absent[ids[ok]] = False
    assert torch.equal(out.cpu()[absent], base[absent])


@pytest.mark.parametrize("B,S", [(4, 52), (3, 130)])
def test_bert_embed_backward_det(dev, B, S):
    H, V = 768, 30522
    g = torch.Generator(device="cpu").manual_seed(S)
    ids = torch.randint(0, 3000, (B, S), generator=g)
    ids[:, -5:] = 0                                   # padding positions
    ids[:, 1::4] = 1012                               # a frequent token
    types = (torch.rand(B, S, generator=g) < 0.4).long()
    d = torch.randn(B * S, H, generator=g)
    ids_d, types_d, d_d = ids.to(dev), types.to(dev), d.to(dev)
    bw, bp, bt = (torch.randn(V, H, generator=g), torch.randn(512, H, generator=g),
                  torch.randn(2, H, generator=g))

    def run():
        w, p, t = bw.to(dev), bp.to(dev), bt.to(dev)
        ws = _ws("mmda_bert_embed_backward_det_workspace_bytes", B, S, H, V)
        _call("mmda_bert_embed_backward_det", _p(d_d), _p(ids_d), _p(types_d), B, S, H, V, _p(w), _p(p),
              _p(t), _p(ws))
        return torch.cat([w.flatten(), p.flatten(), t.flatten()])
    out = _repeat_bitwise(run).cpu().double()
    fi, dd = ids.flatten(), d.double()
    ok = fi > 0
    rw = bw.double().index_add(0, fi[ok], dd[ok])
    rp = bp.double().clone()
    rp[:S] += dd.view(B, S, H).sum(0)
    rt = bt.double().index_add(0, types.flatten(), dd)
    ref = torch.cat([rw.flatten(), rp.flatten(), rt.flatten()])
    assert (out - ref).abs().max() <= 1e-5 * ref.abs().max()
    assert torch.equal(out[:H], bw.double()[0])      # padding_idx 0 gets no gradient


@pytest.mark.parametrize("B", [1, 37, 256])
def test_loss_det_entries(dev, B):
    """DiffLoss / CMD statistics against fp64 (moments from X0; DXN and colsum2 from the kernel's
    own XN and Gm) and bitwise over repeats"""
    d = 128
    g = torch.Generator(device="cpu").manual_seed(B)
    X0 = torch.randn(B, 6, d, generator=g).to(dev)
    segA = X0.sum(0).flatten().contiguous()
    Gm = torch.randn(6, d, d, generator=g).to(dev)
    alpha = 0.5

    def run():
        XN, inv = torch.zeros(6, B, d, device=dev), torch.zeros(6, B, device=dev)
        mom = torch.zeros(12 * d, device=dev)
        DXN, c2 = torch.full((6, B, d), float("nan"), device=dev), torch.zeros(6 * d, device=dev)
        ws = _ws("mmda_loss_det_workspace_bytes", B, d)
        _call("mmda_loss_phase2_det", _p(X0), _p(segA), _p(XN), _p(inv), _p(mom), B, d, float(B), _p(ws))
        _call("mmda_loss_dxn_det", _p(XN), _p(Gm), _p(DXN), B, d, alpha)
        dxn_pre = DXN.clone()
        _call("mmda_loss_phase4a_det", _p(DXN), _p(inv), _p(c2), B, d, _p(ws))
        return torch.cat([mom, XN.flatten(), inv.flatten(), dxn_pre.flatten(), DXN.flatten(), c2])
    out = _repeat_bitwise(run).double()
    o = 0
    def take(n):
        nonlocal o
        o += n
        return out[o - n:o]
    mom, XN, inv = take(12 * d), take(6 * B * d).view(6, B, d), take(6 * B).view(6, B)
    dxn_pre, DXN, c2 = take(6 * B * d).view(6, B, d), take(6 * B * d).view(6, B, d), take(6 * d)
    X = X0.double().permute(1, 0, 2)                                   # [6][B][d]
    xc = X - X.mean(1, keepdim=True)
    ref_mom = torch.stack([torch.stack([(xc[i] ** k).sum(0) for k in (2, 3, 4, 5)]) for i in (3, 4, 5)])
    rel = lambda a, b: float((a - b).abs().max() / (b.abs().max() + 1e-30))
    assert rel(mom.view(3, 4, d), ref_mom) <= 1e-5
    assert rel(XN, xc / (xc.norm(dim=2, keepdim=True) + 1e-6)) <= 1e-5
    pa, pb = (0, 1, 2, 2, 2, 0), (3, 4, 5, 0, 1, 1)
    G = Gm.double()
    ref_dxn = torch.zeros(6, B, d, dtype=torch.float64, device=dev)
    for p in range(6):
        ref_dxn[pa[p]] += XN[pb[p]] @ G[p].t()
        ref_dxn[pb[p]] += XN[pa[p]] @ G[p]
    ref_dxn *= alpha
    assert rel(dxn_pre, ref_dxn) <= 1e-5
    ref_scaled = dxn_pre * inv[:, :, None]
    assert rel(DXN, ref_scaled) <= 1e-6
    assert rel(c2.view(6, d), ref_scaled.sum(1)) <= 1e-5


# ------------------------------------------------------------------ whole steps ---------------
def _state(tr):
    n = tr.n_active
    return torch.cat([tr.p_arena[:n], tr.g_arena[:n], tr.m[:n], tr.v[:n]]).clone()


def _trainer(cfg, seed=5, use_graph=False, **kw):
    from mmda_b200 import MISA
    from mmda_b200.trainer import FusedTrainer
    torch.manual_seed(seed)
    return FusedTrainer(MISA(cfg).cuda().train(), use_graph=use_graph, **kw)


def _steps(tr, batches, steps, start=0):
    """per step: the losses and the parameters, gradients and both optimizer moments"""
    hist = []
    for it in range(start, start + steps):
        b = batches[it % len(batches)]
        L = tr.step(b.sentences.cuda(), b.visual.cuda(), b.acoustic.cuda(), b.lengths, b.labels.cuda(),
                    *((b.bert_sent.cuda(), b.bert_sent_type.cuda(), b.bert_sent_mask.cuda())
                      if tr.use_bert else ()))
        hist.append((L[:6].clone(), _state(tr)))
    torch.cuda.synchronize()
    return hist


def _run(cfg, batches, steps, use_graph=False, seed=5):
    tr = _trainer(cfg, seed, use_graph)
    hist = _steps(tr, batches, steps)
    graphed = tr._graph is not None
    tr.close()
    return hist, graphed


def _identical(h1, h2):
    assert len(h1) == len(h2)
    for i, ((l1, s1), (l2, s2)) in enumerate(zip(h1, h2)):
        assert torch.equal(l1, l2), (i, (l1 - l2).abs().max())
        assert torch.equal(s1, s2), (i, (s1 - s2).abs().max())
        assert torch.isfinite(s1).all(), i


def _c2(**kw):
    from mmda_b200 import mosei_config
    return mosei_config(vocab_size=2000, use_confidNet=True, **kw)


def _batches(cfg, lengths="ragged", n=3, seq_len=50):
    from mmda_b200.synthetic import batch_for
    return [batch_for(cfg, seed=60 + i, lengths=lengths, seq_len=seq_len) for i in range(n)]


def test_c2_two_eager_runs_are_bit_identical(dev, det):
    cfg = _c2()
    bs = _batches(cfg)
    _identical(_run(cfg, bs, 10)[0], _run(cfg, bs, 10)[0])


def test_c2_ragged_graph_replay_equals_eager_and_itself(dev, det):
    """ragged lengths: a graph step runs over the packed rows rounded up to a row bucket (and its
    first warm-up steps over B*T rows); the fixed-order reductions make that padding invisible"""
    cfg = _c2()
    bs = _batches(cfg)
    graph, graphed = _run(cfg, bs, 10, use_graph=True)
    assert graphed
    _identical(graph, _run(cfg, bs, 10)[0])
    _identical(graph, _run(cfg, bs, 10, use_graph=True)[0])


def test_c2_checkpoint_resume_equals_uninterrupted_run(dev, det):
    """model + optimizer state after step 5 into a fresh (graph-mode) trainer: steps 6..10 are the
    uninterrupted run's, bit for bit"""
    cfg = _c2()
    bs = _batches(cfg, n=4)
    tr = _trainer(cfg, use_graph=True)
    _steps(tr, bs, 5)
    ckpt_model = {k: v.detach().clone() for k, v in tr.model.state_dict().items()}
    ckpt_optim = tr.optimizer_state_dict()
    ref = _steps(tr, bs, 5, start=5)
    tr.close()
    tr2 = _trainer(cfg, seed=99, use_graph=True)
    tr2.model.load_state_dict(ckpt_model)
    tr2.load_optimizer_state_dict(ckpt_optim)
    got = _steps(tr2, bs, 5, start=5)
    tr2.close()
    for (l1, s1), (l2, s2) in zip(got, ref):
        assert torch.equal(l1, l2)
        assert torch.equal(s1, s2), (s1 - s2).abs().max()


_SUBPROCESS = """
import sys, torch
sys.path.insert(0, {tests!r}); sys.path.insert(0, {root!r})
import test_gpu_deterministic as T
torch.use_deterministic_algorithms(True)
cfg = T._c2()
hist, _ = T._run(cfg, T._batches(cfg), 4, use_graph=True)
torch.save([(l.cpu(), s.cpu()) for l, s in hist], {out!r})
"""


def test_c2_subprocess_run_equals_in_process_run(dev, det, tmp_path):
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    out = str(tmp_path / "run.pt")
    code = _SUBPROCESS.format(tests=here, root=os.path.dirname(here), out=out)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    cfg = _c2()
    mine, _ = _run(cfg, _batches(cfg), 4, use_graph=True)
    theirs = torch.load(out)
    _identical([(l.cpu(), s.cpu()) for l, s in mine], theirs)


def test_c1_parity_with_the_fp64_oracle_holds_with_the_flag_on(dev, det):
    """level 1 and level 2 against the fp64 oracle at C1 within the 1e-5 bound, deterministic"""
    from test_gpu_parity import _full
    _full("mosi", "c1_mosi_b64", "ragged", dev)


def test_graph_cache_keys_the_two_modes_apart(dev):
    cfg = _c2(batch_size=48)
    b = _batches(cfg, lengths="full", n=1, seq_len=12)[0]
    tr = _trainer(cfg, seed=1, use_graph=True)
    args = (b.sentences.cuda(), b.visual.cuda(), b.acoustic.cuda(), b.lengths, b.labels.cuda())
    try:
        for flag in (False, True, False):
            torch.use_deterministic_algorithms(flag)
            for _ in range(4):
                tr.step(*args)
        keys = {k[-1] for k in tr._graphs}
        assert keys == {False, True}, list(tr._graphs)
    finally:
        torch.use_deterministic_algorithms(False)
        tr.close()


@pytest.mark.parametrize("variant", [{"rnncell": "gru"}, {"use_cmd_sim": False},
                                     {"activation": "rrelu"}, {"optimizer": "RMSprop"}],
                         ids=["gru", "adversarial", "rrelu", "rmsprop"])
def test_variants_two_runs_are_bit_identical(dev, det, variant):
    cfg = _c2(batch_size=64, **variant)
    bs = _batches(cfg, seq_len=20)
    _identical(_run(cfg, bs, 5, use_graph=True)[0], _run(cfg, bs, 5, use_graph=True)[0])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("seq_len", [50, 128], ids=["S52", "S130"])
def test_bert_two_runs_are_bit_identical(dev, det, precision, seq_len):
    """the BERT text encoder (use_bert=True): S = seq_len + 2 positions, fp32 and bf16 operands"""
    from mmda_b200 import mosei_config
    cfg = mosei_config(vocab_size=200, batch_size=8, use_bert=True, use_confidNet=True,
                       precision=precision)
    bs = _batches(cfg, n=2, seq_len=seq_len)
    assert bs[0].bert_sent.shape[1] == seq_len + 2
    _identical(_run(cfg, bs, 3)[0], _run(cfg, bs, 3)[0])


def test_level1_backward_and_evaluate_repeat(dev, det):
    from mmda_b200 import MISA
    from mmda_b200.evaluate import evaluate
    cfg = _c2(batch_size=64)
    b = _batches(cfg, n=1, seq_len=20)[0]
    grads = []
    for _ in range(2):      # a fresh model each time: the dropout masks follow the forward count
        torch.manual_seed(2)
        model = MISA(cfg).cuda().train()
        out = model(b.sentences.cuda(), b.visual.cuda(), b.acoustic.cuda(), b.lengths)
        loss = sum(v.float().pow(2).mean() for v in out if torch.is_tensor(v) and v.requires_grad)
        loss.backward()
        grads.append([p.grad.clone() for p in model.parameters() if p.grad is not None])
    assert len(grads[0]) > 10
    for a, c in zip(*grads):
        assert torch.equal(a, c)
    m1 = evaluate(model, [b])
    m2 = evaluate(model, [b])
    assert m1 == m2


def _dp_worker(rank, world, port, q):
    import os
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.dirname(here))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.use_deterministic_algorithms(True)
    from mmda_b200 import MISA
    from mmda_b200.trainer import FusedTrainer
    cfg = _c2(batch_size=64)
    bs = [b.slice(rank * 32, (rank + 1) * 32) for b in _batches(cfg, seq_len=20)]
    runs = []
    for _ in range(2):
        torch.manual_seed(4)
        tr = FusedTrainer(MISA(cfg).to(dev).train(), process_group=dist.group.WORLD)
        hist = []
        for it in range(5):
            b = bs[it % len(bs)]
            L = tr.step(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths,
                        b.labels.to(dev))
            hist.append(torch.cat([L[:6].clone(), _state(tr)]).cpu())
        tr.close()
        runs.append(torch.stack(hist))
    q.put((rank, bool(torch.equal(runs[0], runs[1]))))
    dist.destroy_process_group()


def test_two_gpu_data_parallel_runs_are_bit_identical():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=600) for _ in range(2))
    [p.join(60) for p in procs]
    assert all(same for _, same in res), res
