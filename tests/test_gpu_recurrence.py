"""SIMT cluster recurrence (csrc/lstm.cu: lstm_fwd_kernel / lstm_bwd_kernel, LSTM and GRU cells)
through the C ABI against the fp64 restatement in tools/dev_lstm_tc.py (pinned to nn.LSTM / nn.GRU
by tests/test_recurrence_reference.py): hidden / cell states, saved gate activations, final states
in original batch order and the BPTT output d(gates), 1e-5 scale-relative, for a case list that
reaches every launch plan class (cluster size C, batch tile BT, contraction split KS), and the
support kernels of the recurrence (weight packing, GRU expand / fold, h shift) bit-exact."""
import ctypes
import json
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
TOL = 1e-5
MMDA_ERR_UNSUPPORTED = -3
ALL_CLASSES = {(1, 8, 4), (1, 32, 4), (2, 8, 4), (4, 32, 16), (8, 32, 16), (8, 40, 16)}
BT40_CANDIDATES = (256, 300, 512)     # the 40-row tile depends on the device's cluster occupancy
NAN = float("nan")

# id, H, B (None: the batch that selects BT = 40 at H = 300), T, ragged, lengths, pad, rnn2 layout,
# plan class the case is there to reach
CASES = [
    ("b1_t1", 74, 1, 1, 0, None, 0, False, (1, 8, 4)),
    ("b9_all_len1", 74, 9, 1, 0, None, 0, True, (1, 8, 4)),            # B = BT + 1, Tmax = 1
    ("b7_ragged", 74, 7, 9, 1, None, 0, False, (1, 8, 4)),             # B = BT - 1
    ("b70_one_long", 35, 70, 20, 0, "one_long", 0, True, (1, 32, 4)),  # later tiles: Lmax = 1
    ("b65_equal", 40, 65, 7, 0, None, 0, False, (1, 32, 4)),           # B = 2 BT + 1
    ("h128", 128, 9, 6, 1, None, 0, False, (2, 8, 4)),
    ("h117_padded", 117, 17, 5, 1, None, 3, True, (2, 8, 4)),
    ("h160_b33", 160, 33, 6, 1, None, 0, False, (4, 32, 16)),          # B = BT + 1
    ("h129_b31", 129, 31, 5, 1, None, 0, True, (4, 32, 16)),           # B = BT - 1
    ("h300_b64", 300, 64, 12, 1, None, 0, False, (8, 32, 16)),
    ("h161_b300", 161, 300, 5, 1, None, 0, False, (8, 32, 16)),        # 2 x 10 clusters > one wave
    ("h304_b33", 304, 33, 4, 1, None, 0, True, (8, 32, 16)),           # widest SIMT plan
    ("h300_bt40", 300, None, 20, 1, None, 0, False, (8, 40, 16)),
    ("h300_bt40_one_long", 300, None, 8, 0, "one_long", 0, True, (8, 40, 16)),
]


def lib():
    from mmda_b200._lib import LIB
    return LIB


def plan(B, H):
    """-> ((C, BT, KS), n_tiles) of mmda_lstm_plan; KS = 16 iff H > 128."""
    out = (ctypes.c_int * 6)()
    lib().call("mmda_lstm_plan", B, H, out)
    return (out[0], out[2], 16 if H > 128 else 4), out[3]


def bt40_batch():
    for B in BT40_CANDIDATES:
        if plan(B, 300)[0] == (8, 40, 16):
            return B
    pytest.fail(f"no batch in {BT40_CANDIDATES} selects the 40-row tile at H=300 on this device "
                f"(plans: {[plan(B, 300) for B in BT40_CANDIDATES]}); the (8, 40, 16) kernels stay untested")


def case_batch(B):
    return bt40_batch() if B is None else B


def make(case, cell, seed=0, **kw):
    import dev_lstm_tc as D
    name, H, B, T, ragged, pattern, pad, rnn2, _ = case
    B = case_batch(B)
    lens = [T] + [1] * (B - 1) if pattern == "one_long" else None
    return D.make_case(B, H, T, ragged, torch.device("cuda:0"), seed=seed or B + H, cell=cell,
                       lens=lens, pad=pad, utt_layout=(4 * H, H, 3 * H) if rnn2 else None, **kw)


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def owned_cols(c):
    ld, uo_f, uo_r = c["utt_layout"]
    m = torch.zeros(ld, dtype=torch.bool, device=c["gates"].device)
    m[uo_f:uo_f + c["H"]] = True
    m[uo_r:uo_r + c["H"]] = True
    return m


@pytest.fixture(scope="module")
def report():
    rows = []
    yield rows
    out = os.path.join(ROOT, "test_reports")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "recurrence_parity.txt"), "w") as f:
        f.write("case cell B H Tmax (C,BT,KS) n_tiles | kernel vs fp64 | fp32 torch vs fp64\n")
        for r in rows:
            f.write(f"{r['case']} {r['cell']} B={r['B']} H={r['H']} Tmax={r['Tmax']} "
                    f"{tuple(r['plan'])} tiles={r['n_tiles']} | "
                    + " ".join(f"{k}={v:.2e}" for k, v in r["err"].items()) + " | "
                    + " ".join(f"{k}={v:.2e}" for k, v in r["fp32_torch"].items()) + "\n")
        seen = {}
        for r in rows:
            seen.setdefault(r["cell"], set()).add(tuple(r["plan"]))
        f.write("classes reached: " + json.dumps({k: sorted(v) for k, v in seen.items()}) + "\n")


def check(c, name, report):
    """Forward + backward through the C ABI against fp64; returns the kernel outputs."""
    import dev_lstm_tc as D
    lstm = c["cell"] == "lstm"
    klass, n_tiles = plan(c["B"], c["H"])
    y64, s64, a64, u64 = D.ref64(c)
    dG64 = D.ref64_bwd(c, a64, s64) if lstm else D.ref64_grad(c)
    o = D.run(c, "simt", fill=NAN)
    # the backward may only write the scratch mmda_lstm_scratch_bytes reported
    assert o["scratch_overrun"] == 0, \
        f"backward wrote {o['scratch_overrun']} floats past the mmda_lstm_scratch_bytes buffer"
    own = owned_cols(c)
    assert torch.isnan(o["utt"][:, ~own]).all(), "utt columns outside the final-state slices were written"
    err = {"y": D.rel(o["y"], y64), "act": D.rel(o["act"], a64),
           "utt": D.rel(o["utt"][:, own], u64[:, own]), "dG": D.rel(o["dG"], dG64)}
    if lstm:
        err["c"] = D.rel(o["c"], s64)
    # what an fp32 torch run of the same recurrence gets: the yardstick for the bound
    y32, s32, a32, _ = D.ref64(c, torch.float32)
    dG32 = D.ref64_bwd(c, a32, s32, torch.float32) if lstm else D.ref64_grad(c, torch.float32)
    report.append(dict(case=name, cell=c["cell"], B=c["B"], H=c["H"], Tmax=c["Tmax"], plan=klass,
                       n_tiles=n_tiles, err=err,
                       fp32_torch={"y": D.rel(y32, y64), "dG": D.rel(dG32, dG64)}))
    bad = {k: v for k, v in err.items() if not v <= TOL}     # NaN (an unwritten element) fails
    assert not bad, (name, c["cell"], klass, bad)
    return o


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_simt_recurrence_vs_fp64(cell, case, report):
    import dev_lstm_tc as D
    c = make(case, cell)
    assert plan(c["B"], c["H"])[0] == case[-1], "the case no longer reaches the plan class it covers"
    o = check(c, case[0], report)
    # same inputs, same launch twice: the accumulation order is fixed, so the bits are too
    o2 = D.run(c, "simt", fill=NAN)
    for k in ("y", "c", "act", "utt", "dG"):
        if o[k] is not None:
            assert same_bits(o[k], o2[k]), f"{k} differs between two identical launches"
    # save_for_backward = 0 with c = NULL: the same y and final states, gates left as they came
    o0 = D.run(c, "simt", save=0, fill=NAN)
    assert same_bits(o0["y"], o["y"]) and same_bits(o0["utt"], o["utt"])
    assert same_bits(o0["act"], c["gates"]), "the forward wrote gates without save_for_backward"


def test_case_list_reaches_every_plan_class():
    reached = {plan(case_batch(B), H)[0] for _, H, B, *_ in CASES}
    assert reached == ALL_CLASSES, f"missing {ALL_CLASSES - reached}, unexpected {reached - ALL_CLASSES}"


@pytest.mark.parametrize("H,B,T", [(74, 9, 6), (128, 9, 5), (160, 33, 4), (300, 64, 5)])
@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_padded_tmax_gives_the_same_bits(cell, H, B, T):
    """Tmax past the longest length (offsets extended, batch size 0 there) changes nothing."""
    import dev_lstm_tc as D
    case = ("pad", H, B, T, 1, None, 0, False, None)
    a = D.run(make(case, cell, seed=7), "simt")
    b = D.run(make(case[:6] + (6,) + case[7:], cell, seed=7), "simt")
    assert b["scratch_overrun"] == 0
    for k in ("y", "c", "act", "utt", "dG"):
        if a[k] is not None:
            assert same_bits(a[k], b[k]), f"{k} depends on the padding of Tmax"


@pytest.mark.parametrize("H,B,T", [(74, 9, 6), (160, 33, 5), (300, 40, 6)])
@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_dy_null_equals_dy_zero(cell, H, B, T, report):
    """rnn2 passes dy = NULL (its sequence output is discarded): the same bits as dy = 0, and the
    gradient of the final states alone matches fp64."""
    import dev_lstm_tc as D
    c = make(("dy_null", H, B, T, 1, None, 0, True, None), cell, seed=9)
    c["dy"] = None
    o = check(c, f"dy_null_h{H}", report)
    c["dy"] = torch.zeros(c["N"], 2 * H, device=c["gates"].device)
    assert same_bits(D.run(c, "simt", fill=NAN)["dG"], o["dG"])


@pytest.mark.parametrize("B", [8, 64])
@pytest.mark.parametrize("H", [115, 116])
@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_backward_scratch_holds_for_long_sequences(cell, H, B, report):
    """mmda_lstm_scratch_bytes(B, H) sizes the backward scratch for every Tmax.  At H = 115 / 116
    the backward once staged offsets[Tmax + 1] in shared memory, so Tmax = 600 moved it to a
    2-CTA cluster whose scratch is twice the reported size; run() puts a sentinel after the
    reported size and fails on any word written there."""
    c = make((f"scratch_h{H}", H, B, 600, 1, None, 0, False, None), cell)
    check(c, f"scratch_h{H}_b{B}_t600", report)


@pytest.mark.parametrize("H", [305, 320])
def test_gru_sizes_past_the_simt_plan_are_unsupported(H):
    """305 <= H <= 320: no shared-memory resident W_hh plan (the tensor-core path has no GRU
    cell); the entries return MMDA_ERR_UNSUPPORTED before any launch."""
    L = lib()
    assert L.raw("mmda_lstm_scratch_bytes")(64, H) == -1
    assert L.raw("mmda_lstm_plan")(64, H, (ctypes.c_int * 6)()) == MMDA_ERR_UNSUPPORTED
    st = torch.cuda.current_stream().cuda_stream
    x = torch.zeros(1, device="cuda:0")      # never read: the plan is refused before any launch
    assert L.raw("mmda_gru_forward")(None, None, None, None, None, None, None, None, 4 * H, 0,
                                     2 * H, 64, H, 10, 1, st) == MMDA_ERR_UNSUPPORTED
    assert L.raw("mmda_gru_backward")(None, None, None, P(x), None, None, 4 * H, 0, 2 * H, None,
                                      None, None, P(x), 64, H, 10, st) == MMDA_ERR_UNSUPPORTED


# ---------------------------------------------------------------------------------------------
# support kernels, bit-exact against torch indexing
# ---------------------------------------------------------------------------------------------
def P(t):
    return None if t is None else t.data_ptr()


def spread(*shape, g):
    """fp32 values over many binades (rounding of the tf32 conversion is exercised)."""
    return torch.randn(*shape, generator=g) * torch.pow(10.0, torch.randint(-6, 6, shape, generator=g).float())


def test_lstm_pack_weights_tf32_split():
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(22)
    H, I, ld = 37, 23, 29
    w = [spread(4 * H, I, g=g) for _ in range(2)]
    b = [spread(4 * H, g=g) for _ in range(4)]       # b_ih_f, b_hh_f, b_ih_r, b_hh_r
    wd, bd = [x.to(dev) for x in w], [x.to(dev) for x in b]
    sentinel = -3.0
    out_a = torch.full((8 * H, ld), sentinel, device=dev)
    out_b = torch.full((8 * H, ld), sentinel, device=dev)
    bias = torch.full((8 * H,), sentinel, device=dev)
    lib().call("mmda_lstm_pack_weights", P(wd[0]), P(wd[1]), P(bd[0]), P(bd[1]), P(bd[2]), P(bd[3]),
               H, I, P(out_a), P(out_b), ld, P(bias), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    # row dir*4H + u*4 + g of the copy = row g*H + u of weight_ih_l0{,_reverse}
    W = torch.stack(w).view(2, 4, H, I).transpose(1, 2).reshape(8 * H, I)
    bias_ref = (torch.stack([b[0] + b[1], b[2] + b[3]])).view(2, 4, H).transpose(1, 2).reshape(-1)
    assert same_bits(bias.cpu(), bias_ref)
    got = out_a.cpu()
    assert torch.all(got[:, I:] == sentinel), "pitch columns past I were written"
    got = got[:, :I]
    lo = out_b.cpu()
    assert torch.all(lo[:, I:] == sentinel)
    lo = lo[:, :I]
    bits = got.view(torch.int32)
    assert torch.all(bits & 0x1FFF == 0), "hi is not tf32-representable"
    rna = ((W.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)   # round to nearest, ties away
    assert same_bits(got, rna)
    assert same_bits(got + lo, W), "hi + lo != w"


def test_gru_expand_and_fold():
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(31)
    H, I = 19, 13
    st = torch.cuda.current_stream().cuda_stream
    w_ih, w_hh, b_ih, b_hh = (torch.randn(*s, generator=g).to(dev)
                              for s in ((3 * H, I), (3 * H, H), (3 * H,), (3 * H,)))
    w4_ih, w4_hh, b4_ih, b4_hh = (torch.full(s, NAN, device=dev)
                                  for s in ((4 * H, I), (4 * H, H), (4 * H,), (4 * H,)))
    lib().call("mmda_gru_expand_weights", P(w_ih), P(w_hh), P(b_ih), P(b_hh), H, I, P(w4_ih),
               P(w4_hh), P(b4_ih), P(b4_hh), st)
    torch.cuda.synchronize()
    zI, zH, z = torch.zeros(H, I, device=dev), torch.zeros(H, H, device=dev), torch.zeros(H, device=dev)
    # x side (r, z, n, 0); h side (r, z, 0, n)
    assert same_bits(w4_ih, torch.cat([w_ih, zI]))
    assert same_bits(w4_hh, torch.cat([w_hh[:2 * H], zH, w_hh[2 * H:]]))
    assert same_bits(b4_ih, torch.cat([b_ih, z]))
    assert same_bits(b4_hh, torch.cat([b_hh[:2 * H], z, b_hh[2 * H:]]))

    dw4 = [torch.randn(*s, generator=g).to(dev) for s in ((4 * H, I), (4 * H, H), (4 * H,), (4 * H,))]
    real = [torch.randn(*s, generator=g).to(dev) for s in ((3 * H, I), (3 * H, H), (3 * H,), (3 * H,))]
    acc = [r.clone() for r in real]          # the fold accumulates (+=) onto the real gradients
    lib().call("mmda_gru_fold_grads", *[P(x) for x in dw4], H, I, *[P(x) for x in acc], st)
    torch.cuda.synchronize()
    h_side = lambda t: torch.cat([t[:2 * H], t[3 * H:]])    # slots r, z, n(h) = 0, 1, 3
    assert same_bits(acc[0], real[0] + dw4[0][:3 * H])
    assert same_bits(acc[1], real[1] + h_side(dw4[1]))
    assert same_bits(acc[2], real[2] + dw4[2][:3 * H])
    assert same_bits(acc[3], real[3] + h_side(dw4[3]))


def test_lstm_shift_h_keeps_the_pitch_columns():
    import dev_lstm_tc as D
    dev = torch.device("cuda:0")
    H, Hp = 21, 24
    c = D.make_case(13, H, 7, 1, dev, seed=41)
    N, ls, off = c["N"], c["ls_cpu"], c["off_cpu"]
    bs = off[1:] - off[:-1]
    row_t = torch.repeat_interleave(torch.arange(c["Tmax"]), bs)
    row_j = torch.cat([torch.arange(int(n)) for n in bs])
    y = torch.randn(N, 2 * H, generator=torch.Generator().manual_seed(42))
    sentinel = -5.0
    hp = torch.full((N, 2, Hp), sentinel, device=dev)
    yd, td, jd = y.to(dev), row_t.int().to(dev), row_j.int().to(dev)   # alive until the kernel ran
    lib().call("mmda_lstm_shift_h", P(yd), P(hp), P(td), P(jd), P(c["lens"]), P(c["off"]), N, H, Hp,
               torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ref = torch.full((N, 2, Hp), sentinel)
    ref[:, :, :H] = 0
    for r, (t, j) in enumerate(zip(row_t.tolist(), row_j.tolist())):
        if t >= 1:                       # forward direction: y at t - 1
            ref[r, 0, :H] = y[off[t - 1] + j, :H]
        if t + 1 < ls[j]:                # reverse direction: y at t + 1
            ref[r, 1, :H] = y[off[t + 1] + j, H:]
    assert same_bits(hp.cpu(), ref)
