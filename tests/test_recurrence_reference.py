"""The fp64 recurrence reference of tools/dev_lstm_tc.py (the yardstick of the recurrence kernel
tests) pinned to torch on the CPU: ref64 against nn.LSTM / nn.GRU on pack_padded_sequence
inputs, its saved-state backward against autograd, and the d(gates) slots against torch's
parameter and input gradients."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
TOL = 1e-12


def torch_case(cell, lens, H, I, pad, layout, seed):
    """nn.LSTM / nn.GRU (bidirectional, fp64) on packed inputs, and the same launch in the packed
    gate layout the recurrence kernels take: G = x W_ih^T + b in the gate-interleaved order."""
    import dev_lstm_tc as D
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    rnn = (torch.nn.LSTM if cell == "lstm" else torch.nn.GRU)(I, H, bidirectional=True,
                                                             dtype=torch.float64)
    lens_t = torch.tensor(lens)
    B, T = len(lens), max(lens)
    x = torch.randn(B, T, I, generator=g, dtype=torch.float64, requires_grad=True)
    packed = torch.nn.utils.rnn.pack_padded_sequence(x, lens_t, batch_first=True,
                                                     enforce_sorted=False)
    si = packed.sorted_indices
    ls = lens_t[si]
    Tmax = T + pad
    off = torch.zeros(Tmax + 1, dtype=torch.int64)
    off[1:T + 1] = torch.cumsum(packed.batch_sizes, 0)
    off[T + 1:] = off[T]
    X = packed.data.detach()
    gates, whh = [], []
    for sfx in ("", "_reverse"):
        w_ih, w_hh = getattr(rnn, "weight_ih_l0" + sfx), getattr(rnn, "weight_hh_l0" + sfx)
        b_ih, b_hh = getattr(rnn, "bias_ih_l0" + sfx), getattr(rnn, "bias_hh_l0" + sfx)
        with torch.no_grad():
            if cell == "lstm":
                pre = X @ w_ih.T + b_ih + b_hh                                   # [N][4H] (g, u)
                w4 = w_hh.clone()
            else:   # 4-slot layout: x side (r, z, n, 0) + biases (b_ir+b_hr, b_iz+b_hz, b_in, b_hn)
                xs = X @ w_ih.T + b_ih
                xs[:, :2 * H] += b_hh[:2 * H]
                pre = torch.cat([xs, b_hh[2 * H:].expand(len(X), H)], 1)
                w4 = torch.cat([w_hh[:2 * H], torch.zeros(H, H, dtype=torch.float64), w_hh[2 * H:]])
        gates.append(pre.view(-1, 4, H).transpose(1, 2))                        # [N][H][4]
        whh.append(w4)
    N = len(X)
    layout = layout or (4 * H, 0, 2 * H)
    dy = torch.randn(N, 2 * H, generator=g, dtype=torch.float64)
    dutt = torch.randn(B, layout[0], generator=g, dtype=torch.float64)
    c = dict(B=B, H=H, Tmax=Tmax, N=N, lens=ls, sidx=si, off=off,
             gates=torch.stack(gates, 1).reshape(N, 8 * H).contiguous(), whh=whh, dy=dy,
             dutt=dutt, ls_cpu=ls, si_cpu=si, off_cpu=off, cell=cell, utt_layout=layout)
    return D, rnn, x, packed, c


CASES = [([5, 3, 5, 1, 2], 0, None), ([1], 0, None), ([6, 1, 1, 1, 1], 2, "rnn2"),
         ([4, 4, 4], 0, None), ([1, 1, 1], 3, None)]


@pytest.mark.parametrize("lens,pad,layout", CASES)
@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_ref64_matches_torch_rnn(cell, lens, pad, layout):
    H, I = 5, 3
    D, rnn, x, packed, c = torch_case(cell, lens, H, I, pad,
                                      (4 * H, H, 3 * H) if layout == "rnn2" else None, 11)
    out, hn = rnn(packed)
    hN = hn[0] if cell == "lstm" else hn
    y, cs, act, utt = D.ref64(c)
    assert D.rel(y, out.data) <= TOL
    ld, uo_f, uo_r = c["utt_layout"]
    assert D.rel(utt[:, uo_f:uo_f + H], hN[0]) <= TOL and D.rel(utt[:, uo_r:uo_r + H], hN[1]) <= TOL
    owned = torch.zeros(ld, dtype=torch.bool)
    owned[uo_f:uo_f + H] = owned[uo_r:uo_r + H] = True
    assert torch.all(utt[:, ~owned] == 0)
    ls, off, si = c["ls_cpu"], c["off_cpu"], c["si_cpu"]
    j = torch.arange(len(lens))
    rows_t = torch.repeat_interleave(torch.arange(max(lens)), packed.batch_sizes)
    rows_j = torch.cat([torch.arange(int(b)) for b in packed.batch_sizes])
    Y = y.view(-1, 2, H)
    if cell == "lstm":   # final cell states: fwd at t = L-1, bwd at t = 0; h = o tanh(c)
        cN = hn[1]
        assert D.rel(cs[off[ls - 1] + j, :H], cN[0][si]) <= TOL
        assert D.rel(cs[off[0] + j, H:], cN[1][si]) <= TOL
        o = act.view(-1, 2, H, 4)[..., 3]
        assert D.rel(o * torch.tanh(cs.view(-1, 2, H)), Y) <= TOL
    else:                # saved (r, z, n, W_hn h + b_hn) reproduce h' = (1 - z) n + z h
        z, n = act.view(-1, 2, H, 4)[..., 1], act.view(-1, 2, H, 4)[..., 2]
        hp = torch.zeros_like(Y)
        for row, (t, jj) in enumerate(zip(rows_t.tolist(), rows_j.tolist())):
            if t >= 1:
                hp[row, 0] = Y[off[t - 1] + jj, 0]
            if t + 1 < ls[jj]:
                hp[row, 1] = Y[off[t + 1] + jj, 1]
        assert D.rel((1 - z) * n + z * hp, Y) <= TOL
    # the d(gates) slots, mapped onto the parameters, are torch's gradients
    dy, dutt = c["dy"], c["dutt"]
    loss = (out.data * dy).sum() + (hN[0] * dutt[:, uo_f:uo_f + H]).sum() + \
        (hN[1] * dutt[:, uo_r:uo_r + H]).sum()
    loss.backward()
    dG = D.ref64_grad(c).view(-1, 2, H, 4)
    dX = torch.zeros_like(packed.data)
    for d, sfx in enumerate(("", "_reverse")):
        w_ih = getattr(rnn, "weight_ih_l0" + sfx).detach()
        db_ih, db_hh = getattr(rnn, "bias_ih_l0" + sfx).grad, getattr(rnn, "bias_hh_l0" + sfx).grad
        S = dG[:, d].sum(0).T                                   # [4][H] summed over tokens
        if cell == "lstm":
            dX += dG[:, d].transpose(1, 2).reshape(-1, 4 * H) @ w_ih
            assert D.rel(S.reshape(-1), db_ih) <= TOL and D.rel(S.reshape(-1), db_hh) <= TOL
        else:
            dX += dG[:, d, :, :3].transpose(1, 2).reshape(-1, 3 * H) @ w_ih
            assert D.rel(S[:3].reshape(-1), db_ih) <= TOL
            assert D.rel(S[[0, 1, 3]].reshape(-1), db_hh) <= TOL
    assert D.rel(dX, x.grad[si[rows_j], rows_t]) <= TOL


@pytest.mark.parametrize("lens,pad", [([7, 3, 7, 1, 2, 5], 0), ([1], 0), ([9, 1, 1, 1], 2)])
@pytest.mark.parametrize("with_dy", [True, False])
def test_ref64_bwd_matches_autograd(lens, pad, with_dy):
    import dev_lstm_tc as D
    c = D.make_case(0, 6, 0, 0, torch.device("cpu"), seed=3, lens=lens, pad=pad,
                    utt_layout=(24, 6, 18))
    if not with_dy:
        c["dy"] = None
    y, cs, act, utt = D.ref64(c)
    assert D.rel(D.ref64_bwd(c, act, cs), D.ref64_grad(c)) <= TOL


def test_padded_tmax_changes_nothing():
    """Steps past the longest length have batch size 0: the reference gives the same values."""
    import dev_lstm_tc as D
    for cell in ("lstm", "gru"):
        a = D.make_case(0, 4, 0, 0, torch.device("cpu"), seed=5, cell=cell, lens=[3, 1, 2])
        b = D.make_case(0, 4, 0, 0, torch.device("cpu"), seed=5, cell=cell, lens=[3, 1, 2], pad=4)
        assert b["Tmax"] == a["Tmax"] + 4 and torch.all(b["off_cpu"][a["Tmax"]:] == a["N"])
        for u, v in zip(D.ref64(a), D.ref64(b)):
            assert torch.equal(u, v)
        assert torch.equal(D.ref64_grad(a), D.ref64_grad(b))
