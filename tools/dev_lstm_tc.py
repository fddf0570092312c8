"""GPU dev driver for the tensor-core recurrence (csrc/lstm_tc.cu): parity against the SIMT
recurrence (csrc/lstm.cu) and an fp64 torch restatement on the same packed inputs, then timing.

    python tools/dev_lstm_tc.py [B H T ragged]
"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mmda_b200._lib import LIB  # noqa: E402


def P(t):
    return None if t is None else t.data_ptr()


def make_case(B, H, T, ragged, dev, seed=0, cell="lstm", lens=None, pad=0, utt_layout=None):
    """Random packed inputs of one bidirectional recurrence launch.

    lens: explicit per-sample lengths (then B and T are taken from it); pad: extra steps of Tmax
    past the longest length (offsets repeat N there, batch size 0); utt_layout: (utt_ld, off_f,
    off_r), default (4H, 0, 2H); rnn2 writes (4H, H, 3H).  For cell="gru" W_hh is in the 4-slot
    layout [W_hr; W_hz; 0; W_hn] that mmda_gru_expand_weights produces."""
    g = torch.Generator().manual_seed(seed)
    if lens is not None:
        lens = torch.as_tensor(lens, dtype=torch.int64)
        B = len(lens)
    elif ragged:
        lens = torch.randint(1, T + 1, (B,), generator=g)
        lens[0] = T
    else:
        lens = torch.full((B,), T)
    ls, si = torch.sort(lens, descending=True)
    Tmax = int(ls[0]) + pad
    bs = torch.tensor([(ls > t).sum() for t in range(Tmax)])
    off = torch.zeros(Tmax + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(bs, 0)
    N = int(off[-1])
    layout = utt_layout or (4 * H, 0, 2 * H)
    gates = torch.randn(N, 8 * H, generator=g) * 0.7
    whh = [torch.nn.init.orthogonal_(torch.empty(4 * H, H), generator=g) for _ in range(2)]
    if cell == "gru":
        for w in whh:
            w[2 * H:3 * H] = 0
    dy = torch.randn(N, 2 * H, generator=g) * 0.1
    dutt = torch.randn(B, layout[0], generator=g) * 0.1
    d = dict(B=B, H=H, Tmax=Tmax, N=N, lens=ls.int().to(dev), sidx=si.int().to(dev),
             off=off.int().to(dev), gates=gates.to(dev), whh=[w.to(dev) for w in whh],
             dy=dy.to(dev), dutt=dutt.to(dev), ls_cpu=ls, si_cpu=si, off_cpu=off, cell=cell,
             utt_layout=layout)
    return d


def ref64(c, dtype=torch.float64, gates=None):
    """Restatement of the recurrence on the packed layout (oracle/explicit.py::lstm_direction
    semantics for the LSTM; nn.GRU's cell on the 4-slot layout for the GRU), in `dtype`.

    -> y [N][2H], the state the backward takes (LSTM: c; GRU: y) [N][2H], the saved activations
    [N][8H] (LSTM: i,f,g,o; GRU: r, z, n, W_hn h + b_hn) and utt (B, utt_ld), zero outside the
    final-state columns.  `gates` replaces c["gates"] (autograd)."""
    B, H, Tmax = c["B"], c["H"], c["Tmax"]
    gru = c["cell"] == "gru"
    G = (c["gates"] if gates is None else gates).to(dtype).view(-1, 2, H, 4)
    dev = G.device
    ls, off = c["ls_cpu"], c["off_cpu"]
    ld, uo_f, uo_r = c["utt_layout"]
    y = torch.zeros(c["N"], 2, H, dtype=dtype, device=dev)
    cc = torch.zeros_like(y)
    act = torch.zeros(c["N"], 2, H, 4, dtype=dtype, device=dev)
    for d in range(2):
        W = c["whh"][d].to(dtype).view(4, H, H)        # [g][u][k]
        h = torch.zeros(B, H, dtype=dtype, device=dev)
        cs = torch.zeros_like(h)
        ts = range(Tmax) if d == 0 else range(Tmax - 1, -1, -1)
        for t in ts:
            n = int((ls > t).sum())
            if n == 0:
                continue
            rows = slice(int(off[t]), int(off[t]) + n)
            pre = G[rows, d] + torch.einsum("guk,bk->bug", W, h[:n])
            if gru:
                r, z, hn3 = torch.sigmoid(pre[..., 0]), torch.sigmoid(pre[..., 1]), pre[..., 3]
                nn_ = torch.tanh(pre[..., 2] + r * hn3)
                hn = (1 - z) * nn_ + z * h[:n]
                a = torch.stack([r, z, nn_, hn3], -1)
            else:
                i, f, g_, o = (torch.sigmoid(pre[..., 0]), torch.sigmoid(pre[..., 1]),
                               torch.tanh(pre[..., 2]), torch.sigmoid(pre[..., 3]))
                cn = f * cs[:n] + i * g_
                hn = o * torch.tanh(cn)
                cs = cs.clone()
                cs[:n] = cn
                cc[rows, d] = cn
                a = torch.stack([i, f, g_, o], -1)
            h = h.clone()
            h[:n] = hn
            y[rows, d] = hn
            act[rows, d] = a
    # final states in original order: fwd = h at t = L-1, bwd = h at t = 0
    j = torch.arange(B)
    si = c["si_cpu"].to(dev)
    utt = torch.zeros(B, ld, dtype=dtype, device=dev)
    utt[si, uo_f:uo_f + H] = y[(off[ls - 1] + j).to(dev), 0]
    utt[si, uo_r:uo_r + H] = y[(off[0] + j).to(dev), 1]
    y = y.view(-1, 2 * H)
    return y, (y if gru else cc.view(-1, 2 * H)), act.view(-1, 8 * H), utt


def ref64_grad(c, dtype=torch.float64):
    """BPTT output d(gates) [N][8H] by autograd through ref64: for the GRU slot 3 is d(W_hn h +
    b_hn) = d n_pre * r, the other slots are the pre-activation gradients."""
    G = c["gates"].to(dtype).detach().requires_grad_()
    y, _, _, utt = ref64(c, dtype, gates=G)
    loss = (utt * c["dutt"].to(dtype)).sum()
    if c["dy"] is not None:
        loss = loss + (y * c["dy"].to(dtype)).sum()
    (dG,) = torch.autograd.grad(loss, G)
    return dG


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


SENTINEL = -7.0e37      # fills the guard half of the backward scratch


def run(c, which, save=1, fill=0.0):
    """One forward + backward launch pair through the C ABI.  y / c / utt start filled with
    `fill`; save=0 runs the forward alone with c = NULL.  The SIMT backward gets twice the scratch
    mmda_lstm_scratch_bytes reports, the second half filled with SENTINEL; out["scratch_overrun"]
    counts the guard words it changed."""
    B, H, Tmax, N = c["B"], c["H"], c["Tmax"], c["N"]
    ld, uo_f, uo_r = c["utt_layout"]
    gru = c["cell"] == "gru"
    assert not (gru and which == "tc"), "the tensor-core recurrence has no GRU cell"
    dev = c["gates"].device
    st = torch.cuda.current_stream().cuda_stream
    G = c["gates"].clone()
    y = torch.full((N, 2 * H), fill, device=dev)
    cc = torch.full((N, 2 * H), fill, device=dev) if save and not gru else None
    utt = torch.full((B, ld), fill, device=dev)
    w0, w1 = P(c["whh"][0]), P(c["whh"][1])
    lens, sidx, off = P(c["lens"]), P(c["sidx"]), P(c["off"])
    out = {}
    if which == "tc":
        nb = LIB.raw("mmda_lstm_tc_workspace_bytes")(B, H, Tmax)
        assert nb > 0, nb
        ws = torch.zeros(nb // 4 + 1, dtype=torch.int32, device=dev)
        LIB.call("mmda_lstm_tc_forward", P(G), w0, w1, P(y), P(cc), lens, sidx, off, P(utt), ld,
                 uo_f, uo_r, B, H, Tmax, save, P(ws), st)
        torch.cuda.synchronize()
        out["err_fwd"] = int(ws[0])
    elif gru:
        LIB.call("mmda_gru_forward", P(G), w0, w1, P(y), lens, sidx, off, P(utt), ld, uo_f, uo_r,
                 B, H, Tmax, save, st)
    else:
        LIB.call("mmda_lstm_forward", P(G), w0, w1, P(y), P(cc), lens, sidx, off, P(utt), ld, uo_f,
                 uo_r, B, H, Tmax, save, st)
    torch.cuda.synchronize()
    out.update(y=y.clone(), c=None if cc is None else cc.clone(), act=G.clone(), utt=utt.clone())
    if not save:
        return out
    # backward on the forward's own saved state
    if which == "tc":
        LIB.call("mmda_lstm_tc_backward", P(G), w0, w1, P(cc), P(c["dy"]), P(c["dutt"]), ld, uo_f,
                 uo_r, lens, sidx, off, B, H, Tmax, P(ws), st)
        torch.cuda.synchronize()
        out["err_bwd"] = int(ws[0])
    else:
        nb = LIB.raw("mmda_lstm_scratch_bytes")(B, H)
        assert nb > 0, nb
        scr = torch.full((2 * (nb // 4),), SENTINEL, device=dev)
        scr[: nb // 4] = 0
        LIB.call("mmda_gru_backward" if gru else "mmda_lstm_backward", P(G), w0, w1,
                 P(y if gru else cc), P(c["dy"]), P(c["dutt"]), ld, uo_f, uo_r, lens, sidx, off,
                 P(scr), B, H, Tmax, st)
        torch.cuda.synchronize()
        out["scratch_overrun"] = int((scr[nb // 4:] != SENTINEL).sum())
    out["dG"] = G.clone()
    return out


def ref64_bwd(c, act, cc, dtype=torch.float64):
    """Explicit LSTM BPTT from saved activations: d(pre-activation gates) [N][8H]."""
    B, H, Tmax = c["B"], c["H"], c["Tmax"]
    dev = act.device
    A = act.to(dtype).view(-1, 2, H, 4)
    C = cc.to(dtype).view(-1, 2, H)
    dy = None if c["dy"] is None else c["dy"].to(dtype).view(-1, 2, H)
    dutt = c["dutt"].to(dtype)
    ls, off, si = c["ls_cpu"], c["off_cpu"], c["si_cpu"].to(dev)
    _, uo_f, uo_r = c["utt_layout"]
    dG = torch.zeros_like(A)
    for d in range(2):
        W = c["whh"][d].to(dtype).view(4, H, H)
        dh_rec = torch.zeros(B, H, dtype=dtype, device=dev)
        dc = torch.zeros_like(dh_rec)
        ts = range(Tmax - 1, -1, -1) if d == 0 else range(Tmax)
        for t in ts:
            n = int((ls > t).sum())
            if n == 0:
                continue
            rows = slice(int(off[t]), int(off[t]) + n)
            dh = torch.zeros(n, H, dtype=dtype, device=dev) if dy is None else dy[rows, d].clone()
            lsn = ls[:n].to(dev)
            fin = (lsn - 1 == t) if d == 0 else torch.full((n,), t == 0, device=dev)
            uo = uo_f if d == 0 else uo_r
            dh = dh + fin[:, None] * dutt[si[:n]][:, uo:uo + H]
            dh = dh + dh_rec[:n]      # rows that just became active still carry zeros
            i, f, g_, o = A[rows, d, :, 0], A[rows, d, :, 1], A[rows, d, :, 2], A[rows, d, :, 3]
            ct = C[rows, d]
            tp = t - 1 if d == 0 else t + 1
            cp = torch.zeros_like(ct)
            if 0 <= tp < Tmax:
                npv = int((ls > tp).sum())
                m = min(n, npv)
                cp[:m] = C[int(off[tp]):int(off[tp]) + m, d]
            tc = torch.tanh(ct)
            do = dh * tc * o * (1 - o)
            dcc = dc[:n]
            dcc = dcc + dh * o * (1 - tc * tc)
            di = dcc * g_ * i * (1 - i)
            df = dcc * cp * f * (1 - f)
            dg = dcc * i * (1 - g_ * g_)
            dG[rows, d] = torch.stack([di, df, dg, do], -1)
            dc = dc.clone(); dh_rec = dh_rec.clone()
            dc[:n] = dcc * f
            pre = torch.stack([di, df, dg, do], 1)      # [n][4][H]
            dh_rec[:n] = torch.einsum("bgu,guk->bk", pre, W)
    return dG.view(-1, 8 * H)


def timeit(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    B, H, T, ragged = 256, 300, 50, 0
    if len(sys.argv) > 4:
        B, H, T, ragged = (int(x) for x in sys.argv[1:5])
    dev = torch.device("cuda:0")
    c = make_case(B, H, T, ragged, dev)
    plan = (torch.zeros(8, dtype=torch.int32))
    import ctypes
    arr = (ctypes.c_int * 8)()
    LIB.call("mmda_lstm_tc_plan", B, H, c["Tmax"], arr)
    print("plan S,G,BT,NT,Kp,smem_f,smem_b,ctas:", list(arr), flush=True)
    y64, c64, a64, u64 = ref64(c)
    dG64 = ref64_bwd(c, a64, c64)
    res = {}
    for which in ("simt", "tc"):
        o = run(c, which)
        res[which] = o
        row = {k: rel(o[k], r) for k, r in (("y", y64), ("c", c64), ("act", a64), ("utt", u64), ("dG", dG64))}
        row.update({k: v for k, v in o.items() if k.startswith("err")})
        print(which, "vs fp64:", json.dumps(row), flush=True)
    print("tc vs simt:", json.dumps({k: rel(res["tc"][k], res["simt"][k]) for k in ("y", "c", "act", "utt", "dG")}),
          flush=True)

    # ---- timing (forward, backward) ----
    st = torch.cuda.current_stream().cuda_stream
    N = c["N"]
    G = c["gates"].clone()
    y = torch.zeros(N, 2 * H, device=dev); cc = torch.zeros(N, 2 * H, device=dev)
    utt = torch.zeros(B, 4 * H, device=dev)
    nb = LIB.raw("mmda_lstm_tc_workspace_bytes")(B, H, c["Tmax"])
    ws = torch.zeros(nb // 4 + 1, dtype=torch.int32, device=dev)
    scr = torch.zeros(max(1, LIB.raw("mmda_lstm_scratch_bytes")(B, H) // 4), device=dev)
    Gs = res["tc"]["act"]

    def f_tc():
        G.copy_(c["gates"])
        LIB.call("mmda_lstm_tc_forward", P(G), P(c["whh"][0]), P(c["whh"][1]), P(y), P(cc), P(c["lens"]),
                 P(c["sidx"]), P(c["off"]), P(utt), 4 * H, 0, 2 * H, B, H, c["Tmax"], 1, P(ws), st)

    def f_simt():
        G.copy_(c["gates"])
        LIB.call("mmda_lstm_forward", P(G), P(c["whh"][0]), P(c["whh"][1]), P(y), P(cc), P(c["lens"]),
                 P(c["sidx"]), P(c["off"]), P(utt), 4 * H, 0, 2 * H, B, H, c["Tmax"], 1, st)

    def b_tc():
        G.copy_(Gs)
        LIB.call("mmda_lstm_tc_backward", P(G), P(c["whh"][0]), P(c["whh"][1]), P(res["tc"]["c"]), P(c["dy"]),
                 P(c["dutt"]), 4 * H, 0, 2 * H, P(c["lens"]), P(c["sidx"]), P(c["off"]), B, H, c["Tmax"],
                 P(ws), st)

    def b_simt():
        G.copy_(Gs)
        LIB.call("mmda_lstm_backward", P(G), P(c["whh"][0]), P(c["whh"][1]), P(res["tc"]["c"]), P(c["dy"]),
                 P(c["dutt"]), 4 * H, 0, 2 * H, P(c["lens"]), P(c["sidx"]), P(c["off"]), P(scr), B, H,
                 c["Tmax"], st)

    def copy_only():
        G.copy_(Gs)

    t_copy = timeit(copy_only)
    print("ms (copy subtracted): " + json.dumps({
        "fwd_tc": timeit(f_tc) - t_copy, "fwd_simt": timeit(f_simt) - t_copy,
        "bwd_tc": timeit(b_tc) - t_copy, "bwd_simt": timeit(b_simt) - t_copy, "copy": t_copy}), flush=True)


if __name__ == "__main__":
    main()
