"""Loss, head and metric kernels (csrc/loss.cu, mmda_threshold) through the C ABI against fp64.

Every phase of the fused loss (phase1, phase2, gram, finalize, dxn, phase4a, phase4b, grad_misc,
domain) runs in the order the trainer runs it, and each intermediate -- segA, XN and inv_norm, the
moment sums and Grams (segB), the six losses and the CMD coefficients, DXN before and after
phase4a, segC, dZ, dscores, dtcp, dR, dO -- is compared with the torch mirror
`loss_phases_ref.phased_loss` evaluated in fp64 on the same fp32 inputs (the mirror is pinned to
autograd of the oracle by test_loss_phases_cpu.py).  Bound: 1e-5 scale-relative, or 3x the error
of the same mirror run in fp32 where that fp32 evaluation itself comes within 3x of 1e-5.  The
case matrix crosses the warp width and the d <= 256 column limit, the B = 192 / 193 change of the
phase2 / phase4a grid, NC up to 8, scores at the BCE clamps, the adversarial domain term, and the
data-parallel statistics split (W shards summing their segments where the all-reduce would).

Ill-conditioned cases (shared tokens with nearly equal moments, where the CMD gradient is a ratio
of vanishing differences) show how far even an exact-formula fp32 evaluation is from fp64 there;
the fp32 mirror's error is reported beside the kernel's on every row.  The heads
(mmda_linear_skinny), the threshold and the evaluation metrics are checked the same way, and
every refused argument must raise and write nothing.  Every row lands in
test_reports/loss_kernels.txt."""
import os

import numpy as np
import pytest
import torch

from helpers import ROOT, max_rel
from loss_phases_ref import domain_loss, phased_loss

pytestmark = pytest.mark.gpu
TOL = 1e-5
NAN = float("nan")
EDGE_SCORES = (0.0, 1.0, 1e-7, 1.0 - 2.0 ** -24)     # -100 log clamp and 1e-12 gradient clamp
WD, WS, WR, WC = 0.3, 0.7, 0.7, 0.3
LOSS_KEYS = ("cls", "diff", "sim", "recon", "conf", "total")
ACTS = {0: lambda v: v, 1: lambda v: torch.where(v > 0, v, 0.01 * v), 2: torch.sigmoid,
        3: torch.relu, 4: torch.tanh}


# ------------------------------------------------------------------------------------------
# report
# ------------------------------------------------------------------------------------------
class Table:
    """Rows of (case, quantity, kernel error, bound, fp32 mirror error); written at module end."""

    def __init__(self):
        self.rows = []

    def add(self, case, qty, got, ref, bound=TOL, mirror=None, scale=None):
        err = max_rel_scaled(got, ref, scale)
        self.rows.append((case, qty, err, bound, mirror))
        return err

    def exact(self, case, qty, ok):
        self.rows.append((case, qty, 0.0 if ok else float("inf"), 0.0, None))

    def check(self, case):
        bad = [(q, e, b) for c, q, e, b, _ in self.rows if c == case and not e <= b]    # NaN fails
        assert not bad, f"{case}: " + ", ".join(f"{q} err={e:.3e} > {b:.1e}" for q, e, b in bad)

    def write(self):
        out = os.path.join(ROOT, "test_reports")
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "loss_kernels.txt"), "w") as f:
            f.write("status case quantity | kernel vs fp64 | bound | fp32 mirror vs fp64\n")
            for c, q, e, b, m in self.rows:
                f.write(f"{'ok  ' if e <= b else 'FAIL'} {c:44s} {q:14s} err={e:.3e} bound={b:.1e}"
                        + (f" mirror32={m:.3e}" if m is not None else "") + "\n")
            worst = {}
            for c, q, e, b, m in self.rows:
                key = (q, "ill" if c.startswith("ill") else "std")
                if e == e and e > worst.get(key, (-1,))[0]:
                    worst[key] = (e, c)
            f.write("worst per quantity (std = well-conditioned matrix, ill = ill-conditioned):\n")
            for (q, reg), (e, c) in sorted(worst.items()):
                f.write(f"  {reg} {q:14s} {e:.3e}  ({c})\n")


@pytest.fixture(scope="module")
def table():
    t = Table()
    yield t
    t.write()


@pytest.fixture(scope="module")
def k():
    assert torch.cuda.is_available(), "GPU tests need a B200"
    from mmda_b200.engine import Kernels
    kk = Kernels()
    kk.bind_stream()
    return kk


def P(t):
    return None if t is None else t.data_ptr()


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------
def make_inputs(B, d, NC, seed, edges=True, tokens=None):
    """fp32 CPU tensors drawn as in test_loss_phases_cpu._rand_outputs: tokens and scores in
    (0.05, 0.95), every class with a positive label; some scores at the clamp edges."""
    g = torch.Generator().manual_seed(seed)
    X0 = torch.rand(B, 6, d, generator=g) * 0.9 + 0.05
    if tokens is not None:
        X0 = tokens(X0, g)
    O = torch.randn(3, B, d, generator=g)
    R = torch.randn(3, B, d, generator=g)
    s = torch.rand(B, NC, generator=g) * 0.9 + 0.05
    t = torch.rand(B, NC, generator=g)
    y = (torch.rand(B, NC, generator=g) < 0.4).float()
    edge = torch.zeros(B, NC, dtype=torch.bool)
    if edges:
        n = B * NC
        pos = torch.randperm(n, generator=g)[:2 * len(EDGE_SCORES)]
        for j, p in enumerate(pos.tolist()):
            s.view(-1)[p] = EDGE_SCORES[j % len(EDGE_SCORES)]
            y.view(-1)[p] = float(j // len(EDGE_SCORES) == 0)
            edge.view(-1)[p] = True
    y[0] = 1.0
    DL = (torch.rand(3 * B, 3, generator=g) * 2 - 1) * 80
    return dict(X0=X0, O=O, R=R, s=s, t=t, y=y, DL=DL, edge=edge)


def reference(inp, Bg, w_conf, adv, dtype=torch.float64):
    c = lambda v: v.to(dtype)
    w = dict(diff=WD, sim=WS, recon=WR, conf=w_conf)
    return phased_loss(c(inp["X0"]), c(inp["O"]), c(inp["R"]), c(inp["s"]), c(inp["t"]), c(inp["y"]),
                       float(Bg), w, DL=c(inp["DL"]) if adv else None, intermediates=True)


# ------------------------------------------------------------------------------------------
# the kernel chain
# ------------------------------------------------------------------------------------------
class Shard:
    """Device buffers of one rank (layouts of FusedTrainer._loss_buffers); `misalign` puts segB
    one float past a 16-byte boundary, which takes finalize's scalar Gram path."""

    def __init__(self, inp, B, d, NC, dev, misalign=False):
        self.B, self.d, self.NC = B, d, NC
        f = lambda *s: torch.full(s, NAN, device=dev)
        self.X0 = inp["X0"].to(dev).contiguous()
        self.O, self.R = inp["O"].to(dev).contiguous(), inp["R"].to(dev).contiguous()
        self.s, self.t, self.y = (inp[n].to(dev).contiguous() for n in ("s", "t", "y"))
        self.DL = inp["DL"].to(dev).contiguous()
        self.segA = torch.zeros(6 * d + 6 * NC + 4, device=dev)
        nB = 12 * d + 6 * d * d
        self._segB = torch.zeros(nB + 4, device=dev)
        self.segB = self._segB[1:1 + nB] if misalign else self._segB[:nB]
        self.segC = torch.zeros(6 * d, device=dev)
        self.losses = torch.zeros(8, device=dev)
        self.coef = torch.zeros(15 * d, device=dev)
        self.XN, self.inv, self.DXN = f(6, B, d), f(6, B), f(6, B, d)
        self.dZ, self.dSC, self.dTCP = f(B, 6, d), f(B, NC), f(B, NC)
        self.dR, self.dO, self.dDL = f(3, B, d), f(3, B, d), f(3 * B, 3)
        self.DXN_pre = None

    @property
    def G(self):
        return self.segB[12 * self.d:].view(6, self.d, self.d)


def stages(k, sh, Bg, w_conf, adv, early):
    """The loss chain of FusedTrainer as (launch, all-reduced segment) stages: `_loss_early` +
    `loss_and_grads(early_ev)` when early, else `loss_and_grads` with `_loss_tokens(mode=3)`."""
    B, d, NC = sh.B, sh.d, sh.NC
    w_sim = 0.0 if adv else WS
    alpha = WD * 2.0 / float(d * d)

    def p1(roles):
        if roles == 1:
            k._c("mmda_loss_phase1", P(sh.X0), None, None, None, None, None, P(sh.segA), B, d, NC, 1)
        else:
            k._c("mmda_loss_phase1", P(sh.X0), P(sh.O), P(sh.R), P(sh.s), P(sh.t), P(sh.y), P(sh.segA),
                 B, d, NC, roles)
        if roles & 2 and adv:
            k._c("mmda_loss_domain", P(sh.DL), P(sh.dDL), P(sh.segA), B, d, NC, Bg, WS)

    def p2():
        k._c("mmda_loss_phase2", P(sh.X0), P(sh.segA), P(sh.XN), P(sh.inv), P(sh.segB), B, d, Bg)
        k._c("mmda_loss_gram", P(sh.XN), P(sh.G), B, d)

    def fin(mode):
        k._c("mmda_loss_finalize", P(sh.segA), P(sh.segB), P(sh.losses), P(sh.coef), d, NC, Bg,
             WD, WS, WR, w_conf, int(adv), mode)

    def p3(mode):
        fin(mode)
        k._c("mmda_loss_dxn", P(sh.XN), P(sh.G), P(sh.DXN), B, d, alpha)
        sh.DXN_pre = sh.DXN.clone()
        k._c("mmda_loss_phase4a", P(sh.DXN), P(sh.inv), P(sh.segC), B, d)

    def p4b():
        k._c("mmda_loss_phase4b", P(sh.X0), P(sh.DXN), P(sh.segA), P(sh.segB), P(sh.segC), P(sh.coef),
             P(sh.dZ), B, d, Bg, w_sim, 0)

    def misc():
        k._c("mmda_loss_grad_misc", P(sh.s), P(sh.t), P(sh.y), P(sh.O), P(sh.R), P(sh.segA), P(sh.dSC),
             P(sh.dTCP), P(sh.dR), P(sh.dO), B, d, NC, Bg, WR, w_conf)

    if early:
        return [(lambda: p1(1), sh.segA[:6 * d]), (p2, sh.segB), (lambda: p3(1), sh.segC),
                (lambda: (p4b(), p1(2)), sh.segA[6 * d:]), (lambda: (fin(2), misc()), None)]
    return [(lambda: p1(3), sh.segA), (p2, sh.segB), (lambda: p3(3), sh.segC),
            (lambda: (p4b(), misc()), None)]


def run_chain(k, shards, Bg, w_conf, adv, early):
    """Run the shards in lock-step; between stages every shard's segment is replaced by the sum
    over the shards (what the sum all-reduce leaves on every rank)."""
    plans = [stages(k, sh, Bg, w_conf, adv, early) for sh in shards]
    for st in range(len(plans[0])):
        for pl in plans:
            pl[st][0]()
        segs = [pl[st][1] for pl in plans]
        if len(shards) > 1 and segs[0] is not None:
            tot = segs[0].clone()
            for s in segs[1:]:
                tot += s
            for s in segs:
                s.copy_(tot)
    torch.cuda.synchronize()


def ref_quantities(ref, edge):
    """Name -> tensor for one run of the mirror; `edge` marks the clamp-edge scores."""
    L, g, I = ref
    A = I["segA"]
    q = {"colsum": A["colsum"], "bce": A["bce"], "sqtcp": A["sq"], "sum_ys": A["sys"], "sum_y": A["sy"],
         "sumexp": A["se"], "recon_sq": A["rsq"], "XN": I["XN"].permute(1, 0, 2), "inv_norm": I["inv"].t(),
         "moments": I["M"], "gram": I["G"], "coef": I["coef"], "DXN": I["DXN"].permute(1, 0, 2),
         "DXN*inv": I["dxc"].permute(1, 0, 2), "segC": I["colsum2"], "dZ": g["d_tokens"],
         "dZ[private]": g["d_tokens"][:, :3], "dtcp": g["d_tcp"], "dR": g["d_recon"], "dO": g["d_orig"],
         "dscores": g["d_scores"][~edge], "dscores@edge": g["d_scores"][edge]}
    if "d_domain" in g:
        q["dom_sum"], q["dDL"] = A["dom"], g["d_domain"]
    q.update({"L." + n: L[n] for n in LOSS_KEYS})
    return q


def kernel_quantities(sh, edge):
    d, NC = sh.d, sh.NC
    segA = sh.segA.cpu().double()
    cls = segA[6 * d:]
    edge = edge.to(sh.dSC.device)
    q = {"colsum": segA[:6 * d].view(6, d), "bce": cls[0:NC], "sqtcp": cls[NC:2 * NC],
         "sum_ys": cls[2 * NC:3 * NC], "sum_y": cls[3 * NC:4 * NC], "sumexp": cls[5 * NC:6 * NC],
         "recon_sq": cls[6 * NC:6 * NC + 3], "XN": sh.XN, "inv_norm": sh.inv,
         "moments": sh.segB[:12 * d].view(3, 4, d), "gram": sh.G, "coef": sh.coef.view(3, 5, d),
         "DXN": sh.DXN_pre, "DXN*inv": sh.DXN, "segC": sh.segC.view(6, d), "dZ": sh.dZ,
         "dZ[private]": sh.dZ[:, :3], "dtcp": sh.dTCP, "dR": sh.dR, "dO": sh.dO,
         "dscores": sh.dSC[~edge], "dscores@edge": sh.dSC[edge], "dom_sum": cls[6 * NC + 3], "dDL": sh.dDL,
         "nnz": cls[4 * NC:5 * NC]}
    q.update({"L." + n: sh.losses[i] for i, n in enumerate(LOSS_KEYS)})
    return q


def compare(table, case, sh, inp, ref, mirror, skip=()):
    """Every intermediate and output of one single-rank chain against the fp64 mirror `ref`.
    Bound: max(1e-5, 3 x the error of `mirror`, the same formulas run in fp32).  That is the hard
    1e-5 unless an exact-formula fp32 evaluation itself comes within 3x of it, as it does where
    a result divides by a vanishing difference: the CMD coefficients of nearly equal moments, or
    the row norms at d = 1, where a row's one centred entry can be ~0.  segC is a column sum of
    entries that nearly cancel (the rows of DXN are centred but for the row scaling), so its error
    is measured against the sum of the magnitudes it adds, max_c sum_b |DXN*inv[b][c]|."""
    r64, r32 = ref_quantities(ref, inp["edge"]), ref_quantities(mirror, inp["edge"])
    got = kernel_quantities(sh, inp["edge"])
    seg_scale = float(r64["DXN*inv"].abs().sum(1).max())
    for q, r in r64.items():
        if q in skip or r.numel() == 0 or (q == "dZ[private]" and "dZ" not in skip):
            continue
        sc = seg_scale if q == "segC" else None
        m = max_rel_scaled(r32[q], r, sc)
        table.add(case, q, got[q], r, max(TOL, 3 * m) if m == m else TOL, m, scale=sc)
    table.exact(case, "nnz", torch.equal(got["nnz"], ref[2]["segA"]["nnz"]))


def max_rel_scaled(a, b, scale=None):
    """max_rel, or max |a - b| / scale."""
    a, b = (v.detach().double().cpu() if torch.is_tensor(v) else torch.tensor(v, dtype=torch.float64)
            for v in (a, b))
    if scale is None:
        return max_rel(a, b)
    return float((a - b).abs().max()) / (scale + 1e-30)


# ------------------------------------------------------------------------------------------
# 1. the chain over the case matrix
# ------------------------------------------------------------------------------------------
# (B, d, NC, confid, adversarial, early split, segB misaligned)
CASES = [(192, dd, nc, cf, False, False, False) for dd, nc, cf in
         [(1, 1, True), (31, 6, False), (32, 7, True), (33, 8, False), (128, 6, True), (200, 7, True),
          (256, 8, False)]]
CASES += [(b, 128, 6, True, False, False, False) for b in (2, 7, 8, 9, 191, 193, 256, 1000, 4096)]
CASES += [(b, 33, 1, False, False, False, False) for b in (2, 9, 193)]
CASES += [(4096, 256, 8, True, False, False, False), (1000, 200, 7, False, False, False, False)]
CASES += [(b, 128, 6, True, True, False, False) for b in (1, 85, 86, 1000)]        # adversarial
CASES += [(256, 128, 6, True, False, True, False), (193, 33, 7, False, True, True, False),
          (256, 128, 6, True, False, False, True), (9, 33, 6, True, False, False, True),
          (1, 128, 6, True, False, False, False), (1, 31, 8, False, False, True, False)]


def case_id(c):
    B, d, NC, cf, adv, early, mis = c
    return (f"B{B}_d{d}_nc{NC}" + ("_conf" if cf else "") + ("_adv" if adv else "")
            + ("_early" if early else "") + ("_misaligned" if mis else ""))


@pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
def test_loss_chain_vs_fp64(case, k, table):
    B, d, NC, confid, adv, early, mis = case
    name = case_id(case)
    w_conf = WC if confid else 0.0
    inp = make_inputs(B, d, NC, seed=B * 1000 + d * 10 + NC)
    sh = Shard(inp, B, d, NC, torch.device("cuda:0"), misalign=mis)
    run_chain(k, [sh], float(B), w_conf, adv, early)
    ref, mirror = reference(inp, B, w_conf, adv), reference(inp, B, w_conf, adv, dtype=torch.float32)
    skip = ()
    if B <= 2:
        # the centred odd moments (at B = 1 all of them) vanish for every token: the CMD
        # coefficients are 0/0 in the reference as well, and outside the adversarial variant so
        # is the shared tokens' dZ (the private tokens' dZ is still checked)
        skip = ("coef",) + (() if adv else ("dZ",))
    compare(table, name, sh, inp, ref, mirror, skip=skip)
    table.check(name)


# ------------------------------------------------------------------------------------------
# 2. the data-parallel statistics split on one GPU
# ------------------------------------------------------------------------------------------
DP_CASES = [(2, 96, 128, 6, True, False, True), (4, 48, 128, 7, False, False, False),
            (8, 24, 33, 6, True, False, True), (8, 128, 128, 8, True, False, False),
            (2, 43, 128, 6, True, True, True)]


@pytest.mark.parametrize("case", DP_CASES, ids=[f"W{c[0]}_B{c[1]}_d{c[2]}_nc{c[3]}" + ("_conf" if c[4] else "")
                                                + ("_adv" if c[5] else "") + ("_early" if c[6] else "")
                                                for c in DP_CASES])
def test_data_parallel_split_vs_global_batch(case, k, table):
    W, B, d, NC, confid, adv, early = case
    name = f"dp_W{W}_B{B}_d{d}_nc{NC}" + ("_adv" if adv else "") + ("_early" if early else "")
    w_conf = WC if confid else 0.0
    Bg = W * B
    inp = make_inputs(Bg, d, NC, seed=77 + W * B)
    dev = torch.device("cuda:0")
    shards = []
    for r in range(W):
        sl = slice(r * B, (r + 1) * B)
        part = dict(X0=inp["X0"][sl], O=inp["O"][:, sl], R=inp["R"][:, sl], s=inp["s"][sl], t=inp["t"][sl],
                    y=inp["y"][sl], DL=inp["DL"].view(3, Bg, 3)[:, sl].reshape(3 * B, 3))
        shards.append(Shard(part, B, d, NC, dev))
    run_chain(k, shards, float(Bg), w_conf, adv, early)
    L, g, I = reference(inp, Bg, w_conf, adv)
    cat = lambda name, dim: torch.cat([getattr(s, name) for s in shards], dim)
    table.add(name, "dZ", cat("dZ", 0), g["d_tokens"])
    table.add(name, "dR", cat("dR", 1), g["d_recon"])
    table.add(name, "dtcp", cat("dTCP", 0), g["d_tcp"])
    edge = inp["edge"]
    dsc = cat("dSC", 0).cpu()
    table.add(name, "dscores", dsc[~edge], g["d_scores"][~edge])
    table.add(name, "dscores@edge", dsc[edge], g["d_scores"][edge])
    if adv:
        table.add(name, "dDL", torch.cat([s.dDL.view(3, B, 3) for s in shards], 1).view(-1, 3), g["d_domain"])
    for i, q in enumerate(LOSS_KEYS):
        table.add(name, "L." + q, shards[0].losses[i], L[q])
    table.add(name, "coef", shards[0].coef.view(3, 5, d), I["coef"])
    table.exact(name, "losses equal on every shard",
                all(same_bits(s.losses, shards[0].losses) for s in shards[1:]))
    table.check(name)


# ------------------------------------------------------------------------------------------
# 3. ill-conditioned regime: shared tokens with nearly equal moments
# ------------------------------------------------------------------------------------------
def _near(scale):
    def f(X0, g):
        X0 = X0.clone()
        for j in (4, 5):
            X0[:, j] = X0[:, 3] + scale * torch.randn(X0[:, 3].shape, generator=g)
        return X0
    return f


ILL = [("uniform", 256, None), ("near_1e-2", 256, _near(1e-2)), ("near_1e-3", 256, _near(1e-3)),
       ("offset_10", 256, lambda X0, g: X0 + 10.0), ("near_1e-2", 4096, _near(1e-2))]


@pytest.mark.parametrize("case", ILL, ids=[f"{c[0]}_B{c[1]}" for c in ILL])
def test_ill_conditioned_vs_fp32_mirror(case, k, table):
    tag, B, tokens = case
    name, d, NC = f"ill_{tag}_B{B}_d128", 128, 6
    inp = make_inputs(B, d, NC, seed=5 + B, edges=False, tokens=tokens)
    sh = Shard(inp, B, d, NC, torch.device("cuda:0"))
    run_chain(k, [sh], float(B), WC, False, False)
    ref = reference(inp, B, WC, False)
    mirror = reference(inp, B, WC, False, dtype=torch.float32)
    compare(table, name, sh, inp, ref, mirror)
    table.check(name)


# ------------------------------------------------------------------------------------------
# 4. the adversarial domain term alone
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 85, 86, 1000])
def test_domain_cross_entropy_vs_fp64(B, k, table):
    d, NC, Bg = 128, 6, float(B)
    g = torch.Generator().manual_seed(B)
    DL = (torch.rand(3 * B, 3, generator=g) * 2 - 1) * 80
    DL[0] = torch.tensor([80.0, -80.0, -80.0])      # label logit far above the others: loss ~ 0
    DL[-1] = torch.tensor([80.0, 80.0, -80.0])      # label logit far below: loss ~ 160
    dev = torch.device("cuda:0")
    DLd = DL.to(dev)
    segA = torch.full((6 * d + 6 * NC + 4,), NAN, device=dev)
    dDL = torch.full((3 * B, 3), NAN, device=dev)
    k._c("mmda_loss_domain", P(DLd), P(dDL), P(segA), B, d, NC, Bg, WS)
    torch.cuda.synchronize()
    ref_sum, ref_grad = domain_loss(DL.double(), Bg, WS)
    name = f"domain_B{B}"
    table.add(name, "dom_sum", segA[6 * d + 6 * NC + 3], ref_sum)
    table.add(name, "dDL", dDL, ref_grad)
    others = torch.cat([segA[:6 * d + 6 * NC + 3], segA[6 * d + 6 * NC + 4:]])
    table.exact(name, "rest of segA untouched", bool(torch.isnan(others).all()))
    table.check(name)


# ------------------------------------------------------------------------------------------
# 5. exact identities
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,d,NC", [(193, 128, 6), (9, 33, 8)])
def test_split_launches_are_bit_identical(B, d, NC, k, table):
    name = f"identities_B{B}_d{d}"
    dev = torch.device("cuda:0")
    inp = make_inputs(B, d, NC, seed=11)
    a, b = Shard(inp, B, d, NC, dev), Shard(inp, B, d, NC, dev)
    p1 = lambda sh, roles: k._c("mmda_loss_phase1", P(sh.X0), P(sh.O), P(sh.R), P(sh.s), P(sh.t), P(sh.y),
                                P(sh.segA), B, d, NC, roles)
    p1(a, 1); p1(a, 2); p1(b, 3)
    torch.cuda.synchronize()
    table.exact(name, "phase1 roles 1+2 == 3", same_bits(a.segA, b.segA))
    s2 = b.segA.clone()
    p1(b, 3)
    table.exact(name, "phase1 rerun", same_bits(s2, b.segA))
    # one phase2 / gram (atomics in phase2: compare the rest on the same segB)
    k._c("mmda_loss_phase2", P(a.X0), P(a.segA), P(a.XN), P(a.inv), P(a.segB), B, d, float(B))
    k._c("mmda_loss_gram", P(a.XN), P(a.G), B, d)
    G1 = a.G.clone()
    k._c("mmda_loss_gram", P(a.XN), P(a.G), B, d)
    torch.cuda.synchronize()
    table.exact(name, "gram rerun", same_bits(G1, a.G))
    b.segB.copy_(a.segB)
    fin = lambda sh, mode: k._c("mmda_loss_finalize", P(sh.segA), P(sh.segB), P(sh.losses), P(sh.coef), d, NC,
                                float(B), WD, WS, WR, WC, 0, mode)
    fin(a, 1); fin(a, 2); fin(b, 3)
    torch.cuda.synchronize()
    table.exact(name, "finalize mode 1+2 == 3", same_bits(a.losses[:6], b.losses[:6])
                and same_bits(a.coef, b.coef))
    k._c("mmda_loss_dxn", P(a.XN), P(a.G), P(a.DXN), B, d, WD * 2.0 / (d * d))
    k._c("mmda_loss_phase4a", P(a.DXN), P(a.inv), P(a.segC), B, d)
    dZ0 = torch.randn(B, 6, d, device=dev)
    acc, fresh = dZ0.clone(), torch.full_like(dZ0, NAN)
    p4b = lambda out, accumulate: k._c("mmda_loss_phase4b", P(a.X0), P(a.DXN), P(a.segA), P(a.segB), P(a.segC),
                                       P(a.coef), P(out), B, d, float(B), WS, accumulate)
    p4b(acc, 1); p4b(fresh, 0)
    torch.cuda.synchronize()
    table.exact(name, "phase4b accumulate", same_bits(acc, dZ0 + fresh))
    table.check(name)


# ------------------------------------------------------------------------------------------
# 6. heads and metrics
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [768, 1030, 4096])
def test_linear_skinny_vs_fp64(K, k, table):
    """Both load paths: float4 when x, w, K and ldx allow it, else scalar (K % 4 != 0, or x / w
    one float off a 16-byte boundary); more than one 256-quad sweep at K = 4096; strided y."""
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(K)
    layouts = [("aligned", 0, 0)] + ([("x+1", 1, 0), ("w+1", 0, 1)] if K % 4 == 0 else [])
    for M in (37, 1000):
        for lay, xo, wo in layouts:
            xs = torch.rand(M * K + 4, generator=g) * 2 - 1
            x = xs.to(dev)[xo:xo + M * K].view(M, K)
            for N in range(1, 9):
                ws = torch.randn(8 * K + 4, generator=g) / K ** 0.5
                w = ws.to(dev)[wo:wo + N * K].view(N, K)
                bias = torch.randn(N, generator=g).to(dev)
                ldy = N + 3
                for act in range(5):
                    b = bias if (N + act) % 2 == 0 else None
                    y = torch.full((M, ldy), NAN, device=dev)
                    k._c("mmda_linear_skinny", P(x), K, P(w), P(b), P(y), ldy, M, N, K, act)
                    torch.cuda.synchronize()
                    pre = x.double() @ w.double().t() + (b.double() if b is not None else 0.0)
                    name = f"skinny_K{K}_M{M}_{lay}_N{N}_act{act}" + ("_bias" if b is not None else "")
                    table.add(name, "y", y[:, :N], ACTS[act](pre))
                    table.exact(name, "y columns past N untouched", bool(torch.isnan(y[:, N:]).all()))
                    table.check(name)


def test_threshold_is_exact(k, table):
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(3)
    for n in (1, 1000, (1 << 20) + 3):
        thr = 0.5
        x = torch.rand(n, generator=g)
        x[::3] = thr                                   # ties must map to 0
        x[1::7] = torch.nextafter(torch.tensor(thr), torch.tensor(1.0))
        xd = x.to(dev)
        out = torch.full((n,), NAN, device=dev)
        k._c("mmda_threshold", P(xd), P(out), n, thr)
        torch.cuda.synchronize()
        table.exact(f"threshold_n{n}", "x > thr", torch.equal(out.cpu(), (x > thr).float()))
        table.check(f"threshold_n{n}")


@pytest.mark.parametrize("NC", [1, 6, 8])
def test_eval_accumulate_vs_fp64(NC, k, table):
    from mmda_b200.evaluate import metrics_from_stats
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(NC)
    stats = torch.zeros(4 + 3 * NC, device=dev)
    jac = bce = 0.0
    tp = np.zeros(NC); fp = np.zeros(NC); fn = np.zeros(NC)
    Bs = (1, 255, 256, 257, 1000)
    for B in Bs:
        s = torch.rand(B, NC, generator=g) * 0.9 + 0.05
        s.view(-1)[:min(4, B * NC)] = torch.tensor(EDGE_SCORES)[:min(4, B * NC)]
        pred = (torch.rand(B, NC, generator=g) < 0.5).float()
        y = (torch.rand(B, NC, generator=g) < 0.4).float()
        sd, pd, yd = s.to(dev), pred.to(dev), y.to(dev)
        k._c("mmda_eval_accumulate", P(sd), P(pd), P(yd), P(stats), B, NC)
        t, p = y.numpy() > 0, pred.numpy() > 0
        jac += float(((t & p).sum(1) / np.maximum((t | p).sum(1), 1)).sum())
        s64, y64 = s.double(), y.double()
        bce += float(-(y64 * torch.log(s64).clamp_min(-100) + (1 - y64) * torch.log(1 - s64).clamp_min(-100))
                     .sum() / B)
        tp += (t & p).sum(0); fp += (~t & p).sum(0); fn += (t & ~p).sum(0)
    torch.cuda.synchronize()
    st = stats.cpu().double()
    name = f"eval_nc{NC}"
    table.add(name, "jaccard_sum", st[0], jac)
    table.add(name, "bce_sum", st[2], bce)
    counts = np.concatenate([[sum(Bs)], [len(Bs)], tp, fp, fn])
    got = np.concatenate([[st[1]], [st[3]], st[4:].numpy()])
    table.exact(name, "samples/batches/TP/FP/FN", bool(np.array_equal(got, counts)))
    # the metrics straight from the fp64 quantities
    div = lambda a, b: np.where(b > 0, a / np.where(b > 0, b, 1), 0.0)
    prec, rec, f1 = div(tp, tp + fp), div(tp, tp + fn), div(2 * tp, 2 * tp + fp + fn)
    sup = tp + fn
    w = lambda v: float((v * sup).sum() / sup.sum()) if sup.sum() > 0 else 0.0
    T, F_, N_ = tp.sum(), fp.sum(), fn.sum()
    ref = {"loss": bce / len(Bs), "acc": round(jac / sum(Bs), 4), "f1": f1.mean(), "precision": prec.mean(),
           "recall": rec.mean(), "micro_f1": 2 * T / (2 * T + F_ + N_), "micro_precision": T / (T + F_),
           "micro_recall": T / (T + N_), "weighted_f1": w(f1), "weighted_precision": w(prec),
           "weighted_recall": w(rec)}
    m = metrics_from_stats(stats.tolist(), NC)
    # acc is rounded to 4 decimals: an fp32 Jaccard sum within 1e-5 of the fp64 one may still
    # round one step away when the mean sits on a rounding boundary
    table.exact(name, "metric.acc", abs(m.pop("acc") - ref.pop("acc")) <= 1.0001e-4)
    for key, v in ref.items():      # the counts are exact, so are the metrics built from them
        table.add(name, "metric." + key, m[key], v, TOL if key == "loss" else 1e-12)
    table.check(name)


# ------------------------------------------------------------------------------------------
# 7. refusals: MmdaError, and nothing written
# ------------------------------------------------------------------------------------------
def test_refusals_launch_nothing(k, table):
    from mmda_b200._lib import MmdaError
    dev = torch.device("cuda:0")
    B, d = 16, 257
    big = lambda n: torch.full((n,), NAN, device=dev)
    X0, O, R = torch.rand(B * 6 * d, device=dev), torch.rand(3 * B * d, device=dev), torch.rand(3 * B * d, device=dev)
    s, t, y = torch.rand(B * 9, device=dev), torch.rand(B * 9, device=dev), torch.ones(B * 9, device=dev)
    segA, segB, outs = big(6 * d + 6 * 9 + 4), big(12 * d + 6 * d * d), big(6 * B * d)
    inv, losses, coef = big(6 * B), big(8), big(15 * d)
    DXN = torch.rand(6 * B * d, device=dev)
    DXN0 = DXN.clone()
    calls = [
        ("phase1 d=257", "mmda_loss_phase1", (P(X0), P(O), P(R), P(s), P(t), P(y), P(segA), B, 257, 6, 3)),
        ("phase1 NC=9", "mmda_loss_phase1", (P(X0), P(O), P(R), P(s), P(t), P(y), P(segA), B, 128, 9, 3)),
        ("phase1 roles=0", "mmda_loss_phase1", (P(X0), P(O), P(R), P(s), P(t), P(y), P(segA), B, 128, 6, 0)),
        ("phase1 roles=4", "mmda_loss_phase1", (P(X0), P(O), P(R), P(s), P(t), P(y), P(segA), B, 128, 6, 4)),
        ("phase2 d=257", "mmda_loss_phase2", (P(X0), P(segA), P(outs), P(inv), P(segB), B, 257, float(B))),
        ("finalize mode=0", "mmda_loss_finalize", (P(segA), P(segB), P(losses), P(coef), 128, 6, float(B),
                                                   WD, WS, WR, WC, 0, 0)),
        ("finalize mode=4", "mmda_loss_finalize", (P(segA), P(segB), P(losses), P(coef), 128, 6, float(B),
                                                   WD, WS, WR, WC, 0, 4)),
        ("phase4a d=257", "mmda_loss_phase4a", (P(DXN), P(inv), P(outs), B, 257)),
        ("linear_skinny N=9", "mmda_linear_skinny", (P(X0), 768, P(O), None, P(outs), 9, B, 9, 768, 0)),
        ("eval_accumulate NC=9", "mmda_eval_accumulate", (P(s), P(s), P(y), P(coef), B, 9)),
        ("eval_accumulate B=0", "mmda_eval_accumulate", (P(s), P(s), P(y), P(coef), 0, 6)),
    ]
    for label, fn, args in calls:
        raised = False
        try:
            k._c(fn, *args)
        except MmdaError:
            raised = True
        table.exact("refusals", label + " raises", raised)
    torch.cuda.synchronize()
    untouched = all(bool(torch.isnan(b).all()) for b in (segA, segB, outs, inv, losses, coef))
    table.exact("refusals", "no output written", untouched and torch.equal(DXN, DXN0))
    table.check("refusals")
