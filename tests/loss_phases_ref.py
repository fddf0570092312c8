"""Torch mirror of the phased loss kernels (mmda_b200/csrc/loss.cu), same formulas and the same
three all-reducible statistic segments.  Test helper only: it lets the CPU suite check the
hand-derived loss backward and the batch-sharded decomposition (SURVEY.md row D1) against
autograd of the oracle, with `reduce` standing in for the NCCL all-reduce."""
import torch

PAIRS = ((0, 3), (1, 4), (2, 5), (2, 0), (2, 1), (0, 1))
CMD_PAIRS = ((0, 1), (0, 2), (2, 1))


def domain_loss(DL, Bg, w_sim):
    """Adversarial similarity term (mmda_loss_domain): cross-entropy of the 3B domain logits DL
    (3B,3), rows [pred_t; pred_v; pred_a] with labels 0/1/2.  Returns (batch sum of the row
    losses, d(w_sim * sum / (3 Bg)) / d DL)."""
    B3 = DL.shape[0]
    lab = torch.arange(3, device=DL.device).repeat_interleave(B3 // 3)
    logp = torch.log_softmax(DL, dim=1)
    onehot = torch.nn.functional.one_hot(lab, 3).to(DL.dtype)
    return -(logp * onehot).sum(), w_sim / (3 * Bg) * (logp.exp() - onehot)


def phased_loss(X0, O, R, scores, tcp, y, Bg, w, reduce=lambda t: t, DL=None, intermediates=False):
    """X0 (B,6,d) [p_t,p_v,p_a,s_t,s_v,s_a]; O,R (3,B,d); scores,tcp,y (B,NC).
    w = dict(diff, sim, recon, conf).  DL (3B,3): the domain logits of the adversarial variant
    (use_cmd_sim=False): sim is then their cross-entropy and the CMD gradient is off.  Returns
    (losses dict, grads dict), plus a dict of the phases' intermediates with intermediates=True."""
    B, _, d = X0.shape
    # phase 1
    segA = dict(colsum=X0.sum(0),
                bce=-(y * torch.log(scores).clamp_min(-100) + (1 - y) * torch.log(1 - scores).clamp_min(-100)).sum(0),
                sq=((tcp - y * scores) ** 2).sum(0), sys=(y * scores).sum(0), sy=y.sum(0),
                nnz=(y != 0).to(X0.dtype).sum(0), se=torch.exp(scores).sum(0),
                rsq=((R - O) ** 2).sum((1, 2)))
    if DL is not None:
        segA["dom"], d_domain = domain_loss(DL, Bg, w["sim"])
    segA = {k: reduce(v) for k, v in segA.items()}
    mu = segA["colsum"] / Bg                                   # (6,d)
    # phase 2
    xc = X0 - mu
    inv = 1.0 / (xc.norm(dim=2) + 1e-6)                        # (B,6)
    XN = xc * inv.unsqueeze(2)
    M = torch.stack([(xc[:, 3:] ** k).sum(0) for k in (2, 3, 4, 5)], 1)      # (3,4,d)
    G = torch.stack([XN[:, a].t() @ XN[:, b] for a, b in PAIRS])            # (6,d,d)
    M, G = reduce(M), reduce(G)
    # finalize
    diff = (G ** 2).sum() / (d * d)
    cmom = torch.cat([mu[3:].unsqueeze(1), M / Bg], 1)          # (3,5,d): c_1..c_5
    coef = torch.zeros_like(cmom)
    cmd = 0.0
    for a, b in CMD_PAIRS:
        for k in range(5):
            dl = cmom[a, k] - cmom[b, k]
            nrm = dl.norm()
            cmd = cmd + nrm
            coef[a, k] += dl / nrm
            coef[b, k] -= dl / nrm
    cmd = cmd / 3
    if DL is not None:
        cmd = segA["dom"] / (3 * Bg)
    cls = (segA["bce"] / Bg).sum()
    recon = segA["rsq"].sum() / (Bg * d) / 3
    conf = ((segA["sq"] / Bg) / segA["nnz"] + (-segA["sys"] + segA["sy"] * torch.log(segA["se"])) / segA["nnz"]).sum()
    total = cls + w["diff"] * diff + w["sim"] * cmd + w["recon"] * recon + w["conf"] * conf
    L = dict(cls=cls, diff=diff, sim=cmd, recon=recon, conf=conf, total=total)
    # diff backward
    alpha = w["diff"] * 2.0 / (d * d)
    DXN = torch.zeros_like(XN)
    for p, (a, b) in enumerate(PAIRS):
        DXN[:, a] += alpha * XN[:, b] @ G[p].t()
        DXN[:, b] += alpha * XN[:, a] @ G[p]
    dxc = DXN * inv.unsqueeze(2)
    colsum2 = reduce(dxc.sum(0))
    dZ = dxc - colsum2 / Bg
    # cmd backward (the adversarial variant has none: at B = 1 its coefficients are 0/0)
    for a in range(3 if DL is None else 0):
        x = xc[:, 3 + a]
        t = coef[a, 0].expand_as(x).clone()
        cprev = X0.new_zeros(d)
        for k in range(2, 6):
            t = t + coef[a, k - 1] * k * (x ** (k - 1) - cprev)
            cprev = M[a, k - 2] / Bg
        dZ[:, 3 + a] += w["sim"] / (3 * Bg) * t
    kr = w["recon"] * 2.0 / (3 * Bg * d)
    dR = kr * (R - O)
    ds = (scores - y) / ((1 - scores) * scores).clamp_min(1e-12) / Bg
    dt = torch.zeros_like(tcp)
    if w["conf"] != 0:
        nnz = segA["nnz"]
        dt = w["conf"] * 2 * (tcp - y * scores) / (Bg * nnz)
        ds = ds - y * dt + w["conf"] * (-y + segA["sy"] * torch.exp(scores) / segA["se"]) / nnz
    grads = dict(d_tokens=dZ, d_recon=dR, d_orig=-dR, d_scores=ds, d_tcp=dt)
    if DL is not None:
        grads["d_domain"] = d_domain
    if not intermediates:
        return L, grads
    return L, grads, dict(segA=segA, mu=mu, XN=XN, inv=inv, M=M, G=G, coef=coef, DXN=DXN, dxc=dxc,
                          colsum2=colsum2)
