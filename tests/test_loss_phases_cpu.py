"""The hand-derived loss backward and its batch-sharded decomposition, checked on CPU against
autograd of the oracle's losses (which are pinned to the reference by the golden fixtures)."""
import types

import pytest
import torch

from loss_phases_ref import phased_loss
from oracle.misa_oracle import oracle_losses

MODS = ("t", "v", "a")


def _rand_outputs(B, d, NC, seed):
    g = torch.Generator().manual_seed(seed)
    X0 = torch.rand(B, 6, d, generator=g, dtype=torch.float64) * 0.9 + 0.05
    O = torch.randn(3, B, d, generator=g, dtype=torch.float64)
    R = torch.randn(3, B, d, generator=g, dtype=torch.float64)
    s = torch.rand(B, NC, generator=g, dtype=torch.float64) * 0.9 + 0.05
    t = torch.rand(B, NC, generator=g, dtype=torch.float64)
    y = (torch.rand(B, NC, generator=g) < 0.4).double()
    y[0] = 1.0
    return X0, O, R, s, t, y


def _autograd(X0, O, R, s, t, y, cfg):
    leaves = [v.clone().requires_grad_(True) for v in (X0, O, R, s, t)]
    X0, O, R, s, t = leaves
    out = {"scores": s, "tcp": t}
    for i, m in enumerate(MODS):
        out[f"utt_private_{m}"], out[f"utt_shared_{m}"] = X0[:, i], X0[:, 3 + i]
        out[f"utt_{m}_orig"], out[f"utt_{m}_recon"] = O[i], R[i]
    L = oracle_losses(out, y, cfg)
    L["total"].backward()
    return L, dict(d_tokens=X0.grad, d_orig=O.grad, d_recon=R.grad, d_scores=s.grad, d_tcp=t.grad)


@pytest.mark.parametrize("confid", [False, True])
def test_phased_loss_matches_autograd(confid):
    cfg = types.SimpleNamespace(use_cmd_sim=True, diff_weight=0.3, sim_weight=0.7, recon_weight=0.7,
                                conf_weight=0.3, use_confidNet=confid)
    X0, O, R, s, t, y = _rand_outputs(24, 16, 6, 0)
    Lr, gr = _autograd(X0, O, R, s, t, y, cfg)
    w = dict(diff=0.3, sim=0.7, recon=0.7, conf=0.3 if confid else 0.0)
    L, g = phased_loss(X0, O, R, s, t, y, 24.0, w)
    for k in ("cls", "diff", "sim", "recon", "conf", "total"):
        assert abs(float(L[k]) - float(Lr[k])) < 1e-10 * max(1, abs(float(Lr[k]))), k
    for k in g:
        ref = gr[k] if gr[k] is not None else torch.zeros_like(g[k])
        assert float((g[k] - ref).abs().max()) < 1e-10, k


def test_sharded_statistics_equal_global_batch():
    """Two shards exchanging only the three stat segments reproduce the global-batch loss and
    per-sample gradients exactly (what the NCCL path does between loss phases)."""
    X0, O, R, s, t, y = _rand_outputs(32, 16, 6, 1)
    w = dict(diff=0.3, sim=0.7, recon=0.7, conf=0.3)
    Lg, gg = phased_loss(X0, O, R, s, t, y, 32.0, w)
    shards = [slice(0, 16), slice(16, 32)]
    # emulate the all-reduce: run both shards in lock-step, summing each reduced quantity
    import threading
    results, box, barrier = [None, None], {}, threading.Barrier(2)
    lock = threading.Lock()

    def make_reduce(rank):
        counter = [0]
        def reduce(tn):
            key = counter[0]; counter[0] += 1
            with lock:
                box.setdefault(key, []).append(tn)
            barrier.wait()
            tot = box[key][0] + box[key][1]
            barrier.wait()
            return tot
        return reduce

    def run(rank):
        sl = shards[rank]
        results[rank] = phased_loss(X0[sl], O[:, sl], R[:, sl], s[sl], t[sl], y[sl], 32.0, w,
                                    reduce=make_reduce(rank))
    th = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    [x.start() for x in th]; [x.join() for x in th]
    for rank in range(2):
        L, g = results[rank]
        for k in Lg:
            assert abs(float(L[k]) - float(Lg[k])) < 1e-10, k
        sl = shards[rank]
        assert float((g["d_tokens"] - gg["d_tokens"][sl]).abs().max()) < 1e-12
        assert float((g["d_scores"] - gg["d_scores"][sl]).abs().max()) < 1e-12
        assert float((g["d_recon"] - gg["d_recon"][:, sl]).abs().max()) < 1e-12


@pytest.mark.parametrize("B", [1, 24])
def test_domain_term_matches_autograd(B):
    """Adversarial variant (use_cmd_sim=False): the domain cross-entropy, its gradient wrt the 3B
    logits (logits up to +-80, so the max subtraction matters) and the CMD-free token gradient."""
    cfg = types.SimpleNamespace(use_cmd_sim=False, diff_weight=0.3, sim_weight=0.7, recon_weight=0.7,
                                conf_weight=0.3, use_confidNet=True)
    X0, O, R, s, t, y = _rand_outputs(B, 16, 6, 2)
    g = torch.Generator().manual_seed(3)
    DL = (torch.rand(3 * B, 3, generator=g, dtype=torch.float64) * 2 - 1) * 80
    leaves = [v.clone().requires_grad_(True) for v in (X0, O, R, s, t, DL)]
    out = {"scores": leaves[3], "tcp": leaves[4]}
    for i, m in enumerate(MODS):
        out[f"utt_private_{m}"], out[f"utt_shared_{m}"] = leaves[0][:, i], leaves[0][:, 3 + i]
        out[f"utt_{m}_orig"], out[f"utt_{m}_recon"] = leaves[1][i], leaves[2][i]
        out[f"domain_label_{m}"] = leaves[5][i * B:(i + 1) * B]
    Lr = oracle_losses(out, y, cfg)
    Lr["total"].backward()
    w = dict(diff=0.3, sim=0.7, recon=0.7, conf=0.3)
    L, g = phased_loss(X0, O, R, s, t, y, float(B), w, DL=DL)
    for k in ("cls", "diff", "sim", "recon", "conf", "total"):
        assert abs(float(L[k]) - float(Lr[k])) < 1e-10 * max(1, abs(float(Lr[k]))), k
    ref = dict(d_tokens=leaves[0].grad, d_orig=leaves[1].grad, d_recon=leaves[2].grad,
               d_scores=leaves[3].grad, d_tcp=leaves[4].grad, d_domain=leaves[5].grad)
    for k in g:
        assert float((g[k] - ref[k]).abs().max()) < 1e-10, k
