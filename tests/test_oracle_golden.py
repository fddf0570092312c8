"""Pin the oracle (oracle/misa_oracle.py) against fixtures produced by the real reference
(oracle/gen_golden.py).  CPU only."""
import json
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, load_small, small_batch, small_cfg, state_from_npz, max_rel
from oracle.misa_oracle import (OracleMISA, oracle_build, oracle_losses, oracle_optimizer,
                                oracle_step)


@pytest.mark.parametrize("name", ["small_ragged", "small_shuffled_confid", "small_adversarial", "small_gru"])
def test_small_fixture_full_tensors(name):
    z, meta = load_small(name)
    cfg = small_cfg(meta)
    model = OracleMISA(cfg)
    model.load_state_dict(state_from_npz(z), strict=True)
    model.eval()
    batch = small_batch(z)
    opt = oracle_optimizer(model, cfg)
    out, L, grads = oracle_step(model, batch, cfg, opt)
    for k in ("cls", "diff", "recon", "sim", "conf", "total"):
        assert abs(float(L[k].detach()) - float(z["loss/" + k])) <= 1e-6 * max(1.0, abs(float(z["loss/" + k]))), k
    np.testing.assert_allclose(out["scores"].detach().numpy(), z["out/scores"], rtol=0, atol=1e-6)
    np.testing.assert_array_equal(out["labels"].numpy(), z["out/labels"])
    for a in ("utt_t_orig", "utt_private_a", "utt_shared_v", "utt_a_recon", "tcp",
              "shared_or_private_s") + (() if meta.get("use_cmd_sim", True) else ("domain_label_v",)):
        np.testing.assert_allclose(out[a].detach().numpy(), z["out/" + a], rtol=0, atol=1e-6)
    none = set(meta["none_grads"])
    # the same clip + Adam step taken from the reference's own gradients
    twin = OracleMISA(cfg)
    twin.load_state_dict(state_from_npz(z), strict=True)
    for n, p in twin.named_parameters():
        p.grad = None if n in none else torch.from_numpy(z["grad/" + n]).to(p.dtype)
    torch.nn.utils.clip_grad_value_([p for p in twin.parameters() if p.requires_grad], cfg.clip)
    oracle_optimizer(twin, cfg).step()
    twin = dict(twin.named_parameters())
    for n, p in model.named_parameters():
        after = torch.from_numpy(z["after/" + n])
        settled = torch.ones(after.shape, dtype=torch.bool)
        if n in none:
            assert grads[n] is None, n
        else:
            g = torch.from_numpy(z["grad/" + n])
            assert max_rel(grads[n], g) < 1e-5, n
            settled = g.abs() > 1e-5 * g.abs().max()
        # after one clip+Adam step.  Adam's first step moves an element by lr * g / (|g| + eps), so
        # where g is within the gradient check's tolerance of zero (the attention key bias has an
        # exactly zero gradient) the step follows the summation order of the CPU and its thread
        # count: there it is checked from the reference's gradients only.
        assert max_rel(twin[n].detach(), after) < 1e-6, n
        err = (p.detach() - after).abs()[settled]
        assert err.numel() == 0 or float(err.max() / (after.abs().max() + 1e-30)) < 1e-6, n


def test_same_seed_same_weights_as_reference():
    """oracle_build must consume the RNG exactly like MISA.__init__ + Solver.build, so the
    full-size summaries (which store seeds, not tensors) are reproducible."""
    from mmda_b200.config import mosi_config
    rec = json.load(open(os.path.join(GOLDEN, "c1_mosi_b64.json")))
    model = oracle_build(mosi_config(vocab_size=2000), rec["seed"])
    for n, p in model.named_parameters():
        s = p.detach().double()
        ref = rec["param0"][n]
        assert abs(float(s.sum()) - ref[0]) <= 1e-6 * max(1.0, ref[1]), n
        assert abs(float(s.norm()) - ref[2]) <= 1e-6 * max(1.0, ref[2]), n


@pytest.mark.parametrize("name,cfgname,kw,lengths", [
    ("c1_mosi_b64", "mosi", {}, "ragged"),
])
def test_full_size_summary(name, cfgname, kw, lengths):
    from mmda_b200 import config as C
    from mmda_b200.synthetic import batch_for
    rec = json.load(open(os.path.join(GOLDEN, name + ".json")))
    cfg = getattr(C, cfgname + "_config")(vocab_size=2000, **kw)
    model = oracle_build(cfg, rec["seed"]).eval()
    opt = oracle_optimizer(model, cfg)
    for it, st in enumerate(rec["steps"]):
        batch = batch_for(cfg, seed=rec["batch_seed"] + it, lengths=lengths)
        out, L, grads = oracle_step(model, batch, cfg, opt)
        for k, v in st["losses"].items():
            assert abs(float(L[k].detach()) - v) <= 2e-6 * max(1.0, abs(v)), (it, k)
        assert max_rel(out["scores"].detach(), st["scores"]) < 1e-5
        for n, p in model.named_parameters():
            g = st["grads"][n]
            if g is None:
                assert grads[n] is None, n
            else:
                assert abs(float(grads[n].double().norm()) - g[2]) <= 1e-4 * max(g[2], 1e-12), n


# ---- collate (SURVEY.md 8f N3): oracle restatement vs the reference's own collate_fn -----------
def test_collate_oracle_matches_reference_collate_fn():
    from oracle.collate_oracle import collate, make_samples, wordpieces
    z = np.load(os.path.join(GOLDEN, "collate_small.npz"), allow_pickle=False)
    meta = json.loads(bytes(z["meta"]).decode())
    samples = make_samples(meta["n"], meta["dv"], meta["da"], seed=meta["seed"])
    for bi in range(3):
        idx = z[f"b{bi}/index"]
        out = collate([samples[i] for i in idx], wp_ids=lambda s: wordpieces(s[0][3]))
        for k in ("sentences", "visual", "acoustic", "labels", "emo_labels", "lengths",
                  "bert_sentences", "bert_sentence_types", "bert_sentence_att_mask"):
            ref = z[f"b{bi}/{k}"]
            assert out[k].shape == ref.shape and out[k].dtype == ref.dtype, (bi, k, out[k].dtype, ref.dtype)
            assert np.array_equal(out[k], ref, equal_nan=True), (bi, k)
        assert list(z[f"b{bi}/ids"]) == out["ids"]


def test_collate_host_side_sort_flatten_and_errors():
    from mmda_b200.collate import DeviceDataset, flatten_split
    from oracle.collate_oracle import collate, make_samples
    samples = make_samples(40, 3, 4, seed=5)
    flat = flatten_split(samples)
    assert flat["offsets"][-1] == flat["words"].shape[0] == flat["visual"].shape[0]
    ds = DeviceDataset(samples, device="cpu")        # host logic only; collate() needs the GPU
    idx = [7, 3, 11, 30, 2, 19, 5, 8, 21]
    order = ds.sort_batch(idx)
    ref = collate([samples[i] for i in idx])
    assert [samples[i][2] for i in order] == ref["ids"]          # same stable descending sort
    assert np.array_equal(ds.lengths[order], ref["lengths"])
    with pytest.raises(ValueError):
        ds.sort_batch([])
    with pytest.raises(IndexError):
        ds.sort_batch([0, 40])
    mosi_like = [((s[0][0], s[0][1], s[0][2], s[0][3]), s[1][:, :1], s[2]) for s in samples]
    with pytest.raises(TypeError):
        DeviceDataset(mosi_like, device="cpu").collate([0, 1])
    with pytest.raises(TypeError):
        collate(mosi_like[:2])
