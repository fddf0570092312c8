"""Tensor-core recurrence (csrc/lstm_tc.cu) through the C ABI against an fp64 restatement of
nn.LSTM's recurrent half (reference src/models.py:48-55,167,176; oracle/explicit.py semantics) on
the packed layout: hidden / cell states, saved gate activations, final states in original batch
order, and the BPTT output d(pre-activation gates).  Tolerance: 1e-5 scale-relative (fp32 mode)."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
TOL = 1e-5


@pytest.mark.parametrize("B,H,T,ragged", [(40, 300, 6, 1), (256, 300, 50, 0), (64, 300, 30, 1),
                                          (100, 200, 20, 1), (300, 300, 12, 1), (7, 160, 9, 1),
                                          (37, 129, 7, 1), (50, 320, 9, 1), (1, 300, 1, 0)])
def test_tc_recurrence_vs_fp64(B, H, T, ragged):
    import dev_lstm_tc as D
    dev = torch.device("cuda:0")
    c = D.make_case(B, H, T, ragged, dev, seed=B + H)
    y64, c64, a64, u64 = D.ref64(c)
    dG64 = D.ref64_bwd(c, a64, c64)
    o = D.run(c, "tc")
    assert o["err_fwd"] == 0 and o["err_bwd"] == 0, "a recurrence CTA gave up waiting for its peers"
    errs = {k: D.rel(o[k], r) for k, r in (("y", y64), ("c", c64), ("act", a64), ("utt", u64), ("dG", dG64))}
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, f"parity_lstm_tc_{B}_{H}_{T}_{ragged}.txt"), "w") as f:
        f.write("\n".join(f"{k} {v:.3e}" for k, v in errs.items()) + "\n")
    bad = {k: v for k, v in errs.items() if not v <= TOL}
    assert not bad, bad
    # same inputs, same launch twice: the accumulation order is fixed, so the bits are too
    o2 = D.run(c, "tc")
    for k in ("y", "c", "act", "utt", "dG"):
        assert torch.equal(o[k], o2[k]), f"{k} differs between two identical launches"


def test_tc_plan_and_unsupported_sizes():
    import ctypes
    from mmda_b200._lib import LIB
    arr = (ctypes.c_int * 8)()
    LIB.call("mmda_lstm_tc_plan", 256, 300, 50, arr)
    S, G, BT, NT, Kp, smf, smb, ctas = list(arr)
    assert S == 10 and Kp == 304 and BT * NT >= 256 and BT <= 64 and ctas == 2 * S * G <= 148
    assert max(smf, smb) <= 232448
    assert LIB.raw("mmda_lstm_tc_workspace_bytes")(256, 74, 50) == -1      # small H: SIMT kernels
    assert LIB.raw("mmda_lstm_tc_workspace_bytes")(256, 400, 50) == -1
