"""BERT self-attention core at long sequences: CUDA-event times of the tiled kernels
(mmda_bert_attention_{forward,backward}_tiled[_mma]) at B = 64, S in {128, 256, 512}, with the
resident kernels at S = 52 / 84 for context and eager torch scaled_dot_product_attention on the
same shapes and dtypes (informational), then the peak device memory of one fused C4-style training
step (BERT + LSTM v/a, layers 0-8 frozen) at the same sequence lengths, each in its own process.

FLOP counts are derived from shapes, per (sample, head) with d = 64:
  forward   4 S^2 d   (Q K^T and P V)
  backward as issued: the dK/dV kernel recomputes Q K^T and d(P) = dO V^T and runs dV, dK
                      (8 S^2 d); the dQ kernel recomputes both again and runs dQ (6 S^2 d): 14 S^2 d
                      in fp32 mode.  In bf16 mode the dQ kernel makes a first pass over the keys
                      (Q K^T, dO V^T: 4 S^2 d) for D = rowsum(dP o P): 18 S^2 d.  The resident
                      backward issues 6 S^2 d (no recompute).
Inputs (qkv at B = 64, S = 512: 302 MB) exceed the 126 MB L2 from S = 256 on; at S <= 128 the
working set can stay L2-resident across iterations.

    python tools/bench_bert_attention.py [--batch 64] [--seqs 128,256,512] [--iters 20]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30)
        power = r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"gpu": name, "power_limit,max_sm_clock": power}


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernels(a, dev):
    from mmda_b200.engine import Kernels, _ptr
    k = Kernels(); k.bind_stream()
    B, nh, d, p = a.batch, 12, 64, 0.1
    rows = []
    cases = [(S, "tiled") for S in a.seqs] + [(52, "resident"), (84, "resident")]
    for S, kind in cases:
        g = torch.Generator().manual_seed(S)
        qkv = torch.randn(B * S, 3 * nh * d, generator=g).to(dev)
        mask = torch.ones(B, S, dtype=torch.int64, device=dev)
        do = torch.randn(B * S, nh * d, generator=g).to(dev)
        ctx = torch.empty(B * S, nh * d, device=dev)
        dqkv = torch.empty_like(qkv)
        lse = torch.empty(B, nh, S, device=dev)
        delta = torch.empty(B, nh, S, device=dev)
        ctx_bf = torch.empty(B * S, nh * d, device=dev, dtype=torch.bfloat16)
        dq_bf = torch.empty(B * S, 3 * nh * d, device=dev, dtype=torch.bfloat16)
        probs = torch.empty(B, nh, S, S, device=dev) if kind == "resident" else None
        for mode in ("fp32", "bf16"):
            if kind == "tiled" and mode == "fp32":
                fwd = lambda: k._c("mmda_bert_attention_forward_tiled", _ptr(qkv), _ptr(mask), _ptr(ctx),
                                   _ptr(lse), B, S, nh, d, p, 1, None, 201)
                bwd = lambda: k._c("mmda_bert_attention_backward_tiled", _ptr(qkv), _ptr(mask), _ptr(ctx),
                                   _ptr(lse), _ptr(do), _ptr(delta), _ptr(dqkv), B, S, nh, d, p, 1, None, 201)
            elif kind == "tiled":
                fwd = lambda: k._c("mmda_bert_attention_forward_tiled_mma", _ptr(qkv), _ptr(mask), _ptr(ctx),
                                   _ptr(ctx_bf), _ptr(lse), B, S, nh, d, p, 1, None, 201)
                bwd = lambda: k._c("mmda_bert_attention_backward_tiled_mma", _ptr(qkv), _ptr(mask),
                                   _ptr(ctx), _ptr(lse), _ptr(do), _ptr(delta), None, _ptr(dq_bf),
                                   B, S, nh, d, p, 1, None, 201)
            elif mode == "fp32":
                fwd = lambda: k._c("mmda_bert_attention_forward", _ptr(qkv), _ptr(mask), _ptr(ctx),
                                   _ptr(probs), B, S, nh, d, p, 1, None, 201)
                bwd = lambda: k._c("mmda_bert_attention_backward", _ptr(qkv), _ptr(probs), _ptr(do),
                                   _ptr(dqkv), B, S, nh, d, p, 1, None, 201)
            elif S <= 64:
                fwd = lambda: k._c("mmda_bert_attention_forward_mma", _ptr(qkv), _ptr(mask), _ptr(ctx),
                                   _ptr(ctx_bf), _ptr(probs), B, S, nh, d, p, 1, None, 201)
                bwd = lambda: k._c("mmda_bert_attention_backward_mma", _ptr(qkv), _ptr(probs), _ptr(do),
                                   None, _ptr(dq_bf), B, S, nh, d, p, 1, None, 201)
            else:
                continue          # bf16 mode runs the fp32 resident pair at 65..84
            fwd()
            tf = timed(fwd, a.iters)
            tb = timed(bwd, a.iters)
            heads = B * nh
            ff = 4 * S * S * d * heads
            fb = ((14 if mode == "fp32" else 18) if kind == "tiled" else 6) * S * S * d * heads
            rows.append({"kernel": f"{kind} {mode}", "B": B, "S": S, "fwd_ms": round(tf, 4),
                         "bwd_ms": round(tb, 4), "fwd_tflops": round(ff / tf / 1e9, 2),
                         "bwd_tflops_issued": round(fb / tb / 1e9, 2)})
            print(json.dumps(rows[-1]), flush=True)
        # eager torch SDPA on the same shapes (informational; dropout 0.1 as in training)
        for dt in (torch.float32, torch.bfloat16):
            q, kk, v = (qkv.view(B, S, 3, nh, d)[:, :, j].transpose(1, 2).to(dt).contiguous().requires_grad_(True)
                        for j in range(3))
            g_o = do.view(B, S, nh, d).transpose(1, 2).to(dt).contiguous()
            sd = lambda: torch.nn.functional.scaled_dot_product_attention(q, kk, v, dropout_p=p)
            tf = timed(lambda: sd(), a.iters)
            tfb = timed(lambda: torch.autograd.grad(sd(), (q, kk, v), g_o), a.iters)
            rows.append({"kernel": f"torch sdpa eager {str(dt)[6:]}", "B": B, "S": S, "fwd_ms": round(tf, 4),
                         "fwd_bwd_ms": round(tfb, 4)})
            print(json.dumps(rows[-1]), flush=True)
        del qkv, do, ctx, dqkv, probs
        torch.cuda.empty_cache()
    return rows


def step_memory_one(batch, precision, S, dev):
    """max_memory_allocated of one fused training step (run in a fresh process per case)"""
    from mmda_b200 import MISA, FusedTrainer, mosei_config
    from mmda_b200.synthetic import batch_for
    cfg = mosei_config(vocab_size=20000, batch_size=batch, use_bert=True, precision=precision)
    torch.manual_seed(1234)
    model = MISA(cfg)
    for n, p in model.named_parameters():
        if "bertmodel.encoder.layer" in n and int(n.split("encoder.layer.")[-1].split(".")[0]) <= 8:
            p.requires_grad = False
    model = model.to(dev).train()
    tr = FusedTrainer(model)
    b = batch_for(cfg, seed=1, lengths="full", seq_len=S - 2)
    args = [t.to(dev) for t in (b.sentences, b.visual, b.acoustic)] + [b.lengths, b.labels.to(dev)] + \
           [t.to(dev) for t in (b.bert_sent, b.bert_sent_type, b.bert_sent_mask)]
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    L = tr.step(*args)
    torch.cuda.synchronize()
    print(json.dumps({"step": f"C4-style fused step {precision}", "B": batch, "S": S,
                      "max_memory_allocated_gb": round(torch.cuda.max_memory_allocated() / 2**30, 3),
                      "probs_buffers": sum(1 for n in tr.eng.ws if n.startswith("bert_probs_")),
                      "loss_finite": bool(torch.isfinite(L[:6]).all())}), flush=True)


def step_memory(a):
    for precision in ("fp32", "bf16"):
        for S in a.seqs:
            subprocess.run([sys.executable, os.path.abspath(__file__), "--step-one", precision, str(S),
                            "--batch", str(a.batch)], check=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--seqs", default="128,256,512")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--no-step", action="store_true", help="skip the fused-step memory rows")
    ap.add_argument("--step-one", nargs=2, metavar=("PRECISION", "S"), help=argparse.SUPPRESS)
    a = ap.parse_args()
    a.seqs = [int(s) for s in a.seqs.split(",")]
    if not torch.cuda.is_available():
        sys.exit("bench_bert_attention.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    if a.step_one:
        step_memory_one(a.batch, a.step_one[0], int(a.step_one[1]), dev)
        return
    print(json.dumps(gpu_info()), flush=True)
    kernels(a, dev)
    if not a.no_step:
        step_memory(a)


if __name__ == "__main__":
    main()
