"""ms per fused training step at the C2 shape (MOSEI 300/35/74-d, vocab 20000, batch 256, seq 50,
full lengths, train mode with dropout, CUDA-graph replay) for every ``config.activation`` the
build supports.  ELU / Hardshrink / Hardtanh ride the fused GEMM epilogue like LeakyReLU; RReLU in
training draws its slopes in an in-place pass after an epilogue-free linear (one forward and one
backward launch per project_m), so its line shows what those launches cost.

The activations are alternated over several rounds in one process, with a 256 MiB memset between
steps inside the timed region (as bench.py).  Prints one JSON line per (round, activation), then a
median per activation; the first line names the GPU and its power limit.

    python tools/bench_activations.py [--steps 50] [--rounds 5]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_optimizer import gpu_info  # noqa: E402


def c2_trainer(activation):
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=20000, batch_size=256, activation=activation)
    torch.manual_seed(1234)
    model = MISA(cfg)
    for n, p in model.named_parameters():
        if "weight_hh" in n:
            torch.nn.init.orthogonal_(p)
    return cfg, FusedTrainer(model.to("cuda").train())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_activations.py measures on the GPU; none is visible")
    from mmda_b200.config import ACTIVATIONS
    from mmda_b200.synthetic import batch_for
    print(json.dumps(gpu_info()), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    names = [n for n in ACTIVATIONS if n != "none"]
    trainers = {}
    for name in names:
        cfg, trainers[name] = c2_trainer(name)
    batches = [batch_for(cfg, seed=1234 + i, lengths="full", seq_len=50) for i in range(4)]
    dev = [(b.sentences.cuda(), b.visual.cuda(), b.acoustic.cuda(), b.lengths, b.labels.cuda())
           for b in batches]
    for name in names:                      # warm-up, includes the one capture per trainer
        for i in range(6):
            trainers[name].step(*dev[i % 4])
    torch.cuda.synchronize()
    times = {name: [] for name in names}
    for r in range(a.rounds):
        for name in names:
            tr = trainers[name]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(a.steps):
                flush.zero_()
                tr.step(*dev[i % 4])
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.steps
            times[name].append(ms)
            print(json.dumps({"step": "C2 fused step, train mode", "activation": name, "round": r,
                              "ms_per_step": ms, "steps": a.steps, "step_graphs": len(tr._graphs),
                              "launches_per_step": tr.launches_per_step,
                              "l2": "256 MiB memset between steps inside the timed region"}), flush=True)
    for name in names:
        ts = sorted(times[name])
        print(json.dumps({"activation": name, "median_ms_per_step": ts[len(ts) // 2],
                          "min_ms_per_step": ts[0], "max_ms_per_step": ts[-1],
                          "rounds": a.rounds}), flush=True)
    for tr in trainers.values():
        tr.close()


if __name__ == "__main__":
    main()
