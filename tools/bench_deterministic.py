"""ms/step of the fused (graph-replayed) training step with torch.use_deterministic_algorithms off
and on, alternated in one process so both modes see the same card state.  Prints one JSON line
with the card name and power limit beside the numbers.

    python tools/bench_deterministic.py [--steps 50] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:       # no nvidia-smi: record that, the timings stand on their own
        return "unknown"


def time_steps(tr, batches, steps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(steps):
        b = batches[i % len(batches)]
        tr.step(*b)
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_deterministic needs a GPU")
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer
    res = {"card": card()}
    for name, lengths, kw, steps in (("c2_full", "full", {}, a.steps), ("c2_ragged", "ragged", {}, a.steps),
                                     ("c4_bert_bf16", "ragged", {"use_bert": True, "precision": "bf16",
                                                                 "batch_size": 512}, max(4, a.steps // 10))):
        cfg = mosei_config(vocab_size=2000, use_confidNet=True, **kw)
        bs = [batch_for(cfg, seed=80 + i, lengths=lengths) for i in range(4)]
        bs = [(b.sentences.cuda(), b.visual.cuda(), b.acoustic.cuda(), b.lengths, b.labels.cuda())
              + ((b.bert_sent.cuda(), b.bert_sent_type.cuda(), b.bert_sent_mask.cuda())
                 if cfg.use_bert else ()) for b in bs]
        torch.manual_seed(0)
        tr = FusedTrainer(MISA(cfg).cuda().train())
        times = {False: [], True: []}
        for flag in (False, True):          # warm-up: every graph of both modes captured
            torch.use_deterministic_algorithms(flag)
            time_steps(tr, bs, 3 * len(bs))
        for _ in range(a.rounds):
            for flag in (False, True):
                torch.use_deterministic_algorithms(flag)
                times[flag].append(time_steps(tr, bs, steps))
        torch.use_deterministic_algorithms(False)
        res[name] = {"off_ms": [round(t, 4) for t in times[False]],
                     "on_ms": [round(t, 4) for t in times[True]]}
        tr.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
