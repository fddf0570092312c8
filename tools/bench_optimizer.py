"""The optimizer step on the device, at the C2 shape (MOSEI 300/35/74-d, vocab 20000, batch 256,
seq 50, full lengths, train mode):

1. CUDA-event times of mmda_adam_clip_step and mmda_rmsprop_clip_step over the C2 trainer's active
   parameter arena, with a 256 MiB memset between launches (the Adam arenas, 4 x n floats, would
   otherwise stay in the 126 MB L2).  Achieved bandwidth counts the bytes the algorithm moves:
   28 B per parameter for Adam (p, g, m, v read; p, m, v written), 20 B for RMSprop (p, g, v read;
   p, v written).  It is reported against the data-sheet HBM bandwidth and against a device-to-device
   copy of 1 GiB measured in the same run.
2. ms per fused C2 step with a learning rate that changes every step (linear warm-up), for eager
   launches (use_graph=False: what a changing rate cost before the rate lived on the device) and
   for CUDA-graph replay, alternated over several rounds in the same process.

Prints one JSON line per result; the first names the GPU and its power limit.

    python tools/bench_optimizer.py [--iters 50] [--steps 30] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_DATASHEET_GBS = 7700.0      # HGX B200 data sheet, one GPU, at up to 1000 W


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30)
        power = r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"gpu": name, "power_limit,max_sm_clock": power}


def c2_trainer(use_graph, optimizer="Adam"):
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.trainer import FusedTrainer
    cfg = mosei_config(vocab_size=20000, batch_size=256, optimizer=optimizer)
    torch.manual_seed(1234)
    model = MISA(cfg)
    for n, p in model.named_parameters():
        if "weight_hh" in n:
            torch.nn.init.orthogonal_(p)
    return cfg, FusedTrainer(model.to("cuda").train(), use_graph=use_graph)


def kernel_times(n, iters, flush):
    from mmda_b200.engine import Kernels, _ptr
    k = Kernels(); k.bind_stream()
    g = torch.Generator(device="cuda").manual_seed(0)
    p = torch.randn(n, device="cuda", generator=g) * 0.1
    gr = torch.randn(n, device="cuda", generator=g)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    st = torch.zeros(5, dtype=torch.float64, device="cuda")
    k._c("mmda_step_state_init", _ptr(st), 0, 0.9, 0.999)
    k._c("mmda_step_state_set_lr", _ptr(st), 1e-4)
    calls = {
        "adam": (28, lambda: k._c("mmda_adam_clip_step", _ptr(p), _ptr(gr), _ptr(m), _ptr(v), n, 1,
                                  1e-4, 1.0, 0.9, 0.999, 1e-8, 1.0, _ptr(st))),
        "rmsprop": (20, lambda: k._c("mmda_rmsprop_clip_step", _ptr(p), _ptr(gr), _ptr(v), n, 1e-4,
                                     1.0, 0.99, 1e-8, 1.0, _ptr(st))),
    }
    times = {name: [] for name in calls}
    for name, (_, fn) in calls.items():        # warm-up (module load)
        fn()
    torch.cuda.synchronize()
    for _ in range(iters):
        for name, (_, fn) in calls.items():    # alternated, each after an L2 flush
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            times[name].append((e0, e1))
    torch.cuda.synchronize()
    # device-to-device copy of 1 GiB: 2 GiB moved, the achievable HBM rate for a plain stream
    src = torch.empty(1 << 28, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    cp = []
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); dst.copy_(src); e1.record()
        cp.append((e0, e1))
    torch.cuda.synchronize()
    copy_ms = sorted(a.elapsed_time(b) for a, b in cp)[len(cp) // 2]
    copy_gbs = 2 * src.numel() * 4 / (copy_ms * 1e-3) / 1e9
    del src, dst
    out = []
    for name, (bpp, _) in calls.items():
        ts = sorted(a.elapsed_time(b) for a, b in times[name])
        med = ts[len(ts) // 2]
        gbs = bpp * n / (med * 1e-3) / 1e9
        out.append({"kernel": f"mmda_{name}_clip_step", "n_params": n, "bytes_per_param": bpp,
                    "iters": iters, "median_us": med * 1e3, "min_us": ts[0] * 1e3,
                    "achieved_gbs": gbs, "frac_of_datasheet_hbm": gbs / HBM_DATASHEET_GBS,
                    "datasheet_hbm_gbs": HBM_DATASHEET_GBS, "d2d_copy_gbs_same_run": copy_gbs,
                    "frac_of_d2d_copy": gbs / copy_gbs, "l2": "256 MiB memset before every launch"})
    return out


def schedule_steps(rounds, steps, flush):
    from mmda_b200.synthetic import batch_for
    trainers = {}
    for mode in (False, True):
        cfg, tr = c2_trainer(mode)
        trainers[mode] = tr
    batches = [batch_for(cfg, seed=1234 + i, lengths="full", seq_len=50) for i in range(4)]
    dev = [(b.sentences.cuda(), b.visual.cuda(), b.acoustic.cuda(), b.lengths, b.labels.cuda())
           for b in batches]
    base, count = cfg.learning_rate, {False: 0, True: 0}

    def run(mode, n):
        tr = trainers[mode]
        for _ in range(n):
            i = count[mode]
            tr.lr = base * min(1.0, (i % 1000 + 1) / 1000.0)      # a new rate every step
            count[mode] += 1
            flush.zero_()
            tr.step(*dev[i % 4])
    for mode in (False, True):
        run(mode, 6)                          # warm-up, includes the one capture
    torch.cuda.synchronize()
    out = []
    for r in range(rounds):
        for mode in (False, True):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            h0 = time.perf_counter()
            run(mode, steps)
            host_ms = 1e3 * (time.perf_counter() - h0) / steps
            e1.record()
            torch.cuda.synchronize()
            tr = trainers[mode]
            out.append({"step": "C2 fused step, lr changes every step", "round": r,
                        "path": "graph replay" if mode else "eager (use_graph=False)",
                        "ms_per_step": e0.elapsed_time(e1) / steps, "host_enqueue_ms_per_step": host_ms,
                        "steps": steps, "step_graphs": len(tr._graphs),
                        "l2": "256 MiB memset between steps inside the timed region"})
    for tr in trainers.values():
        tr.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_optimizer.py measures on the GPU; none is visible")
    print(json.dumps(gpu_info()), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    _, tr = c2_trainer(False)
    n = tr.n_active
    del tr
    for row in kernel_times(n, a.iters, flush):
        print(json.dumps(row), flush=True)
    for row in schedule_steps(a.rounds, a.steps, flush):
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
