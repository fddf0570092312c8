#!/usr/bin/env python
"""Benchmark of the MISA training step (BASELINE.json metric: MOSEI-shape train samples/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of solver.py:139-186 (zero_grad, forward, six losses, backward, clip, Adam)
over one synthetic MOSEI-shaped batch (configs[1]: 300/35/74-d, seq 50, batch 256 per GPU, train
mode with dropout).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEQ, BATCH, VOCAB = 50, 256, 20000     # BASELINE configs[1]; --seq / --batch override (configs[4] sweep)
METRIC, UNIT = "train_samples_per_sec", "samples/s"
DUMP_SAMPLE = 4 << 20                  # --dump-outputs: elements kept of the parameters / gradients


def workload(batch, lengths):
    """One string for both arms (the driver compares the arms' `config`)."""
    return (f"MOSEI-shape synthetic (BASELINE configs[1]): 300/35/74-d, seq {SEQ}, batch {batch}/GPU, "
            f"vocab {VOCAB}, lengths={lengths}, train mode (dropout on), fused step: fwd + 6 losses + "
            "bwd + clip + Adam")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], "measured (MEASURED_PEAKS.json)", d
    return 6650.0, "fallback (B200_PROFILING.md)", {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx, self.first = [], None, gpu_index, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def wait_first(self, timeout_s=4.0):
        """Block until nvidia-smi has delivered its first sample (its start-up takes 0.1-0.5 s,
        longer than a 20-step timed region), so that the following samples fall INSIDE the timed
        regions.  Gives up quietly after ``timeout_s``."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout_s:
            time.sleep(0.01)

    def mark(self):
        """Samples from here on were taken under load (call right before the timed region)."""
        self.first = len(self.rows)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if len(self.rows) <= self.first:
            time.sleep(0.15)          # very short run: take the next sample, right behind the region
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = self.rows[self.first:] or self.rows
        for r in rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for nm, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return dist, dist.group.WORLD, rank, local, world
    return None, None, 0, 0, 1


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's PyTorch CPU path, all host threads
# ------------------------------------------------------------------------------------------
def cpu_steps(steps, warmup, budget_s=150.0, batch=BATCH, lengths="full"):
    """The oracle port of the reference's PyTorch CPU path on all host threads, on the SAME batch
    size as the GPU arm.  A slow host shortens the sample (fewer steps), never the workload."""
    from mmda_b200.config import mosei_config
    from mmda_b200.synthetic import batch_for
    from oracle.misa_oracle import oracle_build, oracle_optimizer, oracle_step
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = mosei_config(vocab_size=VOCAB, batch_size=batch)
    model = oracle_build(cfg, 1234).train()
    opt = oracle_optimizer(model, cfg)
    b = batch_for(cfg, seed=1234, lengths=lengths, seq_len=SEQ)
    t0 = time.perf_counter()
    oracle_step(model, b, cfg, opt)              # first step = warm-up no. 1
    first = time.perf_counter() - t0
    want = steps
    if first * (steps + warmup) > budget_s:
        warmup = 1
        steps = max(1, int(budget_s / max(first, 1e-9)) - 1)
    for _ in range(max(0, warmup - 1)):
        oracle_step(model, b, cfg, opt)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        oracle_step(model, b, cfg, opt)
        ts.append(time.perf_counter() - t0)
    tot = sum(ts)
    sample = f"{steps} steps of the batch-{batch} seq-{SEQ} step after {max(1, warmup)} warm-up"
    if steps != want:
        sample += f" ({want} requested; shortened to fit {budget_s:.0f} s of CPU time)"
    return {"value": batch * steps / tot, "unit": UNIT, "cores": torch.get_num_threads(),
            "kind": "port", "sample": sample, "ms_per_step": 1e3 * tot / steps, "batch": batch,
            "steps": steps}


def run_reference(args, rank):
    if rank != 0:
        return
    cb = cpu_steps(args.steps, args.warmup, budget_s=float("inf"), batch=args.batch, lengths=args.lengths)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT,
            "n_gpus": args.gpus, "steps": cb["steps"], "warmup": args.warmup,
            "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload(args.batch, args.lengths),
                       "global_batch": args.batch, "parallelism": "cpu",
                       "note": "reference PyTorch CPU path via the oracle port (the Python reference "
                               "cannot travel to the GPU box); one process, all host threads"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def roofline_block(cfg, batch0, kdur, clk, args):
    """Roofline of the text-encoder recurrence launch that takes longest (forward or BPTT).
    Everything is derived from the live plan and the live timing; DRAM traffic comes from the
    committed ncu capture when one exists for this exact shape (else null)."""
    import ctypes
    from mmda_b200._lib import LIB
    timed = {k: v for k, v in kdur.items() if v}
    if not timed:
        return None
    kname = max(timed, key=timed.get)
    tc = "_tc_" in kname
    bwd = kname.endswith("backward")
    H = cfg.embedding_size
    ntok = int(batch0.lengths.sum())
    Tmax = int(batch0.lengths.max())
    dur = timed[kname] * 1e-3
    peak, peak_src, pk = peaks()
    sm_hz = ((clk or {}).get("sm_mhz") or 1965.0) * 1e6
    fma_peak = 148 * 128 * 2 * sm_hz / 1e12
    tensor_peak = pk.get("bf16_tflops_sustained", 1403.9)
    alg_bytes = 2 * 10 * H * 4 * ntok              # both directions, 10H fp32 words per token (M3)
    flops = 2 * 2 * 4 * H * H * ntok               # recurrent MACs * 2, both directions (M3)
    bounds_us = {"hbm": alg_bytes / (peak * 1e9) * 1e6, "fp32_fma": flops / (fma_peak * 1e12) * 1e6}
    plan = {}
    if tc:
        arr = (ctypes.c_int * 8)()
        LIB.call("mmda_lstm_tc_plan_select", int(bwd))
        LIB.call("mmda_lstm_tc_plan", args.batch, H, Tmax, arr)
        LIB.call("mmda_lstm_tc_plan_select", 0)
        plan = dict(zip(("slices", "groups", "batch_tile", "tiles", "units_per_cta" if bwd else "k_padded",
                         "smem_fwd", "smem_bwd", "ctas"), list(arr)))
        terms = 3                                  # two fp16 terms per operand: 3 MMAs per product
        issued = flops * terms
        bounds_us["tensor"] = issued / (tensor_peak * 1e12) * 1e6
    else:
        arr = (ctypes.c_int * 6)()
        LIB.call("mmda_lstm_plan", args.batch, H, arr)
        plan = dict(zip(("cluster", "units_per_cta", "batch_tile", "tiles", "smem_fwd", "smem_bwd"), list(arr)))
        plan["ctas"] = 2 * plan["cluster"] * plan["tiles"]
        warps = (plan["units_per_cta"] + 7) // 8 * (plan["batch_tile"] // 8)
        lds = 1536.0 * ((H + 3) // 4) * warps * plan["ctas"] * Tmax   # operand bytes smem -> registers
        bounds_us["smem"] = lds / (148 * 128 * sm_hz) * 1e6
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        key = f"{kname}:B{args.batch}:T{Tmax}:H{H}:{args.lengths}"
        ent = json.load(open(tp)).get(key)
        if ent:
            traffic, traffic_src = ent["dram_bytes"], ent["source"]
    # The roofline this launch is reported against is SURVEY M2(ii)'s: the largest of the HBM,
    # shared-memory and fp32-FMA times of the ALGORITHMIC work (one product per MAC).  For the
    # tensor-core kernel the tensor-pipe time of the ISSUED work (3 MMAs per product) is listed
    # too; it is the smallest of the lot.
    m2 = max(bounds_us, key=bounds_us.get)
    top = {"hbm": ("hbm", alg_bytes / dur / 1e9, peak, "GB/s", peak_src),
           "fp32_fma": ("fp32_fma", flops / dur / 1e12, fma_peak, "TFLOP/s",
                        "148 SM x 128 FMA/clk x 2 x SM clock sampled during the timed region"),
           "tensor": ("tensor", flops / dur / 1e12, tensor_peak, "TFLOP/s",
                      "MEASURED_PEAKS.json bf16_tflops_sustained"),
           "smem": ("smem", None, None, None, None)}[m2]
    if m2 == "smem":      # SIMT kernel bound by operand delivery: report it against HBM as the contract asks
        top = ("hbm", alg_bytes / dur / 1e9, peak, "GB/s", peak_src)
    out = {"kernel": kname + f" (text encoder, H={H}, both directions, {ntok} tokens)",
           "bound": top[0], "achieved": top[1], "peak": top[2], "unit": top[3], "peak_source": top[4],
           "traffic": traffic, "traffic_source": traffic_src,
           "algorithmic_bytes": alg_bytes, "algorithmic_flops": flops,
           "launch_ms": timed[kname], "launch_ms_all": timed, "plan": plan,
           "roofline_time_us": bounds_us, "binding_roofline": m2,
           "frac_of_binding_roofline": bounds_us[m2] * 1e-6 / dur,
           "hbm": {"achieved_gbs": alg_bytes / dur / 1e9, "peak_gbs": peak,
                   "frac": alg_bytes / dur / 1e9 / peak, "peak_source": peak_src},
           "fp32_fma": {"achieved_tflops": flops / dur / 1e12, "peak_tflops": fma_peak,
                        "frac": flops / dur / 1e12 / fma_peak,
                        "peak_source": "148 SM x 128 FMA/clk x 2 x sampled SM clock"}}
    out["frac"] = out["achieved"] / out["peak"]
    if tc:
        out["tensor_issued"] = {"achieved_tflops": flops * terms / dur / 1e12, "peak_tflops": tensor_peak,
                                "frac": flops * terms / dur / 1e12 / tensor_peak,
                                "terms_per_product": terms}
        out["note"] = ("tensor-core recurrence: fp32-accurate operand splits (two fp16 terms per operand, 3 MMAs "
                       "per product); a time step is a serial chain of MMA -> cell update -> L2 exchange, so "
                       "the launch is latency-bound.  `bound`/`frac` are SURVEY M2(ii)'s roofline (the largest of the "
                       "HBM / fp32-FMA times of the algorithmic work: what the best fp32 SIMT kernel could do); "
                       "`tensor_issued` is the tensor pipe's share of its measured peak for the MMAs actually "
                       "issued and `hbm` the algorithmic bytes against the measured copy bandwidth -- both small, "
                       "because neither pipe is what a 50-step serial chain waits for")
    else:
        out["note"] = "SIMT recurrence: bound by shared-memory operand delivery and fp32 FMA issue, not HBM"
    return out


def dp_check(dist, pg, rank, world, dev):
    """Data-parallel parity evidence for the driver (the 2-GPU pytest is skipped on 1-GPU boxes):
    one eval-mode step of a small global batch sharded over all ranks vs the same batch on rank 0
    alone (kernel path) and vs the CPU oracle (losses)."""
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer, LOSS_NAMES
    per = 32
    cfg = mosei_config(vocab_size=500, batch_size=per * world, use_confidNet=True)
    full = batch_for(cfg, seed=77, lengths="ragged", seq_len=20)

    def make():
        torch.manual_seed(5)
        m = MISA(cfg)
        for n, p in m.named_parameters():
            if "weight_hh" in n:
                torch.nn.init.orthogonal_(p)
        return m

    def run(tr, b):
        L = tr.forward_backward(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths,
                                b.labels.to(dev))
        torch.cuda.synchronize()
        return L[:6].clone()

    tr_dp = FusedTrainer(make().to(dev).eval(), process_group=pg, use_graph=False)
    L_dp = run(tr_dp, full.slice(rank * per, (rank + 1) * per))
    out = None
    if rank == 0:
        tr_1 = FusedTrainer(make().to(dev).eval(), use_graph=False)
        L_1 = run(tr_1, full)
        na = tr_1.n_active
        g1, gd = tr_1.g_arena[:na], tr_dp.g_arena[:na]
        out = {"global_batch": per * world, "ranks": world,
               "loss_max_rel_vs_single_gpu": float(((L_dp - L_1).abs() / L_1.abs().clamp_min(1e-6)).max()),
               "grad_max_err_over_max_vs_single_gpu": float((gd - g1).abs().max() / g1.abs().max()),
               "grad_norm_dp": float(gd.norm()), "grad_norm_single_gpu": float(g1.norm())}
        try:
            from oracle.misa_oracle import OracleMISA, oracle_step
            ref = OracleMISA(cfg)
            ref.load_state_dict({k: v.detach().cpu() for k, v in make().state_dict().items()})
            ref.eval()
            _, L, grads = oracle_step(ref, full, cfg, None)
            lo = torch.tensor([float(L[k]) for k in LOSS_NAMES[:6]])
            out["loss_max_rel_vs_cpu_oracle"] = float(((L_dp.cpu() - lo).abs() / lo.abs().clamp_min(1e-6)).max())
            gn = torch.sqrt(sum((g.double() ** 2).sum() for g in grads.values() if g is not None))
            out["grad_norm_cpu_oracle"] = float(gn)
        except Exception as e:      # the oracle is a checker: report, do not fail the bench
            out["oracle_error"] = repr(e)[:200]
    tr_dp.close()
    return out


def dump_outputs(out_dir, tr, losses):
    """Write what one step computed as float32 ``out_dir/<name>.npy``, so that two builds can be
    compared output for output: ``losses`` (the vector ``FusedTrainer.step`` returns), and the
    updated ``params`` and their ``grads``, each flattened in ``named_parameters()`` order (not the
    arena layout, which may change) and sampled at DUMP_SAMPLE fixed, seeded positions when larger
    (32 MiB in all for the MOSEI shape)."""
    import numpy as np
    named = list(tr.model.named_parameters())
    params = torch.cat([p.detach().reshape(-1) for _, p in named])
    grads = torch.cat([tr.G[n].reshape(-1) for n, _ in named])
    idx = None
    if params.numel() > DUMP_SAMPLE:
        perm = torch.randperm(params.numel(), generator=torch.Generator().manual_seed(0))
        idx = perm[:DUMP_SAMPLE].sort().values.to(params.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("losses", losses.reshape(-1)), ("params", params), ("grads", grads)):
        if idx is not None and name != "losses":
            t = t[idx]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    # keep stdout clean for the single JSON line (NCCL / libraries may print banners to fd 1)
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    dist, pg, rank, local, world = dist_setup(args.gpus)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from mmda_b200 import MISA, mosei_config
    from mmda_b200.synthetic import batch_for
    from mmda_b200.trainer import FusedTrainer, LOSS_NAMES
    from mmda_b200._lib import LIB

    cfg = mosei_config(vocab_size=VOCAB, batch_size=args.batch, precision=args.precision)
    torch.manual_seed(1234)
    model = MISA(cfg)
    for n, p in model.named_parameters():         # Solver.build: orthogonal W_hh (solver.py:78-79)
        if "weight_hh" in n:
            torch.nn.init.orthogonal_(p)
    model = model.to(dev).train()
    tr = FusedTrainer(model, process_group=pg)
    eng = model.engine
    nb = 4
    host = [batch_for(cfg, seed=1234 + rank * 100 + i, lengths=args.lengths, seq_len=SEQ) for i in range(nb)]
    for b in host:                                # pinned host buffers for the e2e leg
        for f in ("sentences", "visual", "acoustic", "labels"):
            setattr(b, f, getattr(b, f).pin_memory())
    devb = [(b.sentences.to(dev), b.visual.to(dev), b.acoustic.to(dev), b.lengths, b.labels.to(dev))
            for b in host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    h2d = sum(getattr(host[0], f).numel() * getattr(host[0], f).element_size()
              for f in ("sentences", "visual", "acoustic", "labels")) + 2 * args.batch * 4

    def barrier():
        if dist is not None:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    dp = dp_check(dist, pg, rank, world, dev) if world > 1 else None

    # nvidia-smi sampler: started (and its first sample awaited) BEFORE the warm-up, so that the
    # tool's start-up neither leaves the GPU idle in front of the timed region nor eats it
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        clocks.wait_first()

    # ---- warm-up (also captures the CUDA graph of the step on a single GPU) ----
    # (ragged lengths: one graph per packed-row bucket, so a few more passes until every batch of
    # the rotation replays from a graph)
    for i in range(max(3, args.warmup) + 2 + (3 * nb if args.lengths == "ragged" else 0)):
        tr.step(*devb[i % nb])
    graph_on = tr._graph is not None

    def barrier():
        if dist is not None:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    # ---- timed region: device-resident inputs ----
    barrier()
    l0 = eng.k.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.mark()
    e0.record()
    h0 = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()                              # L2 flush between steps (inside the timed region)
        losses = tr.step(*devb[i % nb])
    host_ms = 1e3 * (time.perf_counter() - h0) / args.steps    # host enqueue time (no sync)
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr, losses)
    launches = (args.steps * tr.launches_per_step) if graph_on else (eng.k.launches - l0)
    n_graphs = len(tr._graphs)
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    value = world * args.batch * args.steps / (ms * 1e-3)

    # ---- per-launch timing of the dominant kernel (text-encoder LSTM recurrence), live, with
    # CUDA events on the launching stream; eager launches (a graph replay hides the launches) ----
    H_POS = {"mmda_lstm_forward": -3, "mmda_lstm_backward": -2,          # (.., B, H, Tmax[, save])
             "mmda_lstm_tc_forward": -4, "mmda_lstm_tc_backward": -3}     # (.., B, H, Tmax[, save], ws)
    kt = {k: [] for k in H_POS}
    orig_c = eng.k._c

    def timed_c(name, *a):
        if name not in kt or a[H_POS[name]] != cfg.embedding_size:       # text encoder only
            return orig_c(name, *a)
        e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_a.record(); orig_c(name, *a); e_b.record()
        kt[name].append((e_a, e_b))

    eng.k._c = timed_c
    tr.use_graph = False
    for i in range(min(args.steps, 10)):
        flush.zero_()
        tr.step(*devb[i % nb])
    torch.cuda.synchronize()
    tr.use_graph = graph_on
    eng.k._c = orig_c
    eng.lstm_tc_check()
    kdur = {k: (sum(a.elapsed_time(b) for a, b in v) / len(v) if v else None) for k, v in kt.items()}

    # ---- e2e: public API with host buffers, H2D + D2H inside the timed region ----
    for i in range(2):
        tr.step_batch(host[i % nb], prefetch=host[(i + 1) % nb]).tolist()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    last, pending = None, None
    for i in range(args.steps):
        flush.zero_()
        # every step: H2D of its inputs (issued one step ahead on a copy stream) + D2H of its
        # losses into pinned memory; the host reads step i's losses after enqueueing step i+1
        # (the usual asynchronous logging loop), all K reads inside the timed region
        fut = tr.step_batch(host[i % nb], prefetch=host[(i + 1) % nb], fetch=True)
        if pending is not None:
            last = pending.result()
        pending = fut
    last = pending.result()
    f1.record()
    barrier()
    t = torch.tensor([f0.elapsed_time(f1)], device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e = world * args.batch * args.steps / (float(t) * 1e-3)
    # the sampler ran through all three timed regions (device-resident steps, per-launch kernel
    # timing, end-to-end steps): every sample after mark() was taken under load
    clk = clocks.stop() if rank == 0 else None

    # captured CUDA graphs hold references to the NCCL communicator: drop them before teardown
    tr.close()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (SURVEY.md section 8d, M2/M3) ----
    roof = roofline_block(cfg, host[0], kdur, clk, args)
    cb = None
    if world == 1 and not args.no_cpu:
        cb = cpu_steps(3, 1, budget_s=40.0, batch=args.batch, lengths=args.lengths)
        cb = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "bf16",
            "data": "synthetic",
            "config": {"workload": workload(args.batch, args.lengths),
                       "global_batch": world * args.batch, "parallelism": f"dp{world}",
                       "l2": "256 MiB memset between steps inside the timed region; per-step working "
                             "set (~0.6 GB of activations) also exceeds the 126 MB L2"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 32,
                    "d2h_read": "every step's losses, read by the host one step behind the enqueue"},
            "gpu_launches": launches, "cuda_graph": graph_on, "step_graphs": n_graphs, "host_enqueue_ms_per_step": host_ms,
            "clocks": clk, "roofline": roof, "cpu_baseline": cb, "dp_check": dp,
            "losses": dict(zip(LOSS_NAMES, last[:6])), "lib": os.path.basename(LIB.load()._name)}
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()


def main():
    global SEQ
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--lengths", default="full", choices=["full", "ragged"])
    ap.add_argument("--seq", type=int, default=SEQ)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's losses, parameters and gradients as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    SEQ = args.seq
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")))
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
