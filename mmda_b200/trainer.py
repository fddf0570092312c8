"""Level-2 fused training step: the reference's ``Solver.train`` inner loop
(src/solver.py:139-193: zero_grad, forward, six losses, weighted sum, backward,
clip_grad_value_, optimizer.step with the Adam or RMSprop that ``config.optimizer`` names) with no
autograd, every stage a C-ABI kernel, parameters / gradients / optimizer state in flat 16-byte
aligned arenas, and -- when a process group is given -- batch-
sharded data parallelism with exact global-batch semantics:

* the three loss statistics segments are all-reduced between loss phases (SURVEY.md row D1:
  DiffLoss, CMD and the conf loss are statistics over the batch axis and do not decompose);
* parameter gradients are all-reduced per bucket (fusion+classifier | heads | visual | acoustic |
  text encoder + embedding) as soon as the backward has produced them, overlapping the remaining
  BPTT; buckets are contiguous ranges of the gradient arena.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch

from ._lib import LIB, MmdaError
from . import engine as _engine
from .config import OPTIMIZERS, optimizer_name
from .engine import MODS, _ptr

ALIGN = 64      # floats; every parameter starts on a 256-byte boundary of the arena
DIFF_PAIRS = ((0, 3), (1, 4), (2, 5), (2, 0), (2, 1), (0, 1))   # solver.py:432-439, token ids
LOSS_NAMES = ("cls", "diff", "sim", "recon", "conf", "total")


ROW_GRANULE = 512  # packed-row bucket of the captured step graphs (FusedTrainer.step)
MAX_GRAPHS = 24    # live step graphs per trainer before the cache is flushed
N_BUCKETS = 7      # gradient buckets 0..6 (all-reduced); N_BUCKETS = parameters without a gradient


def padded_rows(n_rows: int, batch: int, t_pad: int, granule: int = 0) -> int:
    """Launch row count of a captured step for a batch with ``n_rows`` = sum(lengths) packed rows:
    rounded up to the row granule, capped at batch * t_pad (pure function, CPU-tested)."""
    g = granule or ROW_GRANULE
    return min(batch * t_pad, -(-n_rows // g) * g)


def bucket_of(name: str) -> int:
    """Gradient-ready order of the backward (engine.backward): 0 fusion+classifier, 1 heads,
    2 visual encoder, 3 acoustic encoder, 4 text rnn2, 5 text LayerNorm + rnn1, 6 embedding (+ the
    BERT encoder), 7 never (no gradient).  The text encoder is split so that the all-reduce of
    rnn2's 8.6 MB runs under the layer-1 BPTT and the dense 24 MB embedding gradient -- ready only
    after the very last backward kernel -- is not held back by anything else."""
    if name.startswith(("transformer_encoder.", "classifier.", "confidence.")):
        return 0
    if name.startswith(("project_", "private_", "shared.", "recon_", "discriminator.")):
        return 1
    if name.startswith(("vrnn", "vlayer_norm")):
        return 2
    if name.startswith(("arnn", "alayer_norm")):
        return 3
    if name.startswith("bertmodel.pooler."):          # never used, models.py:186-198
        return N_BUCKETS
    if name.startswith("trnn2"):
        return 4
    if name.startswith(("trnn1", "tlayer_norm")):
        return 5
    if name.startswith(("embed.", "bertmodel.")):
        return 6
    if name.startswith("sp_discriminator."):
        return N_BUCKETS
    raise KeyError(name)


def plan_arena(named_shapes: List[Tuple[str, Tuple[int, ...]]], use_confid: bool, never=()):
    """-> (layout {name: (offset, numel)}, bucket ranges [(lo, hi)] for the N_BUCKETS gradient
    buckets, n_active, n_total).  ``never``: names that receive no gradient (frozen, or unused by
    this variant): they live past ``n_active`` and the optimizer never touches them.  Pure
    function (CPU-tested)."""
    never = set(never)

    def bucket(n):
        if (n.startswith("confidence.") and not use_confid) or n in never:
            return N_BUCKETS
        return bucket_of(n)
    order = sorted(range(len(named_shapes)), key=lambda i: (bucket(named_shapes[i][0]), i))
    layout, off = {}, 0
    ranges, cur, lo = [], 0, 0
    for i in order:
        name, shape = named_shapes[i]
        b = bucket(name)
        while cur < b:
            ranges.append((lo, off))
            lo, cur = off, cur + 1
        n = 1
        for s in shape:
            n *= s
        layout[name] = (off, n)
        off += (n + ALIGN - 1) // ALIGN * ALIGN
    while cur < N_BUCKETS:
        ranges.append((lo, off))
        lo, cur = off, cur + 1
    n_active = ranges[N_BUCKETS - 1][1]
    return layout, ranges[:N_BUCKETS], n_active, off


_LIVE_DP_TRAINERS = None     # weak set of data-parallel trainers that may hold captured graphs


def _register_dp_trainer(tr):
    """Captured CUDA graphs reference the NCCL communicator; ``destroy_process_group`` waits on
    them forever.  Wrap it once so that every live data-parallel trainer drops its graph first."""
    global _LIVE_DP_TRAINERS
    import weakref
    import torch.distributed as dist
    if _LIVE_DP_TRAINERS is None:
        _LIVE_DP_TRAINERS = weakref.WeakSet()
        original = dist.destroy_process_group

        def destroy_process_group(*args, **kwargs):
            for t in list(_LIVE_DP_TRAINERS):
                t.close()
            return original(*args, **kwargs)

        dist.destroy_process_group = destroy_process_group
    _LIVE_DP_TRAINERS.add(tr)


class LossFuture:
    """Losses of one step on their way to the host (FusedTrainer.step_batch(fetch=True)): a
    non-blocking device->pinned-host copy issued right behind the step, read with result()."""
    _RING = 4

    def __init__(self, trainer, losses_dev):
        ring = trainer.__dict__.setdefault("_loss_ring", [])
        if len(ring) < self._RING:
            ring.append(torch.empty(losses_dev.numel(), dtype=losses_dev.dtype).pin_memory())
        slot = trainer.__dict__["_loss_slot"] = (trainer.__dict__.get("_loss_slot", -1) + 1) % self._RING
        self.host = ring[min(slot, len(ring) - 1)]
        self.host.copy_(losses_dev.detach().reshape(-1), non_blocking=True)
        self.event = torch.cuda.Event()
        self.event.record()

    def result(self):
        self.event.synchronize()
        return self.host.tolist()


class FusedTrainer:
    def __init__(self, model, lr: Optional[float] = None, process_group=None,
                 global_batch_stats: bool = True, use_graph: Optional[bool] = None):
        self.model = model
        self.cfg = cfg = model.config
        self.use_bert = bool(getattr(cfg, "use_bert", False))
        try:
            self.optimizer = optimizer_name(getattr(cfg, "optimizer", "Adam"))
        except ValueError as e:
            raise MmdaError(str(e)) from None
        self.eng = model.engine
        self.lr = float(cfg.learning_rate if lr is None else lr)
        self.clip = float(cfg.clip)
        self.pg = process_group
        self.world = 1
        if process_group is not None:
            import torch.distributed as dist
            self.dist = dist
            self.world = dist.get_world_size(process_group)
        self.global_stats = global_batch_stats
        self.use_confid = bool(getattr(cfg, "use_confidNet", False))
        self.step_count = 0
        self._build_arena()
        self.m = torch.zeros_like(self.p_arena)     # Adam exp_avg (unused by RMSprop)
        self.v = torch.zeros_like(self.p_arena)     # Adam exp_avg_sq / RMSprop square_avg
        self._pending = []
        self._reduced = set()
        self._defer_ready = None
        self._equal_B = None            # local batch size last verified equal on every rank
        self._early_ran = False         # _loss_early enqueued the token-only part of the losses
        # device-resident step state (step counter = dropout seed offset, Adam bias corrections,
        # learning rate: csrc/adam.cu StepState, 40 bytes)
        self.state = torch.zeros(5, dtype=torch.float64, device=self.p_arena.device)
        self._lr_dev = None             # learning rate last written into self.state
        self.eng.k.bind_stream()
        self.eng.k._c("mmda_step_state_init", _ptr(self.state), 0, 0.9, 0.999)
        # CUDA-graph replay of the whole step (single GPU and data parallel)
        self.use_graph = use_graph if use_graph is not None else True
        self._graphs = {}               # key -> captured step (see step())
        self._graphs_ws = self._graphs_alias = None
        self._graphs_slots = -1
        self._graph_seen = {}
        self.launches_per_step = None
        if self.world > 1 and self.use_graph:
            _register_dp_trainer(self)

    # ------------------------------------------------------------------ arenas -------------
    def _build_arena(self):
        named = [(n, p) for n, p in self.model.named_parameters()]
        if not named[0][1].is_cuda and not _engine._DRYRUN:
            raise MmdaError("FusedTrainer needs the model on a CUDA device (model.to('cuda'))")
        dev = named[0][1].device
        # frozen tensors (src/solver.py:66-73 freezes BERT layers 0-8) and tensors the variant never
        # differentiates sit past n_active: Adam skips them exactly as torch skips grad=None
        never = [n for n, p in named if not p.requires_grad]
        if self.use_bert:
            never += [n for n, _ in named if n.startswith("tlayer_norm.")]
        self.frozen = tuple(never)
        self.layout, self.ranges, self.n_active, n_total = plan_arena(
            [(n, tuple(p.shape)) for n, p in named], self.use_confid, never)
        self.p_arena = torch.zeros(n_total, dtype=torch.float32, device=dev)
        self.g_arena = torch.zeros(n_total, dtype=torch.float32, device=dev)
        self.G: Dict[str, torch.Tensor] = {}
        for n, p in named:
            off, sz = self.layout[n]
            view = self.p_arena[off:off + sz].view(p.shape)
            view.copy_(p.data)
            p.data = view                       # the module's parameters now alias the arena
            self.G[n] = self.g_arena[off:off + sz].view(p.shape)
        self._alias_ver = tuple(p.data_ptr() for _, p in named) + \
            tuple(p.requires_grad for _, p in named)

    def _check_alias(self):
        ver = tuple(p.data_ptr() for p in self.model.parameters()) + \
            tuple(p.requires_grad for p in self.model.parameters())
        if ver != self._alias_ver:     # model.to(...) / embed.weight.data = ... after construction
            m, v, step = self.m, self.v, self.step_count
            old_layout = self.layout
            self._build_arena()
            if old_layout == self.layout and m.device == self.p_arena.device:
                self.m, self.v = m, v
            else:
                self.m, self.v = torch.zeros_like(self.p_arena), torch.zeros_like(self.p_arena)
            self.step_count = step
            self.state = self.state.to(self.p_arena.device)     # the step kernels read it by pointer

    def attach_grads(self):
        """Expose the arena gradients as ``param.grad`` (views; for inspection and tests).
        Parameters the reference leaves at ``grad=None`` stay ``None``."""
        skip = set(self.model.param_names_without_grad())
        for n, p in self.model.named_parameters():
            p.grad = None if n in skip else self.G[n]

    # ------------------------------------------------------------------ collectives --------
    def _allreduce(self, t, async_op=False):
        if self.world > 1:
            return self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.pg,
                                        async_op=async_op)
        return None

    def _check_equal_batch(self, B):
        """Data parallel only: the loss normalisers (``Bg = B * world``) and the DDP-style gradient
        average assume that every rank holds the same number of samples.  Verified with one tiny
        MAX all-reduce whenever the local batch size changes (first step, a short last batch) --
        never inside a graph capture -- so that a ragged last shard raises on every rank instead of
        silently skewing the means, CMD moments and DiffLoss Grams."""
        if self.world == 1 or B == self._equal_B:
            return
        t = torch.tensor([B, -B], dtype=torch.int64, device=self.p_arena.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.pg)
        hi, lo = int(t[0]), -int(t[1])
        if hi != lo:
            raise MmdaError(f"data-parallel step with unequal local batches ({lo}..{hi} samples per "
                            "rank): shard the global batch evenly (drop or pad the last partial batch)")
        self._equal_B = B

    # ------------------------------------------------------------------ losses -------------
    def _loss_buffers(self, B):
        d, NC = self.eng.d, self.eng.NC
        nA, nB, nC = 6 * d + 6 * NC + 4, 12 * d + 6 * d * d, 6 * d
        pad = lambda n: (n + 3) // 4 * 4
        tot = pad(nA) + pad(nB) + pad(nC) + 8 + 15 * d
        st = self.eng.buf("loss_stats", tot)
        o = 0
        segA = st[o:o + nA]; o += pad(nA)
        segB = st[o:o + nB]; o += pad(nB)
        segC = st[o:o + nC]; o += pad(nC)
        losses = st[o:o + 8]; o += 8
        coef = st[o:o + 15 * d]
        return st, segA, segB, segC, losses, coef

    def _loss_early(self, B):
        """DiffLoss / CMD chain on a side stream, forked right after the heads' forward (it reads
        the six tokens only) so that it -- and, data-parallel, its three dependent statistics
        all-reduces -- runs beside the fusion layer and the classifier instead of on the chain
        behind them.  Returns the event the late part waits for."""
        eng, k = self.eng, self.eng.k
        d, NC, cfg = eng.d, eng.NC, self.cfg
        Bg = float(B * self.world) if self.global_stats else float(B)
        sync = self.global_stats and self.world > 1
        st, segA, segB, segC, losses, coef = self._loss_buffers(B)
        X0 = eng.buf("X0", B, 6, d)
        with k.side("loss"):
            st.zero_()
            k._c("mmda_loss_phase1", _ptr(X0), None, None, None, None, None, _ptr(segA), B, d, NC, 1)
            if sync:
                self._allreduce(segA[:6 * d])
            self._loss_tokens(X0, segA, segB, segC, losses, coef, B, Bg, sync, mode=1)
        self._early_ran = True
        return k.mark("loss")

    def _loss_tokens(self, X0, segA, segB, segC, losses, coef, B, Bg, sync, mode):
        """phase 2 .. 4b: centred / normalised tokens, moments, Grams, diff + CMD values and the
        gradient wrt the tokens (dZ)"""
        eng, k = self.eng, self.eng.k
        d, NC, cfg = eng.d, eng.NC, self.cfg
        adv = eng.adversarial
        w_sim = 0.0 if adv else float(cfg.sim_weight)     # CMD part off in the adversarial variant
        w_conf = float(cfg.conf_weight) if self.use_confid else 0.0
        XN = eng.buf("XN", 6, B, d)
        inv = eng.buf("inv_norm", 6, B)
        det = k.det         # torch.are_deterministic_algorithms_enabled() at this step's forward
        if det:
            ws = k.det_ws("mmda_loss_det_workspace_bytes", B, d)
            k._c("mmda_loss_phase2_det", _ptr(X0), _ptr(segA), _ptr(XN), _ptr(inv), _ptr(segB), B, d,
                 Bg, _ptr(ws))
        else:
            k._c("mmda_loss_phase2", _ptr(X0), _ptr(segA), _ptr(XN), _ptr(inv), _ptr(segB), B, d, Bg)
        Gm = segB[12 * d:].view(6, d, d)
        k._c("mmda_loss_gram", _ptr(XN), _ptr(Gm), B, d)     # the six pairs in one launch
        if sync:
            self._allreduce(segB)
        k._c("mmda_loss_finalize", _ptr(segA), _ptr(segB), _ptr(losses), _ptr(coef), d, NC, Bg,
             float(cfg.diff_weight), float(cfg.sim_weight), float(cfg.recon_weight), w_conf,
             int(adv), mode)
        DXN = eng.buf("DXN", 6, B, d)
        alpha = float(cfg.diff_weight) * 2.0 / float(d * d)
        if det:
            k._c("mmda_loss_dxn_det", _ptr(XN), _ptr(Gm), _ptr(DXN), B, d, alpha)
            k._c("mmda_loss_phase4a_det", _ptr(DXN), _ptr(inv), _ptr(segC), B, d, _ptr(ws))
        else:
            k._c("mmda_loss_dxn", _ptr(XN), _ptr(Gm), _ptr(DXN), B, d, alpha)
            k._c("mmda_loss_phase4a", _ptr(DXN), _ptr(inv), _ptr(segC), B, d)
        if sync:
            self._allreduce(segC)
        dZ = eng.buf("dZ", B, 6, d)
        k._c("mmda_loss_phase4b", _ptr(X0), _ptr(DXN), _ptr(segA), _ptr(segB), _ptr(segC),
             _ptr(coef), _ptr(dZ), B, d, Bg, w_sim, 0)
        return dZ

    def loss_and_grads(self, out, labels, B, early_ev=None):
        """Fused losses forward + backward wrt the model outputs (csrc/loss.cu).  When
        `_loss_early` has enqueued the token-only part, wait for its event ``early_ev`` and do
        the rest."""
        eng, k = self.eng, self.eng.k
        d, NC, cfg = eng.d, eng.NC, self.cfg
        Bg = float(B * self.world) if self.global_stats else float(B)
        sync = self.global_stats and self.world > 1
        st, segA, segB, segC, losses, coef = self._loss_buffers(B)
        X0, O, R = out["tokens"], out["orig"], out["recon"]
        SC, TCP = out["scores"], out["tcp"]
        y = labels
        w_conf = float(cfg.conf_weight) if self.use_confid else 0.0
        adv = eng.adversarial
        early, self._early_ran = self._early_ran, False
        if not early:
            st.zero_()
            k._c("mmda_loss_phase1", _ptr(X0), _ptr(O), _ptr(R), _ptr(SC), _ptr(TCP), _ptr(y),
                 _ptr(segA), B, d, NC, 3)
        else:
            k.wait(early_ev)
            k._c("mmda_loss_phase1", _ptr(X0), _ptr(O), _ptr(R), _ptr(SC), _ptr(TCP), _ptr(y),
                 _ptr(segA), B, d, NC, 2)
        dDL = None
        if adv:
            dDL = eng.buf("dDL", 3, B, 3)
            k._c("mmda_loss_domain", _ptr(out["domain"]), _ptr(dDL), _ptr(segA), B, d, NC, Bg,
                 float(cfg.sim_weight))
        if not early:
            if sync:
                self._allreduce(segA)
            dZ = self._loss_tokens(X0, segA, segB, segC, losses, coef, B, Bg, sync, mode=3)
        else:
            if sync:
                self._allreduce(segA[6 * d:])
            k._c("mmda_loss_finalize", _ptr(segA), _ptr(segB), _ptr(losses), _ptr(coef), d, NC, Bg,
                 float(cfg.diff_weight), float(cfg.sim_weight), float(cfg.recon_weight), w_conf,
                 int(adv), 2)
            dZ = eng.buf("dZ", B, 6, d)
        dSC, dTCP = eng.buf("dSCORES", B, NC), eng.buf("dTCP", B, NC)
        dR, dO = eng.buf("dR", 3, B, d), eng.buf("dOrig", 3, B, d)
        k._c("mmda_loss_grad_misc", _ptr(SC), _ptr(TCP), _ptr(y), _ptr(O), _ptr(R), _ptr(segA),
             _ptr(dSC), _ptr(dTCP), _ptr(dR), _ptr(dO), B, d, NC, Bg, float(cfg.recon_weight),
             w_conf)
        return losses, dict(d_scores=dSC, d_tcp=dTCP if self.use_confid else None, d_tokens=dZ,
                            d_orig=dO, d_recon=dR, d_domain=dDL)

    # ------------------------------------------------------------------ step ---------------
    # NCCL runs the collectives of one communicator in the order they were issued.  The encoder
    # phase of the backward is enqueued text-first, so issuing on notification would put rnn2's
    # all-reduce (whose gradients complete LATE: the weight-gradient GEMMs run in the tail) in
    # front of the visual / acoustic / embedding buckets that are complete a millisecond earlier,
    # and everything would drain after the last kernel (measured: five all-reduces back to back at
    # the end of the step, 0.2 ms exposed).  Encoder-phase notifications only record an event; the
    # all-reduces are issued after the backward has been enqueued, in completion order, from a
    # helper stream that waits for exactly those events.
    _ISSUE_ORDER = ("enc_a", "enc_v", "embed", "enc_t_l2", "enc_t")

    def _on_ready(self, tag):
        if self.world == 1 or (tag == "enc_t" and self.use_bert and not self._bert_done):
            return
        if tag in self._ISSUE_ORDER and self._defer_ready is not None:
            self._defer_ready[tag] = self.eng.k.mark()
            return
        self._issue(tag)

    def _issue(self, tag):
        # enc_t_l2: the text rnn2 gradients are complete (issued from the weight-gradient stream);
        # embed: the embedding gradient is complete right after the last dX GEMM of the chain;
        # enc_t: whatever the finer-grained notifications left of the text encoder
        buckets = {"fusion": (0,), "heads": (1,), "enc_v": (2,), "enc_a": (3,), "enc_t_l2": (4,),
                   "embed": (6,), "enc_t": (5, 6)}[tag]
        if tag == "enc_t":
            buckets = tuple(b for b in (4, 5, 6) if b not in self._reduced)
        for b in buckets:
            lo, hi = self.ranges[b]
            self._reduced.add(b)
            if hi > lo:
                self._pending.append(self._allreduce(self.g_arena[lo:hi], async_op=True))

    def _flush_ready(self):
        evs, self._defer_ready = self._defer_ready, None
        if not evs:
            return
        k = self.eng.k
        with k.side("allreduce", after=()):
            for tag in self._ISSUE_ORDER:
                if tag in evs:
                    k.wait(evs[tag])
                    self._issue(tag)
        k.wait(k.mark("allreduce"))

    def forward_backward(self, sentences, visual, acoustic, lengths, labels, bert=None):
        """zero_grad + forward + losses + backward (+ gradient all-reduce).  Returns the device
        tensor of the six loss values [cls, diff, sim, recon, conf, total].  ``bert`` =
        (bert_sent, bert_sent_type, bert_sent_mask) when ``config.use_bert``."""
        self._check_alias()
        self._check_equal_batch(int(lengths.numel()))
        eng = self.eng
        self._write_lr()
        eng.k.bind_stream()
        eng.k._c("mmda_step_state_advance_device_lr", _ptr(self.state), 0.9, 0.999)
        utt_text = None
        if self.use_bert:
            if bert is None or any(t is None for t in bert):
                raise MmdaError("use_bert=True needs bert_sent / bert_sent_type / bert_sent_mask")
            utt_text = eng.bert.forward(bert[0], bert[1], bert[2], train=True,
                                        drop=self.model.training, seed=eng.seed ^ 0xB347,
                                        seed_dev=self.state)
        # the gradient arena (43 MB with a 20k-word embedding) is cleared on a side stream under
        # the forward instead of on the chain between the classifier and the losses, after the
        # previous step's optimizer read it
        with eng.k.side("zero"):
            self.g_arena[:self.n_active].zero_()
        early = {}

        def hook():
            early["ev"] = self._loss_early(int(lengths.numel()))
        out = eng.forward(sentences, visual, acoustic, lengths, train=True, want_sp=False,
                          seed_dev=self.state, utt_text=utt_text, after_heads=hook)
        B = out["scores"].shape[0]
        if labels.shape != (B, eng.NC) or labels.dtype != torch.float32 or \
                not (labels.is_cuda or _engine._DRYRUN):
            raise MmdaError("labels must be a CUDA float32 (B, num_classes) tensor")
        eng.k.wait(eng.k.mark("zero"))
        losses, grads = self.loss_and_grads(out, labels.contiguous(), B, early_ev=early["ev"])
        self._pending = []
        self._reduced = set()
        self._bert_done = False
        self._defer_ready = {} if self.world > 1 else None
        d_utt = eng.backward(self.G, on_ready=self._on_ready, **grads)
        self._flush_ready()
        if self.use_bert:
            eng.bert.backward(self.G, d_utt)
            self._bert_done = True
            self._on_ready("enc_t")
        for w in self._pending:
            w.wait()
        self._pending = []
        return losses

    def _write_lr(self):
        """Store ``self.lr`` in the device step state when it differs from the value last written.
        The advance kernel of every step (and RMSprop) reads it from there, so a captured step
        replays with whatever rate a schedule has set since.  Called outside any capture (step()
        writes it before capturing or replaying); the float the ABI takes is the rounding the
        host-lr path applied, so a constant rate gives the same bits as before."""
        lr = float(self.lr)
        if lr == self._lr_dev:
            return
        self.eng.k.bind_stream()
        LIB.call("mmda_step_state_set_lr", _ptr(self.state), lr, self.eng.k.stream)
        self._lr_dev = lr

    def optimizer_step(self):
        """clip_grad_value_ + the configured optimizer's step over the active arena; the learning
        rate is the one forward_backward / step() stored in the step state."""
        self.step_count += 1
        k = self.eng.k
        k.bind_stream()
        if self.optimizer == "RMSprop":
            o = OPTIMIZERS["RMSprop"]
            k._c("mmda_rmsprop_clip_step", _ptr(self.p_arena), _ptr(self.g_arena), _ptr(self.v),
                 self.n_active, self.lr, self.clip, o["alpha"], o["eps"], self._grad_scale(),
                 _ptr(self.state))
        else:
            k._c("mmda_adam_clip_step", _ptr(self.p_arena), _ptr(self.g_arena), _ptr(self.m),
                 _ptr(self.v), self.n_active, self.step_count, self.lr, self.clip, 0.9, 0.999, 1e-8,
                 self._grad_scale(), _ptr(self.state))

    # -- checkpoint interop: the reference saves / reloads ``optimizer.state_dict()`` next to the
    # model's (src/solver.py:219-220, :238-239); the fused step owns the optimizer state, so it
    # speaks torch.optim.Adam's or torch.optim.RMSprop's format in both directions ---------------
    _STATE_KEYS = {"Adam": ("exp_avg", "exp_avg_sq"), "RMSprop": ("square_avg",)}

    def _adam_params(self):
        """[(index, name, parameter)] in the order ``optimizer(filter(requires_grad, parameters()))``
        (src/solver.py:97-99) numbers them"""
        return [(i, n, p) for i, (n, p) in enumerate(
            (n, p) for n, p in self.model.named_parameters() if p.requires_grad)]

    def _state_arenas(self):
        """{state_dict key: arena} of the configured optimizer"""
        if self.optimizer == "RMSprop":
            return {"square_avg": self.v}
        return {"exp_avg": self.m, "exp_avg_sq": self.v}

    def optimizer_state_dict(self):
        """The optimizer state in ``torch.optim.Adam.state_dict()`` layout (or
        ``torch.optim.RMSprop``'s, with ``config.optimizer = RMSprop``): loadable by the reference's
        optimizer (``self.optimizer.load_state_dict``) built over the same model.  Parameters that
        never received a gradient (``grad=None`` in the reference: torch keeps no state for them)
        have no entry, exactly as torch leaves them."""
        params = self._adam_params()
        arenas = self._state_arenas()
        state = {}
        if self.step_count > 0:
            for i, n, p in params:
                off, sz = self.layout[n]
                if off >= self.n_active:
                    continue
                state[i] = {"step": torch.tensor(float(self.step_count))}
                for key, arena in arenas.items():
                    state[i][key] = arena[off:off + sz].view(p.shape).clone()
        if self.optimizer == "RMSprop":
            group = {"lr": self.lr, "momentum": 0, "alpha": 0.99, "eps": 1e-8, "centered": False,
                     "weight_decay": 0, "capturable": False, "foreach": None, "maximize": False,
                     "differentiable": False}
        else:
            group = {"lr": self.lr, "betas": (0.9, 0.999), "eps": 1e-8, "weight_decay": 0,
                     "amsgrad": False, "maximize": False, "foreach": None, "capturable": False,
                     "differentiable": False, "fused": None, "decoupled_weight_decay": False}
        group["params"] = [i for i, _, _ in params]
        return {"state": state, "param_groups": [group]}

    def load_optimizer_state_dict(self, sd):
        """Inverse of ``optimizer_state_dict``; also accepts a checkpoint written by the
        reference's ``torch.optim.Adam`` / ``torch.optim.RMSprop`` (``checkpoints/optim_*.std``),
        whichever ``config.optimizer`` names.  Restores the optimizer state, the step count (bias
        corrections, dropout stream) and the learning rate (written to the device before the next
        step, so a captured step graph stays valid)."""
        groups = sd["param_groups"]
        if len(groups) != 1:
            raise MmdaError("optimizer state with %d param groups (the reference uses one)" % len(groups))
        g = groups[0]
        keys = set(g) | {k for st in sd["state"].values() for k in st}
        saved = [name for name, ks in self._STATE_KEYS.items()
                 if ks[0] in keys or (name == "Adam" and "betas" in keys)
                 or (name == "RMSprop" and "alpha" in keys)]
        if saved and saved != [self.optimizer]:
            raise MmdaError(f"optimizer state of {' / '.join(saved)}, but config.optimizer is "
                            f"{self.optimizer}: load it into a trainer configured with the same "
                            "optimizer")
        if self.optimizer == "RMSprop":
            o = OPTIMIZERS["RMSprop"]
            if float(g.get("alpha", o["alpha"])) != o["alpha"] or float(g.get("eps", o["eps"])) != o["eps"] \
                    or g.get("momentum", 0) or g.get("centered", False) or g.get("weight_decay", 0) \
                    or g.get("maximize", False):
                raise MmdaError("only RMSprop(alpha=0.99, eps=1e-8, momentum=0, centered=False, "
                                "weight_decay=0) is implemented (src/solver.py:97-99 with "
                                "config.optimizer = RMSprop)")
        elif tuple(g.get("betas", (0.9, 0.999))) != (0.9, 0.999) or float(g.get("eps", 1e-8)) != 1e-8 \
                or g.get("weight_decay", 0) or g.get("amsgrad", False):
            raise MmdaError("only Adam(betas=(0.9, 0.999), eps=1e-8, weight_decay=0) is implemented "
                            "(src/solver.py:97-99 with config.optimizer = Adam)")
        params = self._adam_params()
        if len(g["params"]) != len(params):
            raise MmdaError(f"optimizer state covers {len(g['params'])} parameters, the model has "
                            f"{len(params)} trainable ones")
        pos = {pid: j for j, pid in enumerate(g["params"])}     # saved id -> position in the group
        arenas = self._state_arenas()
        self.m.zero_()
        self.v.zero_()
        steps = set()
        for pid, st in sd["state"].items():
            if pid not in pos:
                raise MmdaError(f"optimizer state for parameter id {pid!r}, which its param group does not list")
            _, n, p = params[pos[pid]]
            off, sz = self.layout[n]
            for key in arenas:
                if tuple(st[key].shape) != tuple(p.shape):
                    raise MmdaError(f"optimizer state of {n}: shape {tuple(st[key].shape)} != {tuple(p.shape)}")
            if off >= self.n_active:
                raise MmdaError(f"optimizer state for {n}, which this variant never differentiates")
            for key, arena in arenas.items():
                arena[off:off + sz].view(p.shape).copy_(st[key])
            steps.add(int(st["step"]))
        if len(steps) > 1:
            raise MmdaError(f"parameters at different {self.optimizer} steps {sorted(steps)}: one "
                            "fused step count only")
        self.step_count = steps.pop() if steps else 0
        self.lr = float(g["lr"])
        self.eng.k.bind_stream()
        # rewrites the step counter and beta products in place: a captured step reads them by
        # pointer, so it stays valid
        self.eng.k._c("mmda_step_state_init", _ptr(self.state), self.step_count, 0.9, 0.999)

    def _grad_scale(self):
        """Per-shard losses (global_batch_stats=False) are normalised by the LOCAL batch, so the
        summed gradients are world x the data-parallel average (DDP semantics: divide)."""
        return 1.0 if (self.global_stats or self.world == 1) else 1.0 / self.world

    def _eager_step(self, sentences, visual, acoustic, lengths, labels, bert=None):
        losses = self.forward_backward(sentences, visual, acoustic, lengths, labels, bert)
        self.optimizer_step()
        return losses

    def step(self, sentences, visual, acoustic, lengths, labels, bert_sent=None,
             bert_sent_type=None, bert_sent_mask=None):
        """One optimisation step.  With ``use_graph`` (the default) the kernel sequence of
        a repeated (shapes, lengths) pattern is captured once into a CUDA graph -- multi-stream
        forks included -- and replayed; per-step scalars, the learning rate included, live in
        ``self.state`` on the device, so changing ``self.lr`` between steps keeps the graph."""
        self._check_equal_batch(int(lengths.numel()))     # before any capture: it reads a value back
        self._write_lr()                                   # before any capture: a host->device copy
        if self.use_bert:       # long step (12 transformer layers): launch overhead is noise
            return self._eager_step(sentences, visual, acoustic, lengths, labels,
                                    (bert_sent, bert_sent_type, bert_sent_mask))
        if not self.use_graph or _engine._DRYRUN:
            return self._eager_step(sentences, visual, acoustic, lengths, labels)
        # Every kernel of the step runs over Np >= N packed rows and the full time extent T of the
        # input tensors (engine._pack, pad mode); the real lengths reach the kernels through the
        # device-side pack buffers, rebuilt before each replay.  So the graph key carries Np --
        # N rounded up to ROW_GRANULE, capped at B*T -- and not the lengths: a ragged data stream
        # needs one graph per row bucket (about ten for MOSEI-like length spreads), not one per
        # batch.  Batches with N == Np (full lengths: the C2 bench) get their own graph without
        # the tail-zeroing launches.
        T, B = int(sentences.shape[0]), int(sentences.shape[1])
        N = int(lengths.sum())
        cap = B * T
        Np = padded_rows(N, B, T)
        if visual.shape[0] != T or acoustic.shape[0] != T or int(lengths.max()) > T:
            return self._eager_step(sentences, visual, acoustic, lengths, labels)
        # a graph holds the launches of one reduction mode: the deterministic flag is part of the key
        key = (tuple(sentences.shape), tuple(visual.shape), tuple(acoustic.shape), Np, N == Np,
               self.model.training, torch.are_deterministic_algorithms_enabled())
        alias = tuple(p.data_ptr() for p in self.model.parameters()) + \
            tuple(p.requires_grad for p in self.model.parameters())
        if self._graphs and (self._graphs_ws != self.eng.ws_version or self._graphs_alias != alias):
            self._drop_graph()          # raw pointers inside the graphs are stale: eager warm-up first
        g = self._graphs.get(key)
        eng = self.eng
        try:
            eng.pad = (T, Np)
            if g is not None:
                # the graph reads the pack buffers (lens / sorted idx / offsets / row maps) by
                # pointer: rebuild them for these lengths (a no-op when nothing else ran on this
                # engine since the same lengths were packed)
                eng._pack(lengths)
                if self._graphs_ws == eng.ws_version:
                    srcs = [sentences, visual, acoustic, labels]
                    if all(d.dtype == s_.dtype and d.device == s_.device for d, s_ in zip(g["inputs"], srcs)):
                        torch._foreach_copy_(g["inputs"], srcs)      # one launch per dtype group
                    else:
                        for dst, src in zip(g["inputs"], srcs):
                            dst.copy_(src, non_blocking=True)
                    g["graph"].replay()
                    self.step_count += 1
                    self.launches_per_step = g["launches"]
                    return g["losses"]
                self._drop_graph()
            seen = self._graph_seen.get(key, 0) + 1
            self._graph_seen[key] = seen
            warm = 3 if not self._graphs else 2
            if seen < warm:
                # warm-up: allocates the workspace, builds the GEMM plans.  The very first ones
                # run at the largest row count this (B, T) can produce so that later, smaller
                # buckets never grow a buffer (growth would invalidate every captured graph)
                if not self._graphs:
                    eng.pad = (T, cap)
                return self._eager_step(sentences, visual, acoustic, lengths, labels)
            self._check_alias()
            if len(self._graphs) >= MAX_GRAPHS:
                self._drop_graph()
            inputs = [t.clone() for t in (sentences, visual, acoustic, labels)]
            eng._pack(lengths)             # outside the capture: its H2D copy must not be recorded
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            l0, count0 = eng.k.launches, self.step_count
            if not self._graphs:
                self._graphs_slots = LIB.raw("mmda_gemm_tc_graph_slots")(-1)
            with torch.cuda.graph(graph):
                losses = self._eager_step(inputs[0], inputs[1], inputs[2], lengths, inputs[3])
            self.launches_per_step = eng.k.launches - l0
            self.step_count = count0       # capture enqueues nothing: the replay runs the step
            if self._graphs and (self._graphs_ws != eng.ws_version):
                self._drop_graph()         # the capture grew a buffer older graphs point into
            self._graphs[key] = dict(graph=graph, inputs=inputs, losses=losses, key=key,
                                     launches=self.launches_per_step)
            self._graphs_ws, self._graphs_alias = eng.ws_version, alias
            graph.replay()
            self.step_count += 1
            return losses
        finally:
            eng.pad = None

    @property
    def _graph(self):
        """the most recently captured graph (introspection / tests)"""
        return next(reversed(self._graphs.values())) if self._graphs else None

    def _drop_graph(self):
        """Forget every captured graph (stale pointers, close()) and hand their GEMM
        tile-scheduler slots back."""
        gs, self._graphs = self._graphs, {}
        self._graph_seen = {}
        if gs:
            for g in gs.values():
                g["graph"] = None
            gs.clear()
            if not _engine._DRYRUN:
                torch.cuda.synchronize()
                LIB.raw("mmda_gemm_tc_graph_slots")(int(self._graphs_slots))

    def close(self):
        """Drop the captured CUDA graph.  Under data parallelism the graph references the NCCL
        communicator and must be gone before ``dist.destroy_process_group()`` (which otherwise
        waits for the graph's resources and hangs); ``torch.distributed.destroy_process_group``
        is wrapped to do this for every live data-parallel trainer, calling it explicitly is
        still fine."""
        self._drop_graph()
        self._graph_seen = {}
        import gc
        gc.collect()
        if not _engine._DRYRUN:
            torch.cuda.synchronize()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        """``with FusedTrainer(model, process_group=pg) as tr: ...`` drops the captured graph on the
        way out -- the explicit alternative to the wrapped ``destroy_process_group``."""
        self.close()
        return False

    def step_batch(self, batch, device=None, prefetch=None, fetch=False):
        """Public end-to-end call: a host ``Batch`` (pinned or pageable) -> one optimisation step.
        Returns the loss tensor on the device; ``.tolist()`` it to read the values.  With
        ``fetch=True`` it returns a ``LossFuture`` instead: the losses are copied to pinned host
        memory right behind the step, and ``.result()`` waits for that copy only -- a training loop
        that reads step i's losses after enqueueing step i+1 keeps the device busy back to back
        (the reference's loop blocks on ``loss.item()`` every step, solver.py:233-240).

        ``prefetch``: the host ``Batch`` of the NEXT call.  Its host->device copies are issued on
        a copy stream right after this step has been enqueued, so they overlap the step's
        kernels; the next ``step_batch(prefetch_batch)`` picks the staged tensors up."""
        dev = device or self.p_arena.device
        fields = ("sentences", "visual", "acoustic", "labels") + \
            (("bert_sent", "bert_sent_type", "bert_sent_mask") if self.use_bert else ())
        k = self.eng.k
        staged = getattr(self, "_staged", None)
        if staged is not None and staged[0] is batch:
            k.wait(staged[2])
            t = staged[1]
        else:
            t = {f: getattr(batch, f).to(dev, non_blocking=True) for f in fields}
        self._staged = None
        extra = [t[f] for f in fields[4:]]
        out = self.step(t["sentences"], t["visual"], t["acoustic"], batch.lengths, t["labels"], *extra)
        if fetch:
            out = LossFuture(self, out)
        if prefetch is not None:
            with k.side("copy", after=()):
                nt = {f: getattr(prefetch, f).to(dev, non_blocking=True) for f in fields}
            main = torch.cuda.current_stream()
            for v in nt.values():
                v.record_stream(main)
            self._staged = (prefetch, nt, k.mark("copy"))
        return out
